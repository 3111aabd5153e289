"""model x sampler x runner API of MCMC.jl on top of the C ABI (see package docstring).

Citations are file:line into the reference tree."""
import os
import time

import numpy as np

from . import _capi as capi
from ._capi import MCMCGPUError

_ctx = None
_device = -1


def set_default_device(device):
    """Switch the process to another GPU.  The old context is closed together with everything that lives in it (cached
    device models and device-resident runs: Context.close releases children first); models re-create their device
    side lazily in the new context, batches of the old context keep only what they had already fetched."""
    global _device, _ctx
    if _ctx is not None:
        _ctx.close()
        _ctx = None
    _device = int(device)


def default_context():
    """One context (one GPU) per process; LOCAL_RANK picks the device under torchrun."""
    global _ctx
    if _ctx is None:
        dev = _device
        if dev < 0 and "LOCAL_RANK" in os.environ:
            dev = int(os.environ["LOCAL_RANK"])
        _ctx = capi.Context(dev)
    return _ctx


# ---------------------------------------------------------------------------------------------------
# models (src/modellers/mcmcmodels.jl:27-33, likmodel.jl:20-58,72-143)
# ---------------------------------------------------------------------------------------------------
class MCMCLikelihoodModel:
    """GPU registry entry standing in for MCMCLikelihoodModel (likmodel.jl:20-58): a likelihood family tag
    plus its data instead of Julia closures.  eval / evalg / evalallg evaluate on the device."""

    def __init__(self, family, init, scale=1.0, pmap=None, X=None, y=None, hyper=(), gradient=True, row_sharded=False):
        init = np.atleast_1d(np.asarray(init, dtype=np.float64))          # likmodel.jl:112
        if init.ndim != 1:
            raise ValueError("init must be a vector")
        self.family = family
        self.size = init.shape[0]                                          # likmodel.jl:40
        self.init = init
        sc = np.asarray(scale, dtype=np.float64)
        self.scale = sc * np.ones(self.size) if sc.ndim == 0 else sc       # likmodel.jl:115
        if self.scale.shape != (self.size,):                               # likmodel.jl:43
            raise AssertionError(f"scale parameter size ({self.scale.shape[0]}) different from initial values ({self.size})")
        self.pmap = pmap if pmap is not None else {"pars": (1, (self.size,))}  # likmodel.jl:118
        if not _ispartition(self.pmap, self.size):                         # likmodel.jl:42, mcmcmodels.jl:9-15
            raise AssertionError("param map is not a partition of parameter vector")
        self.X, self.y, self.hyper = X, y, tuple(hyper)
        self.has_gradient = bool(gradient)
        self.row_sharded = bool(row_sharded)      # X, y are THIS rank's rows; needs init_row_sharding() first
        self._dev = None
        lt = self.eval(self.init)
        if not np.isfinite(lt):                                            # likmodel.jl:54
            raise AssertionError("Initial values out of model support, try other values")

    # -- device handle (lazy) --
    def device_model(self):
        ctx = default_context()
        if self._dev is None or self._dev.h is None or self._dev.ctx is not ctx:   # never built, closed, or of an old context
            self._dev = capi.DeviceModel(ctx, self.family, self.size, self.X, self.y, self.hyper, row_sharded=self.row_sharded)
        return self._dev

    def close(self):
        """release the device side (the packed design matrix) now; it is re-created on the next use, and released
        automatically when the model object is collected"""
        if self._dev is not None:
            self._dev.close()
            self._dev = None

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def eval(self, v):                                                     # likmodel.jl:21
        lt, _ = self.device_model().logtarget_grad(np.asarray(v, dtype=np.float64)[None, :], grad=False)
        return float(lt[0])

    def evalallg(self, v):                                                 # likmodel.jl:25
        if not self.has_gradient:
            raise AssertionError("model has no gradient function")
        lt, g = self.device_model().logtarget_grad(np.asarray(v, dtype=np.float64)[None, :], grad=True)
        return float(lt[0]), g[0]

    def evalg(self, v):                                                    # likmodel.jl:22,126-127
        return self.evalallg(v)[1]

    def __mul__(self, other):                                              # MCMC.jl:87-98
        return _combine(self, other)

    def __repr__(self):                                                    # likmodel.jl:60-66
        return f"LikelihoodModel[{self.family}], with {len(self.pmap)} parameter(s)" + (", with gradient" if self.has_gradient else "")


def _ispartition(pmap, n):                                                 # mcmcmodels.jl:9-15
    c = np.zeros(n)
    for start, shape in pmap.values():
        c[start - 1:start - 1 + int(np.prod(shape))] += 1
    return bool(np.all(c == 1))


def model(family, *, gradient=True, grad=None, init=None, scale=1.0, **kw):
    """Front door (mcmcmodels.jl:27-33).  `family` is either the text of a model expression in the reference's DSL
    (recognised shapes: mcmc.jl_b200/dsl.py; note the reference defaults to gradient=false for expressions, pass it
    explicitly) or the name of a built-in likelihood:

      "normal"      v -> -dot(v,v) (README.md:60,63); init=...; gradient/grad=False drops grad v -> -2v
      "normal_dsl"  v ~ Normal(mu, sigma) (README.md:67-72); v=<init>, mu=0, sigma=1
      "linear"      examples/linear_regression.jl:14-18;   X=, Y=, vars=<init>, prior_sd=1, noise_sd=1
      "logistic"    examples/logistic_regression.jl:16-20; X=, Y=, vars=<init>, prior_sd=1, sign=-1
      "probit"      examples/probit_regression.jl:18-41;   X=, y=, init=, priorstd=10
      "ou"          examples/ornstein.jl:19-27;            x=<series>, tau=, sigma=, mu=
    Parameter names given as keywords (vars=, v=, tau=...) become the pmap / column names, as the DSL does.
    """
    if grad is False:
        gradient = False
    if "~" in family:                                                      # a DSL expression (mcmcmodels.jl:27, likmodel.jl:72-96)
        from .dsl import recognise
        if init is not None:                                               # likmodel.jl:80
            raise AssertionError("'init' kwargs not allowed for model as expression")
        r = recognise(family, kw)
        return MCMCLikelihoodModel(r["family"], r["init"], scale, pmap=r["pmap"], X=r["X"], y=r["y"], hyper=r["hyper"],
                                   gradient=gradient)
    if family == "normal":
        if init is None:
            init = [1.0]                                                   # likmodel.jl:107
        return MCMCLikelihoodModel("normal_fn", init, scale, gradient=gradient)
    if family in ("normal_dsl", "abs_normal"):
        name, v0 = _one_param(kw, ("mu", "sigma"))
        return MCMCLikelihoodModel(family, v0, scale, pmap=_pmap_of([(name, v0)]),
                                   hyper=(kw.get("mu", 0.0), kw.get("sigma", 1.0)), gradient=gradient)
    if family in ("linear", "logistic"):
        X = np.asarray(kw.pop("X"), dtype=np.float64)
        Y = np.asarray(kw.pop("Y", kw.pop("y", None)), dtype=np.float64)
        hy = (kw.pop("prior_sd", 1.0), kw.pop("noise_sd", 1.0)) if family == "linear" else (kw.pop("prior_sd", 1.0), kw.pop("sign", -1.0))
        rs = bool(kw.pop("row_sharded", False))
        name, v0 = _one_param(kw, ())
        return MCMCLikelihoodModel(family, v0, scale, pmap=_pmap_of([(name, v0)]), X=X, y=Y, hyper=hy, gradient=gradient,
                                   row_sharded=rs)
    if family == "probit":
        X = np.asarray(kw.pop("X"), dtype=np.float64)
        y = np.asarray(kw.pop("y", kw.pop("Y", None)), dtype=np.float64)
        if init is None:
            raise ValueError("probit needs init=")
        return MCMCLikelihoodModel("probit", init, scale, X=X, y=y, hyper=(kw.pop("priorstd", 10.0),), gradient=gradient,
                                   row_sharded=bool(kw.pop("row_sharded", False)))
    if family == "ou":
        x = np.asarray(kw.pop("x"), dtype=np.float64)
        hy = (kw.pop("tau_hi", 100.0), kw.pop("sigma_hi", 2.0), kw.pop("mu_hi", 20.0))
        names = [k for k in kw]                                            # keyword order = parameter order (expr_funcs.jl:76-91)
        if sorted(names) != ["mu", "sigma", "tau"] or names != ["tau", "sigma", "mu"]:
            raise ValueError("ou needs tau=, sigma=, mu= in this order")
        v0 = np.array([kw["tau"], kw["sigma"], kw["mu"]], dtype=np.float64)
        pm = {"tau": (1, ()), "sigma": (2, ()), "mu": (3, ())}
        return MCMCLikelihoodModel("ou", v0, scale, pmap=pm, y=x, hyper=hy, gradient=gradient)
    raise ValueError(f"unknown likelihood family {family!r}")


def _one_param(kw, skip):
    names = [k for k in kw if k not in skip]
    if len(names) != 1:
        raise ValueError("give exactly one parameter vector as keyword (e.g. vars=zeros(d))")
    return names[0], np.atleast_1d(np.asarray(kw[names[0]], dtype=np.float64))


def _pmap_of(items):
    pm, pos = {}, 1
    for name, v in items:
        pm[name] = (pos, tuple(np.shape(v)))
        pos += int(np.prod(np.shape(v))) if np.ndim(v) else 1
    return pm


# ---------------------------------------------------------------------------------------------------
# samplers (src/samplers)
# ---------------------------------------------------------------------------------------------------
class EmpMCTuner:
    """samplers.jl:32-50"""

    def __init__(self, targetRate, adaptStep=100, maxStep=200, targetPath=1.0, verbose=False):
        assert adaptStep > 0, f"Adaptation step size ({adaptStep}) should be > 0"
        assert maxStep > 0, f"Adaptation step size ({maxStep}) should be > 0"
        assert 0 < targetRate < 1, f"Target acceptance rate ({targetRate}) should be between 0 and 1"
        self.adaptStep, self.maxStep, self.targetPath, self.targetRate, self.verbose = adaptStep, maxStep, targetPath, targetRate, verbose

    def _cfg(self):
        return dict(adapt_step=self.adaptStep, max_step=self.maxStep, target_path=self.targetPath, target_rate=self.targetRate)


class _Sampler:
    needs_gradient = True

    def __mul__(self, other):
        return _combine(self, other)

    def __rmul__(self, other):
        return _combine(other, self)


class RWM(_Sampler):
    """RWM.jl:24-36"""
    needs_gradient = False

    def __init__(self, scale=1.0, tuner=None):
        assert scale > 0, "scale should be > 0"
        if tuner is not None:
            raise NotImplementedError("RWM has no tuner in the reference (abstract RWMTuner, RWM.jl:19)")
        self.scale, self.tuner = float(scale), None

    def _cfg(self):
        return capi.sampler_cfg("RWM", scale=self.scale)


class RAM(_Sampler):
    """RAM.jl:24-36: RAM() = (1.0, 0.234); RAM(scale); RAM(scale, rate)"""
    needs_gradient = False

    def __init__(self, scale=1.0, rate=0.234):
        assert scale > 0, "scale should be > 0"
        assert 0.0 < rate < 1.0, f"target acceptance rate ({rate}) should be between 0 and 1"
        self.scale, self.rate, self.tuner = float(scale), float(rate), None

    def _cfg(self):
        return capi.sampler_cfg("RAM", scale=self.scale, rate=self.rate)


class MALA(_Sampler):
    """MALA.jl:50-62"""

    def __init__(self, driftStep=1.0, tuner=None, scale=None):
        if isinstance(driftStep, EmpMCTuner):                              # MALA(tuner) (MALA.jl:61, minus its typo)
            driftStep, tuner = 1.0, driftStep
        if scale is not None:
            driftStep = scale
        assert driftStep > 0, "MALA drift step should be > 0"
        self.driftStep, self.tuner = float(driftStep), tuner

    def _cfg(self):
        return capi.sampler_cfg("MALA", scale=self.driftStep, tuner=self.tuner._cfg() if self.tuner else None)


class HMC(_Sampler):
    """HMC.jl:53-74: HMC() = (10, 0.1); HMC(n::Int); HMC(step::Float64); HMC(n, step); optional tuner last."""

    def __init__(self, *args, init=None, scale=None, tuner=None, storeLeaps=False):
        nLeaps, leapStep = 10, 0.1
        args = list(args)
        if args and isinstance(args[-1], EmpMCTuner):
            tuner = args.pop()
        for a in args:
            if isinstance(a, bool):
                storeLeaps = a
            elif isinstance(a, (int, np.integer)):
                nLeaps = int(a)
            elif isinstance(a, (float, np.floating)):
                leapStep = float(a)
            else:
                raise TypeError(f"HMC: unexpected argument {a!r}")
        if init is not None:
            nLeaps = int(init)
        if scale is not None:
            leapStep = float(scale)
        assert nLeaps > 0, "inner steps should be > 0"
        assert leapStep > 0, "inner steps scaling should be > 0"
        # storeLeaps (HMC.jl:145-150): the GPU keeps the Rao-Blackwell sums mean_rb needs instead of the leap states
        self.nLeaps, self.leapStep, self.storeLeaps, self.tuner = nLeaps, leapStep, bool(storeLeaps), tuner

    def _cfg(self):
        return capi.sampler_cfg("HMC", scale=self.leapStep, nleaps=self.nLeaps, tuner=self.tuner._cfg() if self.tuner else None)


class HMCDA(_Sampler):
    """HMCDA.jl:24-43"""

    def __init__(self, rate=0.65, len=2.0, shrinkage=0.05, t0=10.0, step=0.75, storeLeaps=False, max_leaps=0):
        assert 0.0 < rate < 1.0, f"Target acceptance rate ({rate}) should be between 0 and 1"
        assert len > 0, f"len parameter of HMCDA sampler ({len}) must be non-negative"
        assert shrinkage > 0.0, f"shrinkage parameter of HMCDA sampler ({shrinkage}) must be positive"
        assert t0 >= 0, f"t0 parameter of HMCDA sampler ({t0}) must be non-negative"
        if storeLeaps:
            raise NotImplementedError("storeLeaps is outside the hot-path scope (SURVEY.md 8f.2)")
        self.rate, self.len, self.shrinkage, self.t0, self.step, self.max_leaps = rate, len, shrinkage, t0, step, max_leaps
        self.tuner = None

    def _cfg(self):
        return capi.sampler_cfg("HMCDA", rate=self.rate, len=self.len, shrinkage=self.shrinkage, t0=self.t0,
                                step=self.step, max_leaps=self.max_leaps)


class NUTS(_Sampler):
    """No-U-Turn sampler with dual averaging of the step size.  transition="slice" (the default) is slice NUTS (Hoffman &
    Gelman 2014, Algorithms 3 and 6); transition="multinomial" is Stan's transition: multinomial sampling of the
    trajectory with biased progressive sampling between subtrees, U-turn checks across neighbouring subtrees, and per
    kept step Stan's accept_stat, energy and divergence flag (MCMCChainBatch.nuts_stats, chain diagnostics).
    rate is the target mean acceptance statistic (of the last doubling for slice NUTS, Stan's accept_stat over the whole
    trajectory for multinomial NUTS; the default 0.6 is kept for both, Stan's default is 0.8), maxdoublings caps the tree
    at 2^maxdoublings - 1 leapfrogs per step,
    shrinkage / t0 / step are the dual averaging's gamma / t0 / kappa (HMCDA's).  The mass matrix is the identity unless
    inv_metric gives a diagonal inverse metric, (d,) for every chain or (nchains, d) per chain; adapt_metric=True adapts
    each chain's diagonal metric during warm-up in Stan's windows (init_buffer / term_buffer / window, Stan's defaults),
    starting from inv_metric or ones.  metric="dense" makes the metric a full matrix (Stan's dense_e): inv_metric is then
    (d, d) for every chain or (nchains, d, d) per chain, symmetric and positive definite, and the identity when None;
    adapt_metric=True adapts it from each chain's Welford covariance in the same windows.  Runs on the wave engine; the
    model's scale is not used."""

    def __init__(self, rate=0.6, maxdoublings=10, shrinkage=0.05, t0=10.0, step=0.75, inv_metric=None, adapt_metric=False,
                 init_buffer=75, term_buffer=50, window=25, metric="diag", transition="slice"):
        assert 0.0 < rate < 1.0, f"Target acceptance rate ({rate}) should be between 0 and 1"
        assert isinstance(maxdoublings, (int, np.integer)) and 1 <= maxdoublings <= 10, \
            f"maxdoublings parameter of NUTS sampler ({maxdoublings}) must be an integer in 1..10"
        assert shrinkage > 0.0, f"shrinkage parameter of NUTS sampler ({shrinkage}) must be positive"
        assert t0 >= 0, f"t0 parameter of NUTS sampler ({t0}) must be non-negative"
        assert metric in ("diag", "dense"), f"metric of NUTS sampler must be 'diag' or 'dense', got {metric!r}"
        assert transition in ("slice", "multinomial"), \
            f"transition of NUTS sampler must be 'slice' or 'multinomial', got {transition!r}"
        if inv_metric is not None and metric == "diag":
            inv_metric = np.array(inv_metric, dtype=np.float64)
            assert inv_metric.ndim in (1, 2) and inv_metric.size > 0, \
                f"inv_metric of NUTS sampler must be (d,) or (nchains, d), got shape {inv_metric.shape}"
            assert np.all(np.isfinite(inv_metric)) and np.all(inv_metric > 0), "inv_metric of NUTS sampler must be positive and finite"
        elif inv_metric is not None:
            inv_metric = np.array(inv_metric, dtype=np.float64)
            assert inv_metric.ndim in (2, 3) and inv_metric.size > 0 and inv_metric.shape[-1] == inv_metric.shape[-2], \
                f"dense inv_metric of NUTS sampler must be (d, d) or (nchains, d, d), got shape {inv_metric.shape}"
            assert np.all(np.isfinite(inv_metric)), "dense inv_metric of NUTS sampler must be finite"
            assert np.array_equal(inv_metric, np.swapaxes(inv_metric, -1, -2)), "dense inv_metric of NUTS sampler must be symmetric"
            try:
                np.linalg.cholesky(inv_metric)
            except np.linalg.LinAlgError:
                raise AssertionError("dense inv_metric of NUTS sampler must be positive definite") from None
        for name, v, lo in (("init_buffer", init_buffer, 0), ("term_buffer", term_buffer, 0), ("window", window, 1)):
            assert isinstance(v, (int, np.integer)) and v >= lo, f"{name} of NUTS sampler ({v}) must be an integer >= {lo}"
        self.rate, self.maxdoublings, self.shrinkage, self.t0, self.step = rate, int(maxdoublings), shrinkage, t0, step
        self.inv_metric, self.adapt_metric, self.metric, self.transition = inv_metric, bool(adapt_metric), metric, transition
        self.init_buffer, self.term_buffer, self.window = int(init_buffer), int(term_buffer), int(window)
        self.tuner = None

    def _set_metric(self, drun, offset, nchains):
        """the metric and transition calls of a run of chains offset .. offset + drun.C - 1 of nchains (none with the
        defaults)"""
        if self.transition == "multinomial":
            drun.set_nuts_transition(capi.NUTS_MULTINOMIAL)
        if self.metric == "dense":
            m = self.inv_metric
            assert m is None or m.ndim == 2 or m.shape[0] == nchains, \
                f"dense inv_metric of NUTS sampler has {m.shape[0]} matrices for {nchains} chains"
            drun.set_dense_metric(m if m is None or m.ndim == 2 else m[offset:offset + drun.C])
        elif self.inv_metric is not None:
            assert self.inv_metric.ndim == 1 or self.inv_metric.shape[0] == nchains, \
                f"inv_metric of NUTS sampler has {self.inv_metric.shape[0]} rows for {nchains} chains"
            drun.set_metric(self.inv_metric if self.inv_metric.ndim == 1 else self.inv_metric[offset:offset + drun.C])
        if self.adapt_metric:
            drun.set_metric_adaptation(self.init_buffer, self.term_buffer, self.window)

    def _cfg(self):
        return capi.sampler_cfg("NUTS", nleaps=self.maxdoublings, rate=self.rate, shrinkage=self.shrinkage, t0=self.t0,
                                step=self.step)


# ---------------------------------------------------------------------------------------------------
# runners (src/runners)
# ---------------------------------------------------------------------------------------------------
class SerialMC:
    """SerialMC.jl:12-35: SerialMC(steps=, burnin=, thinning=) == range (burnin+1):thinning:steps;
    SerialMC(range(a, b+1[, s])); SerialMC(a, b) == a:b.  Runs one chain -- on the GPU."""
    nchains = 1

    def __init__(self, *args, steps=100, burnin=0, thinning=1):
        if len(args) == 1 and isinstance(args[0], range):
            r = args[0]
            first, step, last = r.start, r.step, r[-1]
        elif len(args) == 2:
            first, step, last = int(args[0]), 1, int(args[1])
        elif len(args) == 3:
            first, step, last = int(args[0]), int(args[1]), int(args[2])
        elif not args:
            first, step, last = burnin + 1, thinning, steps
            last = first + ((last - first) // step) * step if last >= first else last
        else:
            raise TypeError("SerialMC(range) | SerialMC(first, last) | SerialMC(first, step, last) | SerialMC(steps=, burnin=, thinning=)")
        self.burnin, self.thinning, self.len = first - 1, step, last       # SerialMC.jl:21-23
        assert self.burnin >= 0, f"Burnin rounds ({self.burnin}) should be >= 0"
        assert self.len > self.burnin, f"Total MCMC length ({self.len}) should be > to burnin ({self.burnin})"
        assert self.thinning >= 1, f"Thinning ({self.thinning}) should be >= 1"
        self.r = range(first, last + 1, step)

    seed, store_gradients, engine, shard = 0, True, "auto", "chains"

    def __rmul__(self, other):
        return _combine(other, self)


class GPUMC(SerialMC):
    """The many-chain runner added beside SerialMC (SURVEY.md 8b): same range arguments plus
    nchains, seed, shard ("chains": chains split over ranks, no communication), store_gradients, engine."""

    def __init__(self, *args, nchains=1, seed=0, shard="chains", store_gradients=True, engine="auto", store_draws=True, **kw):
        super().__init__(*args, **kw)
        assert nchains >= 1
        assert shard in ("chains", "rows")
        self.nchains, self.seed, self.shard, self.store_gradients, self.engine = int(nchains), int(seed), shard, store_gradients, engine
        # store_draws=False: the fused engine keeps no draws and accumulates mean / var(:iid, :bm) / ess(:bm) / acceptance while
        # sampling (closed-form families); the batch then answers mean(), var(vtype="bm"), ess(vtype="bm"), acceptance() only
        self.store_draws = bool(store_draws)


class SeqMC:
    """SeqMC.jl:24-37: SeqMC(steps=, burnin=, trigger=)"""
    nchains = 1

    def __init__(self, steps=1, burnin=0, trigger=1e-10):
        assert burnin >= 0, f"Burnin rounds ({burnin}) should be >= 0"
        assert steps > burnin, f"Steps ({steps}) should be > to burnin ({burnin})"
        self.steps, self.burnin, self.trigger = int(steps), int(burnin), float(trigger)

    def __rmul__(self, other):
        return _combine(other, self)


class SerialTempMC:
    """SerialTempMC.jl:16-29: SerialTempMC(steps=, burnin=, swapPeriod=)"""
    nchains = 1

    def __init__(self, steps=1, burnin=0, swapPeriod=5):
        assert burnin >= 0, f"Burnin rounds ({burnin}) should be >= 0"
        assert steps > burnin, f"Steps ({steps}) should be > to burnin ({burnin})"
        self.steps, self.burnin, self.swapPeriod = int(steps), int(burnin), int(swapPeriod)

    def __rmul__(self, other):
        return _combine(other, self)


# ---------------------------------------------------------------------------------------------------
# tasks and the * operator (MCMC.jl:33-38,87-98; samplers.jl:53)
# ---------------------------------------------------------------------------------------------------
class MCMCTask:
    def __init__(self, model, sampler, runner):
        self.model, self.sampler, self.runner = model, sampler, runner


class _Partial:
    def __init__(self, models, samplers):
        self.models, self.samplers = models, samplers

    def __mul__(self, runner):
        return _combine(self, runner)


def _aslist(x):
    return (list(x), True) if isinstance(x, (list, tuple)) else ([x], False)


def _combine(a, b):
    """m * s -> partial; partial * r -> MCMCTask or list of tasks, broadcasting arrays like MCMC.jl:87-98."""
    if isinstance(a, (MCMCLikelihoodModel, list, tuple)) and not isinstance(a, _Partial) and \
            (isinstance(b, _Sampler) or (isinstance(b, (list, tuple)) and b and isinstance(b[0], _Sampler))):
        return _Partial(a, b)
    if isinstance(a, _Partial):
        ms, ml = _aslist(a.models)
        ss, sl = _aslist(a.samplers)
        rs, rl = _aslist(b)
        n = max(len(ms) if ml else 1, len(ss) if sl else 1, len(rs) if rl else 1)
        for lst, isl in ((ms, ml), (ss, sl), (rs, rl)):
            if isl and len(lst) != n:
                raise ValueError("array arguments of * must have the same length")
        tasks = [MCMCTask(ms[i] if ml else ms[0], ss[i] if sl else ss[0], rs[i] if rl else rs[0]) for i in range(n)]
        return tasks if (ml or sl or rl) else tasks[0]
    return NotImplemented


# allow [samplers] * runner after model * [samplers]
list_mul = _combine


# ---------------------------------------------------------------------------------------------------
# chains (MCMC.jl:58-84)
# ---------------------------------------------------------------------------------------------------
def _colnames(m):
    """SerialMC.jl:70-79"""
    cn = [None] * m.size
    for k, (start, shape) in m.pmap.items():
        if len(shape) == 0:
            cn[start - 1] = str(k)
        elif len(shape) == 1:
            for i in range(shape[0]):
                cn[start - 1 + i] = f"{k}.{i + 1}"
        else:
            idx = 0
            for j in range(shape[1]):
                for i in range(shape[0]):
                    cn[start - 1 + idx] = f"{k}.{i + 1}.{j + 1}"
                    idx += 1
    return cn


class MCMCChain:
    """MCMC.jl:58-71: range, samples (S x d DataFrame), gradients, diagnostics {"step", "accept"}, task, runTime."""

    def __init__(self, rng, samples, gradients, diagnostics, task, runTime, columns):
        import pandas as pd
        if gradients is not None and gradients.size:
            assert samples.shape == gradients.shape, "samples and gradients must have the same number of rows and columns"
        self.range = rng
        self._s = np.ascontiguousarray(samples)
        self.samples = pd.DataFrame(self._s, columns=columns)
        self.gradients = pd.DataFrame(gradients, columns=columns) if gradients is not None else pd.DataFrame()
        self.diagnostics, self.task, self.runTime = diagnostics, task, runTime

    def __repr__(self):                                                    # MCMC.jl:82-84
        return f"{self.samples.shape[1]} parameters, {self.samples.shape[0]} samples (per parameter), {round(self.runTime, 1)} sec."


class MCMCChainBatch:
    """Result of a many-chain run: draws stay on the device until asked for; batch[i] materialises the i-th
    MCMCChain lazily (building 65 536 DataFrames eagerly would dwarf the GPU time, SURVEY.md section 7)."""

    def __init__(self, task, drun, runTime, info, chain_offset=0):
        self.task, self._run, self.runTime, self.info = task, drun, runTime, info
        self.nchains, self.range = drun.C, task.runner.r
        self.chain_offset = chain_offset
        self._host = None

    def arrays(self):
        """dict(samples (C,S,d), grads (C,S,d)?, accept (C,S), logtarget (C,S))"""
        if self._host is None:
            self._host = self._run.fetch()
        return self._host

    def __len__(self):
        return self.nchains

    def __getitem__(self, i):
        a = self.arrays()
        diags = {"step": np.array(list(self.range)), "accept": a["accept"][i].astype(bool)}
        s = self.task.sampler
        if isinstance(s, NUTS):
            eps, leaps = self.diag()
            diags["epsilon"] = eps[i]
            diags["ndoublings"] = np.floor(np.log2(leaps[i])).astype(np.int64) + 1    # the tree of 2^(n-1) .. 2^n - 1 leapfrogs
            if s.inv_metric is not None or s.adapt_metric or s.metric == "dense":
                diags["inv_metric"] = self.inv_metric()[i]
            if s.transition == "multinomial":
                diags.update({k: v[i] for k, v in self.nuts_stats().items()})
        g = a.get("grads")
        return MCMCChain(self.range, a["samples"][i], None if g is None else g[i], diags, self.task, self.runTime,
                         _colnames(self.task.model))

    def __iter__(self):
        return (self[i] for i in range(self.nchains))

    def diag(self):
        """(C, S) step sizes and (C, S) leapfrog counts of the kept steps (HMCDA, NUTS, RAM, tuned samplers)"""
        if getattr(self, "_diag", None) is None:
            self._diag = self._run.fetch_diag()
        return self._diag

    def nuts_stats(self):
        """multinomial NUTS: dict of (C, S) arrays of the kept steps -- accept_stat (Stan's mean Metropolis acceptance over
        the trajectory), energy (H of the draw) and divergent (bool: the last subtree stopped at H - H0 > 1000)"""
        if getattr(self, "_nuts_stats", None) is None:
            self._nuts_stats = self._run.fetch_nuts_stats()
        return self._nuts_stats

    def inv_metric(self):
        """the inverse metric of every chain at the end of the run (NUTS): (C, d) diagonal (ones for the identity), or
        (C, d, d) for a dense metric"""
        if getattr(self, "_minv", None) is None:
            dense = getattr(self.task.sampler, "metric", "diag") == "dense"
            self._minv = self._run.get_dense_metric() if dense else self._run.get_metric()
        return self._minv

    def stats(self, vtype="imse", **kw):
        return self._run.stats(vtype, kw.get("maxlag", -1), kw.get("batchlen", 100))

    def rb(self):
        """(C, S, d) Rao-Blackwellised draws of an HMC(storeLeaps=true) run"""
        return self._run.fetch_rb()

    def close(self):
        """release the device-resident draws (also done when the batch is collected, or by `with run(...) as batch`)"""
        self._run.close()

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()


# ---------------------------------------------------------------------------------------------------
# tall data: rows of X sharded over the ranks of a torchrun launch (SURVEY.md 8e.2)
# ---------------------------------------------------------------------------------------------------
def shard_rows(N, rank=None, world=None):
    """rows [lo, hi) of rank g: contiguous blocks [g*N/G, (g+1)*N/G)"""
    world = int(os.environ.get("WORLD_SIZE", "1")) if world is None else world
    rank = int(os.environ.get("RANK", "0")) if rank is None else rank
    return (rank * N) // world, ((rank + 1) * N) // world


def broadcast_unique_id(dist, make_id, rank):
    """rank 0 creates the 128-byte NCCL unique id, every rank receives it through the process group `dist`
    (any backend: the id is plain bytes)"""
    import torch
    buf = torch.zeros(128, dtype=torch.uint8)
    if rank == 0:
        buf = torch.frombuffer(bytearray(make_id()), dtype=torch.uint8).clone()
    dev = "cuda" if dist.get_backend() == "nccl" else "cpu"
    buf = buf.to(dev)
    dist.broadcast(buf, src=0)
    return bytes(buf.cpu().numpy().tobytes())


def init_row_sharding():
    """one NCCL communicator over all ranks, owned by the library (per-leapfrog all-reduce of the partial
    log-likelihood and gradient).  torch.distributed must be initialised (it only carries the unique id)."""
    import torch.distributed as dist
    ctx = default_context()
    rank, world = dist.get_rank(), dist.get_world_size()
    uid = broadcast_unique_id(dist, capi.Context.comm_unique_id, rank)
    ctx.comm_init(rank, world, uid)
    return rank, world


# ---------------------------------------------------------------------------------------------------
# run / prun / resume (runners.jl:7-68, SerialMC.jl:37-97)
# ---------------------------------------------------------------------------------------------------
def _rank_slice(nchains):
    """chain sharding across ranks of a torchrun launch: contiguous global chain ids, Philox keyed by global id"""
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    per = (nchains + world - 1) // world
    lo = min(rank * per, nchains)
    return lo, min(lo + per, nchains) - lo


def _run_task(t, init=None, normals=None, uniforms=None, shard_over_ranks=False):
    m, s, r = t.model, t.sampler, t.runner
    if s.needs_gradient and not m.has_gradient:                            # MALA.jl:72, HMC.jl:111, HMCDA.jl:79
        raise AssertionError(f"{type(s).__name__} sampler requires model with gradient function")
    t0 = time.time()
    nchains, offset = r.nchains, 0
    if shard_over_ranks and r.shard == "chains":
        offset, nchains = _rank_slice(r.nchains)
    ini = m.init if init is None else np.asarray(init, dtype=np.float64)
    if ini.ndim == 2:
        ini = ini[offset:offset + nchains]
    stream = not getattr(r, "store_draws", True)
    drun = capi.DeviceRun(m.device_model(), s._cfg(), (r.r.start, r.r.step, r.r[-1]), nchains, ini, scale=m.scale,
                          seed=r.seed, chain_offset=offset, normals=normals, uniforms=uniforms,
                          store_grad=bool(r.store_gradients) and not stream, store_logtarget=not stream,
                          engine="fused" if stream else r.engine, store_rb=bool(getattr(s, "storeLeaps", False)), stream_stats=stream)
    try:
        if isinstance(s, NUTS):
            s._set_metric(drun, offset, r.nchains)
        info = drun.execute()
    except AssertionError:
        drun.close()
        raise
    except MCMCGPUError as e:
        drun.close()
        if e.code == capi.E_SUPPORT:
            raise AssertionError("Initial values out of model support, try other values") from e
        raise
    return MCMCChainBatch(t, drun, time.time() - t0, info, offset)


def run(*args, **kw):
    """run(task) | run([tasks]) | run(model, sampler, runner) | run(chain) (runners.jl:7-45).
    A SerialMC task returns one MCMCChain; a GPUMC task returns an MCMCChainBatch."""
    if len(args) == 3:
        return run(args[0] * args[1] * args[2], **kw)
    (t,) = args
    if isinstance(t, (MCMCChain, MCMCChainBatch)):
        return run(t.task, **kw)
    if isinstance(t, (list, tuple)):
        last = t[-1].runner
        assert all(type(x.runner) is type(last) for x in t), "Runners do not have the same runner type"  # runners.jl:19
        if isinstance(last, SeqMC):                                        # runners.jl:29-30
            return _run_seqmc(list(t), **kw)
        if isinstance(last, SerialTempMC):                                 # runners.jl:27-28
            return _run_serialtempmc(list(t), **kw)
        return [run(x, **kw) for x in t]
    batch = _run_task(t, **kw)
    if isinstance(t.runner, GPUMC):
        return batch
    chain = batch[0]
    if getattr(t.sampler, "storeLeaps", False):
        chain.diagnostics["rb"] = batch.rb()[0]
    chain.runTime = batch.runTime
    batch.close()
    return chain


def _population_tasks(tasks):
    m0 = tasks[-1].model
    assert all(t.model.size == m0.size for t in tasks), "Models do not have the same parameter vector size"   # SeqMC.jl:47
    for t in tasks:
        if t.sampler.needs_gradient and not t.model.has_gradient:
            raise AssertionError(f"{type(t.sampler).__name__} sampler requires model with gradient function")
        if getattr(t.sampler, "tuner", None) is not None or isinstance(t.sampler, (HMCDA, NUTS)):
            raise NotImplementedError("population runners take RWM, MALA or HMC tasks without tuner")
    return m0, [t.model.hyper for t in tasks], [t.sampler._cfg() for t in tasks]


def _run_seqmc(tasks, particles=None, seed=0, normals=None, uniforms=None, res_uniforms=None):
    """run(targets; particles=...) with SeqMC runners (SeqMC.jl:39-122): one MCMCChain holding (steps-burnin)*npart
    samples, diagnostics "weigths" (sic, SeqMC.jl:119) and "particle"."""
    t0 = time.time()
    r = tasks[-1].runner
    m0, hypers, samplers = _population_tasks(tasks)
    if particles is None:                                                  # SeqMC.jl:39 default: 100 particles of randn()
        particles = np.random.default_rng(seed).standard_normal((100, m0.size))
    particles = np.asarray([np.atleast_1d(p) for p in particles], dtype=np.float64)
    same_family = all(t.model.family == m0.family for t in tasks)
    if same_family and m0.family in ("normal_fn", "normal_dsl", "abs_normal") and m0.size <= 8:
        # closed-form ladder: one thread mutates one particle, everything in registers
        res = default_context().run_seqmc(m0.family, m0.size, hypers, samplers, r.steps, r.burnin, r.trigger, particles, seed=seed,
                                          normals=normals, uniforms=uniforms, res_uniforms=res_uniforms)
    else:
        # any models (regression families, d > 8, mixed families): particles are chains of one-step runs of the wave engine,
        # the likelihood kernel evaluates the whole population at once
        res = default_context().run_seqmc_models([t.model.device_model() for t in tasks], samplers, r.steps, r.burnin, r.trigger,
                                                 particles, seed=seed, normals=normals, uniforms=uniforms, res_uniforms=res_uniforms)
    npart, S = particles.shape[0], (r.steps - r.burnin) * particles.shape[0]
    diags = {"weigths": res["weights"], "particle": np.tile(np.arange(1, npart + 1), r.steps - r.burnin)}
    chain = MCMCChain(range(r.burnin + 1, S + 1), res["samples"], None, diags, tasks, time.time() - t0, _colnames(m0))
    chain.info = res["info"]
    chain.n_resamples = res["n_resamples"]
    return chain


def _run_serialtempmc(tasks, nreplicas=1, seed=0, **draws):
    """run(tasks) with SerialTempMC runners (SerialTempMC.jl:31-85): one MCMCChain of steps-burnin draws (the reference
    stores them column-per-step, :47,77; here rows are draws like every other chain) and the visited task in
    diagnostics["task"]; nreplicas > 1 returns a list of independent replicas."""
    t0 = time.time()
    r = tasks[-1].runner
    m0, hypers, samplers = _population_tasks(tasks)
    inits = np.stack([t.model.init for t in tasks])
    closed = all(t.model.family == m0.family for t in tasks) and m0.family in ("normal_fn", "normal_dsl", "abs_normal") and m0.size <= 8
    try:
        if closed:      # one thread = one replica, the whole run in one launch
            res = default_context().run_serialtemp(m0.family, m0.size, hypers, samplers, r.steps, r.burnin, r.swapPeriod, nreplicas,
                                                   inits, seed=seed, **draws)
        else:           # any models: replicas regrouped by task, each group a one-step run of the wave engine (K1)
            res = default_context().run_serialtemp_models([t.model.device_model() for t in tasks], samplers, r.steps, r.burnin,
                                                          r.swapPeriod, nreplicas, inits, seed=seed, **draws)
    except MCMCGPUError as e:
        if e.code == capi.E_SUPPORT:
            raise AssertionError("Initial values out of model support, try other values") from e
        raise
    chains = []
    for c in range(nreplicas):
        ch = MCMCChain(range(1, 3), res["samples"][c], None, {"task": res["at"][c] + 1}, tasks, time.time() - t0, _colnames(m0))
        ch.info = res["info"]
        chains.append(ch)
    return chains[0] if nreplicas == 1 else chains


def prun(tasks, **kw):
    """runners.jl:35-42 (pmap over workers): here every task already runs on the GPU; under torchrun a GPUMC task
    is chain-sharded over the ranks (each rank returns its own slice)."""
    if isinstance(tasks, MCMCTask):
        return _run_task(tasks, shard_over_ranks=True, **kw)
    return [_run_task(t, shard_over_ranks=True, **kw) if isinstance(t.runner, GPUMC) else run(t, **kw) for t in tasks]


def resume(c, steps=100):
    """runners.jl:48-68 / SerialMC.jl:93-97: like the reference, a fresh run from model.init keeping the thinning."""
    t = c.task if isinstance(c, (MCMCChain, MCMCChainBatch)) else c
    if isinstance(t, (list, tuple)):
        return [resume(x, steps=steps) for x in t]
    r = t.runner
    if isinstance(r, GPUMC):
        nr = GPUMC(steps=steps, thinning=r.thinning, nchains=r.nchains, seed=r.seed, shard=r.shard,
                   store_gradients=r.store_gradients, engine=r.engine)
    else:
        nr = SerialMC(steps=steps, thinning=r.thinning)
    return run(MCMCTask(t.model, t.sampler, nr))


# ---------------------------------------------------------------------------------------------------
# stats (src/stats): all estimators run on the device
# ---------------------------------------------------------------------------------------------------
_VTYPES = ("bm", "iid", "imse", "ipse")                                  # var.jl:135
_ACTYPES = ("bm", "imse", "ipse")                                        # ess.jl:4


def _stats(c, vtype, pars=None, **kw):
    if isinstance(c, MCMCChainBatch):
        st = c.stats(vtype, **kw)
    else:
        st = default_context().stats(c._s[None, :, :], vtype, kw.get("maxlag", -1), kw.get("batchlen", 100))
        st = {k: v[0] for k, v in st.items()}
    if pars is not None:
        idx = [p - 1 for p in ([pars] if np.isscalar(pars) else list(pars))]
        st = {k: (v[..., idx] if v.ndim and v.shape[-1] >= max(idx) + 1 else v) for k, v in st.items()}
    return st


def mean(c, pars=None):                                                    # mean.jl:6
    return _stats(c, "iid", pars)["mean"]


def mean_rb(c, pars=None, s="hmc"):
    """mean.jl:37-41: mean of an HMC(storeLeaps=true) chain from the Rao-Blackwell samples (mean.jl:11-35)"""
    assert s == "hmc"
    rb = c.rb() if isinstance(c, MCMCChainBatch) else c.diagnostics["rb"][None]
    out = rb.mean(axis=1)
    if pars is not None:
        out = out[:, [p - 1 for p in ([pars] if np.isscalar(pars) else list(pars))]]
    return out if isinstance(c, MCMCChainBatch) else out[0]


def var(c, pars=None, vtype="imse", **kw):                                 # var.jl:137-151
    assert vtype in _VTYPES, f"Unknown variance type {vtype}"
    return _stats(c, vtype, pars, **kw)["var"]


def std(c, pars=None, vtype="imse", **kw):
    """Monte Carlo standard error = sqrt(var(c; vtype)) -- what describe() prints as "MC Error"
    (summary.jl:38-40); the reference's own std() dispatch is broken (var.jl:13,88-89,160)."""
    assert vtype in _VTYPES, f"Unknown standard error type {vtype}"
    return np.sqrt(var(c, pars, vtype, **kw))


def ess(c, pars=None, vtype="imse", **kw):                                 # ess.jl:6-10
    assert vtype in _ACTYPES, f"Unknown ESS type {vtype}"
    return _stats(c, vtype, pars, **kw)["ess"]


def actime(c, pars=None, vtype="imse", **kw):                              # ess.jl:15-19
    assert vtype in _ACTYPES, f"Unknown integrated autocorrelation time type {vtype}"
    return _stats(c, vtype, pars, **kw)["actime"]


def acceptance(c, lags=None, reject=False):                                # summary.jl:6-15
    if isinstance(c, MCMCChainBatch) and c._run.streaming:        # GPUMC(store_draws=False): the rate was accumulated while sampling
        assert lags is None, "a streamed run keeps no per-step accept flags"
        rate = c.stats("iid")["accept_rate"]
        return 100.0 - rate if reject else rate
    if isinstance(c, MCMCChainBatch):
        acc = c.arrays()["accept"].astype(np.float64)
    else:
        acc = np.asarray(c.diagnostics["accept"], dtype=np.float64)[None, :]
    n = acc.shape[1]
    if lags is not None:
        lags = list(lags)
        assert lags[-1] <= n, "Range of acceptance rate not within post-burnin range of MCMC chain"
        acc = acc[:, [l - 1 for l in lags]]
    rlen = acc.shape[1]
    a = acc.sum(axis=1)
    out = (rlen - a) * 100 / rlen if reject else a * 100 / rlen
    return out if isinstance(c, MCMCChainBatch) else float(out[0])


def linearZv(c, grad=None):
    """zv.jl:8-29: (zvChain, a).  c: MCMCChain, MCMCChainBatch, or an (S, d) array with grad an (S, d) array."""
    return _zv(c, grad, 1)


def quadraticZv(c, grad=None):
    """zv.jl:32-66"""
    return _zv(c, grad, 2)


def _zv(c, grad, order):
    if isinstance(c, MCMCChainBatch):
        return c._run.zv(order)
    if isinstance(c, MCMCChain):
        x, g = c._s, c.gradients.values
    else:
        x, g = np.asarray(c, dtype=np.float64), np.asarray(grad, dtype=np.float64)
    zv, a = default_context().zv(x[None], g[None], order)
    return zv[0], a[0]


def describe(c, io=None):
    """summary.jl:24-55 for one chain: Min / Mean / Max / MC Error / ESS / AC Time per parameter."""
    import sys
    io = io or sys.stdout
    st = _stats(c, "imse")
    for i, name in enumerate(c.samples.columns):
        col = c._s[:, i]
        vals = [col.min(), st["mean"][i], col.max(), float(np.sqrt(st["var"][i])), st["ess"][i], st["actime"][i]]
        print(name, file=io)
        for nm, v in zip(["Min", "Mean", "Max", "MC Error", "ESS", "AC Time"], vals):
            print(f"{nm.ljust(10)} {v}", file=io)
        print("NAs        0", file=io)
        print("NA%        0.0%", file=io)
        print(file=io)
