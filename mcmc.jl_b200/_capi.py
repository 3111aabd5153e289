"""ctypes binding of libmcmcgpu.so (include/mcmcgpu.h) -- the same marshalling a Julia `ccall` does.

There is no CPU fallback: if the shared library is missing, or no CUDA device is present, every
compute call raises.
"""
import ctypes as C
import os
import weakref

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("MCMCGPU_LIB") or os.path.join(_HERE, "libmcmcgpu.so")   # MCMCGPU_LIB: A/B timing of two builds (tools/)

OK, E_ARG, E_SUPPORT, E_NOGRAD, E_CUDA, E_COMM, E_STATE = 0, -1, -2, -3, -4, -5, -6
FAM = dict(normal_fn=0, normal_dsl=1, linear=2, logistic=3, probit=4, ou=5, abs_normal=6)
KIND = dict(RWM=0, MALA=1, HMC=2, HMCDA=3, RAM=4, NUTS=5)
NUTS_SLICE, NUTS_MULTINOMIAL = 0, 1                                     # mcmcgpu_run_set_nuts_transition
ENGINE = dict(auto=0, fused=1, wave=2)
VTYPE = dict(iid=0, bm=1, imse=2, ipse=3)


class MCMCGPUError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"libmcmcgpu error {code}: {msg}")
        self.code = code


class SamplerCfg(C.Structure):
    _fields_ = [("kind", C.c_int32), ("nleaps", C.c_int32), ("scale", C.c_double),
                ("rate", C.c_double), ("len", C.c_double), ("shrinkage", C.c_double),
                ("t0", C.c_double), ("step", C.c_double), ("max_leaps", C.c_int64),
                ("tuner_on", C.c_int32), ("adapt_step", C.c_int32), ("max_step", C.c_int32),
                ("target_path", C.c_double), ("target_rate", C.c_double)]


class RunnerCfg(C.Structure):
    _fields_ = [("first", C.c_int64), ("step", C.c_int64), ("last", C.c_int64),
                ("nchains", C.c_int64), ("chain_offset", C.c_int64), ("seed", C.c_uint64),
                ("init_per_chain", C.c_int32), ("store_grad", C.c_int32),
                ("store_logtarget", C.c_int32), ("engine", C.c_int32), ("store_rb", C.c_int32),
                ("stream_stats", C.c_int32), ("stream_batchlen", C.c_int32)]


class RunInfo(C.Structure):
    _fields_ = [("gpu_ms", C.c_double), ("n_grad_evals", C.c_int64), ("n_waves", C.c_int64),
                ("n_launches", C.c_int64), ("eval_ms", C.c_double), ("comm_ms", C.c_double)]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_}


EXPORTS = [
    "mcmcgpu_abi_version", "mcmcgpu_last_error", "mcmcgpu_init", "mcmcgpu_destroy", "mcmcgpu_set_stream",
    "mcmcgpu_set_option", "mcmcgpu_comm_unique_id", "mcmcgpu_comm_init", "mcmcgpu_model_create", "mcmcgpu_model_create_device",
    "mcmcgpu_model_destroy", "mcmcgpu_logtarget_grad", "mcmcgpu_run_chains", "mcmcgpu_run_create",
    "mcmcgpu_run_execute", "mcmcgpu_run_execute_steps", "mcmcgpu_run_set_state", "mcmcgpu_run_get_state",
    "mcmcgpu_run_fetch", "mcmcgpu_run_fetch_rb", "mcmcgpu_run_fetch_diag", "mcmcgpu_run_stats",
    "mcmcgpu_run_destroy", "mcmcgpu_stats", "mcmcgpu_philox_draws", "mcmcgpu_run_seqmc", "mcmcgpu_run_serialtemp", "mcmcgpu_run_zv", "mcmcgpu_zv",
    "mcmcgpu_run_seqmc_models", "mcmcgpu_run_serialtemp_models",
    "mcmcgpu_run_set_metric", "mcmcgpu_run_set_metric_adaptation", "mcmcgpu_run_get_metric",
    "mcmcgpu_run_set_dense_metric", "mcmcgpu_run_get_dense_metric",
    "mcmcgpu_run_set_nuts_transition", "mcmcgpu_run_fetch_nuts_stats",
]

_lib = None


def lib():
    """Load libmcmcgpu.so; raises (no fallback) if it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise MCMCGPUError(E_CUDA, f"{LIB_PATH} not found: build it with `python __graft_entry__.py build` "
                                       "(make -C mcmc.jl_b200/csrc); there is no CPU fallback")
        L = C.CDLL(LIB_PATH)
        dp, vp = C.POINTER(C.c_double), C.c_void_p
        L.mcmcgpu_abi_version.restype = C.c_int32
        L.mcmcgpu_last_error.restype = C.c_char_p
        L.mcmcgpu_init.argtypes = [C.c_int32, C.POINTER(vp)]
        L.mcmcgpu_destroy.argtypes = [vp]
        L.mcmcgpu_set_stream.argtypes = [vp, vp]
        L.mcmcgpu_set_option.argtypes = [vp, C.c_char_p, C.c_int64]
        L.mcmcgpu_comm_unique_id.argtypes = [vp]
        L.mcmcgpu_comm_init.argtypes = [vp, C.c_int32, C.c_int32, vp]
        L.mcmcgpu_model_create.argtypes = [vp, C.c_int32, C.c_int64, C.c_int64, dp, dp, dp, C.c_int32, C.c_int32,
                                           C.POINTER(vp)]
        L.mcmcgpu_model_create_device.argtypes = [vp, C.c_int32, C.c_int64, C.c_int64, vp, vp, dp, C.c_int32, C.c_int32,
                                                  C.POINTER(vp)]
        L.mcmcgpu_model_destroy.argtypes = [vp]
        L.mcmcgpu_logtarget_grad.argtypes = [vp, dp, C.c_int64, dp, dp]
        L.mcmcgpu_run_chains.argtypes = [vp, C.POINTER(SamplerCfg), C.POINTER(RunnerCfg), dp, dp, dp, dp, dp, dp,
                                         C.POINTER(C.c_uint8), dp, C.POINTER(RunInfo)]
        L.mcmcgpu_run_create.argtypes = [vp, C.POINTER(SamplerCfg), C.POINTER(RunnerCfg), dp, dp, dp, dp,
                                         C.POINTER(vp)]
        L.mcmcgpu_run_execute.argtypes = [vp, C.POINTER(RunInfo)]
        L.mcmcgpu_run_execute_steps.argtypes = [vp, C.c_int64, C.POINTER(RunInfo)]
        L.mcmcgpu_run_set_state.argtypes = [vp, C.c_int64, dp, dp, dp]
        L.mcmcgpu_run_get_state.argtypes = [vp, dp, dp, dp, dp]
        L.mcmcgpu_run_set_metric.argtypes = [vp, dp, C.c_int32]
        L.mcmcgpu_run_set_metric_adaptation.argtypes = [vp, C.c_int64, C.c_int64, C.c_int64]
        L.mcmcgpu_run_get_metric.argtypes = [vp, dp]
        L.mcmcgpu_run_set_dense_metric.argtypes = [vp, dp, C.c_int32]
        L.mcmcgpu_run_get_dense_metric.argtypes = [vp, dp]
        L.mcmcgpu_run_set_nuts_transition.argtypes = [vp, C.c_int32]
        L.mcmcgpu_run_fetch_nuts_stats.argtypes = [vp, dp, dp, C.POINTER(C.c_uint8)]
        L.mcmcgpu_run_fetch.argtypes = [vp, dp, dp, C.POINTER(C.c_uint8), dp]
        L.mcmcgpu_run_fetch_rb.argtypes = [vp, dp]
        L.mcmcgpu_run_fetch_diag.argtypes = [vp, dp, C.POINTER(C.c_int64)]
        L.mcmcgpu_run_stats.argtypes = [vp, C.c_int32, C.c_int64, C.c_int64, dp, dp, dp, dp, dp, dp]
        L.mcmcgpu_run_destroy.argtypes = [vp]
        L.mcmcgpu_stats.argtypes = [vp, dp, C.c_int64, C.c_int64, C.c_int64, C.c_int32, C.c_int64, C.c_int64,
                                    dp, dp, dp, dp, dp]
        L.mcmcgpu_run_seqmc.argtypes = [vp, C.c_int32, C.c_int64, C.c_int32, dp, C.POINTER(SamplerCfg), C.c_int64, C.c_int64,
                                        C.c_double, C.c_int64, dp, C.c_uint64, dp, dp, dp, dp, dp, C.POINTER(C.c_int64),
                                        C.POINTER(RunInfo)]
        L.mcmcgpu_run_seqmc_models.argtypes = [vp, C.c_int32, C.POINTER(vp), C.POINTER(SamplerCfg), C.c_int64, C.c_int64, C.c_double,
                                               C.c_int64, dp, C.c_uint64, dp, dp, dp, dp, dp, C.POINTER(C.c_int64), C.POINTER(RunInfo)]
        L.mcmcgpu_run_serialtemp_models.argtypes = [vp, C.c_int32, C.POINTER(vp), C.POINTER(SamplerCfg), C.c_int64, C.c_int64, C.c_int64,
                                                    C.c_int64, C.c_int64, dp, C.c_uint64, dp, dp, dp, dp, dp, C.POINTER(C.c_int32),
                                                    C.POINTER(RunInfo)]
        L.mcmcgpu_run_serialtemp.argtypes = [vp, C.c_int32, C.c_int64, C.c_int32, dp, C.POINTER(SamplerCfg), C.c_int64, C.c_int64,
                                             C.c_int64, C.c_int64, dp, C.c_uint64, dp, dp, dp, dp, dp, C.POINTER(C.c_int32),
                                             C.POINTER(RunInfo)]
        L.mcmcgpu_run_zv.argtypes = [vp, C.c_int32, dp, dp]
        L.mcmcgpu_zv.argtypes = [vp, dp, dp, C.c_int64, C.c_int64, C.c_int64, C.c_int32, dp, dp]
        L.mcmcgpu_philox_draws.argtypes = [vp, C.c_uint64, C.c_int64, C.c_int64, C.c_int64, C.c_int64, dp, dp]
        for n in EXPORTS:
            if n not in ("mcmcgpu_last_error",):
                getattr(L, n).restype = C.c_int32
        _lib = L
    return _lib


def check(rc):
    if rc != OK:
        raise MCMCGPUError(rc, lib().mcmcgpu_last_error().decode())


def dptr(a):
    return None if a is None else a.ctypes.data_as(C.POINTER(C.c_double))


def f64(a, order="C"):
    return None if a is None else np.require(a, dtype=np.float64, requirements=["C" if order == "C" else "F", "A"])


def _destroy(fn_name, handle, _parent):
    # `_parent` only keeps the owning object (context / model) alive until this handle has been released
    getattr(lib(), fn_name)(C.c_void_p(handle))


class _Owned:
    """Lifetime of a library handle: freed by close(), by `with`, or when the Python object is collected -- always
    children first (a run keeps its model alive, a model its context; closing a parent closes its live children)."""
    h = None

    def _own(self, fn_name, parent):
        self._children = weakref.WeakSet()
        self._fin = weakref.finalize(self, _destroy, fn_name, self.h.value, parent)
        if parent is not None:
            parent._children.add(self)

    def close(self):
        if self.h is not None:
            for ch in list(self._children):
                ch.close()
            self.h = None
            self._fin()

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()


class Context(_Owned):
    def __init__(self, device=-1):
        h = C.c_void_p()
        check(lib().mcmcgpu_init(device, C.byref(h)))
        self.h = h
        self._own("mcmcgpu_destroy", None)

    def set_stream(self, stream_ptr):
        check(lib().mcmcgpu_set_stream(self.h, C.c_void_p(stream_ptr) if stream_ptr else None))

    def set_option(self, key, value):
        check(lib().mcmcgpu_set_option(self.h, key.encode(), int(value)))

    @staticmethod
    def comm_unique_id():
        buf = (C.c_char * 128)()
        check(lib().mcmcgpu_comm_unique_id(buf))
        return bytes(buf)

    def comm_init(self, rank, nranks, uid):
        buf = (C.c_char * 128).from_buffer_copy(uid)
        check(lib().mcmcgpu_comm_init(self.h, rank, nranks, buf))

    def philox_draws(self, seed, chain_offset, nchains, d, last):
        z = np.empty((nchains, last + 1, d))
        u = np.empty((nchains, last + 1))
        check(lib().mcmcgpu_philox_draws(self.h, seed, chain_offset, nchains, d, last, dptr(z), dptr(u)))
        return z, u

    def stats(self, samples, vtype="imse", maxlag=-1, batchlen=100, want=("mean", "var_iid", "var", "ess", "actime")):
        """samples: (C, S, d) array (chain-major, the layout run_chains fills)."""
        s = f64(samples)
        Cn, S, d = s.shape
        outs = {k: (np.empty((Cn, d)) if k in want else None) for k in ("mean", "var_iid", "var", "ess", "actime")}
        if vtype == "iid":
            outs["ess"] = outs["actime"] = None
        check(lib().mcmcgpu_stats(self.h, dptr(s), S, d, Cn, VTYPE[vtype], maxlag, batchlen, dptr(outs["mean"]),
                                  dptr(outs["var_iid"]), dptr(outs["var"]), dptr(outs["ess"]), dptr(outs["actime"])))
        return {k: v for k, v in outs.items() if v is not None}

    def zv(self, samples, grads, order=1, want_chain=True):
        """samples, grads: (C, S, d).  Returns (zvchain (C, S, d) or None, a (C, k, d)) -- linearZv / quadraticZv per chain."""
        s, g = f64(samples), f64(grads)
        Cn, S, d = s.shape
        k = d if order == 1 else d * (d + 3) // 2
        zv = np.empty((Cn, S, d)) if want_chain else None
        a = np.empty((Cn, k, d))
        check(lib().mcmcgpu_zv(self.h, dptr(s), dptr(g), S, d, Cn, order, dptr(zv), dptr(a)))
        return zv, a

    def _tasks(self, hypers, samplers):
        hy = np.zeros((len(samplers), 4))
        for t, h in enumerate(hypers):
            hy[t, :len(h)] = h
        return hy, (SamplerCfg * len(samplers))(*samplers)

    def run_seqmc(self, family, d, hypers, samplers, steps, burnin, trigger, particles, seed=0, normals=None, uniforms=None,
                  res_uniforms=None):
        """particles (npart, d); injected draws: normals (steps, nt, npart, d), uniforms / res_uniforms (steps, nt, npart).
        Returns dict(samples ((steps-burnin)*npart, d), weights, n_resamples, info)."""
        particles = f64(particles)
        npart, nt = particles.shape[0], len(samplers)
        hy, sc = self._tasks(hypers, samplers)
        S = max(steps - burnin, 0) * npart
        samples, weights = np.empty((S, d)), np.empty(S)
        nres, info = C.c_int64(0), RunInfo()
        zn, un, ru = f64(normals), f64(uniforms), f64(res_uniforms)
        check(lib().mcmcgpu_run_seqmc(self.h, FAM[family], d, nt, dptr(hy), sc, steps, burnin, trigger, npart, dptr(particles), seed,
                                      dptr(zn), dptr(un), dptr(ru), dptr(samples), dptr(weights), C.byref(nres), C.byref(info)))
        return dict(samples=samples, weights=weights, n_resamples=nres.value, info=info.as_dict())

    def run_seqmc_models(self, models, samplers, steps, burnin, trigger, particles, seed=0, normals=None, uniforms=None,
                         res_uniforms=None):
        """SeqMC over DeviceModels of this context (any family, any d): task t = (models[t], samplers[t]).  With a
        communicator the population is sharded: `particles` is this rank's share, injected draws are the GLOBAL arrays."""
        particles = f64(particles)
        npart, nt, d = particles.shape[0], len(samplers), models[0].d
        mh = (C.c_void_p * nt)(*[m.h for m in models])
        sc = (SamplerCfg * nt)(*samplers)
        S = max(steps - burnin, 0) * npart
        samples, weights = np.empty((S, d)), np.empty(S)
        nres, info = C.c_int64(0), RunInfo()
        zn, un, ru = f64(normals), f64(uniforms), f64(res_uniforms)
        check(lib().mcmcgpu_run_seqmc_models(self.h, nt, mh, sc, steps, burnin, trigger, npart, dptr(particles), seed, dptr(zn), dptr(un),
                                             dptr(ru), dptr(samples), dptr(weights), C.byref(nres), C.byref(info)))
        return dict(samples=samples, weights=weights, n_resamples=nres.value, info=info.as_dict())

    def run_serialtemp_models(self, models, samplers, steps, burnin, swap_period, nrep, inits, seed=0, rep_offset=0, normals=None,
                              uniforms=None, pick=None, swap=None):
        """SerialTempMC over DeviceModels of this context (any family, any d); arrays as run_serialtemp.  rep_offset: global id
        of this context's first replica (replicas shard over GPUs without communication)."""
        inits = f64(inits)
        nt, d = len(samplers), models[0].d
        mh = (C.c_void_p * nt)(*[m.h for m in models])
        sc = (SamplerCfg * nt)(*samplers)
        S = max(steps - burnin, 0)
        samples, at, info = np.empty((nrep, S, d)), np.empty((nrep, S), dtype=np.int32), RunInfo()
        zn, un, pk, sw = f64(normals), f64(uniforms), f64(pick), f64(swap)
        check(lib().mcmcgpu_run_serialtemp_models(self.h, nt, mh, sc, steps, burnin, swap_period, nrep, rep_offset, dptr(inits), seed,
                                                  dptr(zn), dptr(un), dptr(pk), dptr(sw), dptr(samples),
                                                  at.ctypes.data_as(C.POINTER(C.c_int32)), C.byref(info)))
        return dict(samples=samples, at=at, info=info.as_dict())

    def run_serialtemp(self, family, d, hypers, samplers, steps, burnin, swap_period, nrep, inits, seed=0, normals=None,
                       uniforms=None, pick=None, swap=None):
        """inits (nt, d); injected draws per replica: normals (nrep, steps+2, d), uniforms (nrep, steps+2), pick / swap
        (nrep, steps+1).  Returns dict(samples (nrep, steps-burnin, d), at (nrep, steps-burnin), info)."""
        inits = f64(inits)
        nt = len(samplers)
        hy, sc = self._tasks(hypers, samplers)
        S = max(steps - burnin, 0)
        samples, at, info = np.empty((nrep, S, d)), np.empty((nrep, S), dtype=np.int32), RunInfo()
        zn, un, pk, sw = f64(normals), f64(uniforms), f64(pick), f64(swap)
        check(lib().mcmcgpu_run_serialtemp(self.h, FAM[family], d, nt, dptr(hy), sc, steps, burnin, swap_period, nrep, dptr(inits), seed,
                                           dptr(zn), dptr(un), dptr(pk), dptr(sw), dptr(samples),
                                           at.ctypes.data_as(C.POINTER(C.c_int32)), C.byref(info)))
        return dict(samples=samples, at=at, info=info.as_dict())



class DeviceModel(_Owned):
    def __init__(self, ctx, family, d, X=None, y=None, hyper=(), row_sharded=False):
        self.ctx, self.family, self.d = ctx, family, int(d)
        Xf = None if X is None else np.asfortranarray(X, dtype=np.float64)
        yf = None if y is None else np.ascontiguousarray(y, dtype=np.float64)
        N = 0 if (Xf is None and yf is None) else (len(yf) if yf is not None else Xf.shape[0])
        if Xf is not None and Xf.shape != (N, self.d):
            raise MCMCGPUError(E_ARG, f"X must be N x d = {(N, self.d)}, got {Xf.shape}")
        hy = np.asarray(hyper, dtype=np.float64)
        h = C.c_void_p()
        check(lib().mcmcgpu_model_create(ctx.h, FAM[family], N, self.d, dptr(Xf), dptr(yf), dptr(hy) if len(hy) else None,
                                         len(hy), 1 if row_sharded else 0, C.byref(h)))
        self.h, self.N = h, N
        self._own("mcmcgpu_model_destroy", ctx)

    @classmethod
    def from_device(cls, ctx, family, N, d, X_ptr, y_ptr, hyper=(), row_sharded=False):
        """X_ptr / y_ptr: device addresses (e.g. torch tensor .data_ptr()) of an N x d column-major X and y."""
        self = cls.__new__(cls)
        self.ctx, self.family, self.d, self.N = ctx, family, int(d), int(N)
        hy = np.asarray(hyper, dtype=np.float64)
        h = C.c_void_p()
        check(lib().mcmcgpu_model_create_device(ctx.h, FAM[family], int(N), int(d), C.c_void_p(X_ptr), C.c_void_p(y_ptr),
                                                dptr(hy) if len(hy) else None, len(hy), 1 if row_sharded else 0, C.byref(h)))
        self.h = h
        self._own("mcmcgpu_model_destroy", ctx)
        return self

    def logtarget_grad(self, B, grad=True):
        """B: (C, d) parameter vectors. Returns lt (C,), grad (C, d) or None."""
        B = f64(np.atleast_2d(B))
        Cn = B.shape[0]
        lt = np.empty(Cn)
        g = np.empty((Cn, self.d)) if grad else None
        check(lib().mcmcgpu_logtarget_grad(self.h, dptr(B), Cn, dptr(lt), dptr(g)))
        return lt, g



def sampler_cfg(kind, scale=1.0, nleaps=10, rate=0.65, len=2.0, shrinkage=0.05, t0=10.0, step=0.75, max_leaps=0,
                tuner=None):
    s = SamplerCfg()
    s.kind, s.scale, s.nleaps = KIND[kind], scale, nleaps
    s.rate, s.len, s.shrinkage, s.t0, s.step, s.max_leaps = rate, len, shrinkage, t0, step, max_leaps
    if tuner is not None:
        s.tuner_on = 1
        s.adapt_step = tuner.get("adapt_step", 100)
        s.max_step = tuner.get("max_step", 200)
        s.target_path = tuner.get("target_path", 1.0)
        s.target_rate = tuner["target_rate"]
    return s


class DeviceRun(_Owned):
    """Split-form run: inputs resident in HBM after construction; execute() may be timed alone."""

    def __init__(self, model, scfg, rng, nchains, init, scale=None, seed=0, chain_offset=0, normals=None, uniforms=None,
                 store_grad=True, store_logtarget=True, engine="auto", store_rb=False, stream_stats=False, stream_batchlen=0):
        first, step, last = rng
        self.model, self.d = model, model.d
        r = RunnerCfg()
        r.first, r.step, r.last, r.nchains, r.chain_offset, r.seed = first, step, last, nchains, chain_offset, seed
        init = f64(init)
        r.init_per_chain = 1 if init.ndim == 2 else 0
        if init.ndim == 2 and init.shape != (nchains, self.d):
            raise MCMCGPUError(E_ARG, "init must be (d,) or (nchains, d)")
        r.store_grad, r.store_logtarget, r.engine = int(store_grad), int(store_logtarget), ENGINE[engine]
        r.store_rb = int(store_rb)
        r.stream_stats, r.stream_batchlen = int(stream_stats), int(stream_batchlen)
        self.streaming = bool(stream_stats)
        if stream_stats:
            store_grad = store_logtarget = False
            r.store_grad = r.store_logtarget = 0
        self.S = 0 if (step < 1 or last < first) else (last - first) // step + 1
        self.C = nchains
        self.store_grad, self.store_logtarget = store_grad, store_logtarget
        self.has_diag = bool(scfg.kind in (KIND["HMCDA"], KIND["RAM"], KIND["NUTS"]) or scfg.tuner_on)
        sc = None if scale is None else f64(np.broadcast_to(scale, (self.d,)).copy())
        zn = f64(normals)
        un = f64(uniforms)
        if zn is not None and (zn.shape != (nchains, last + 1, self.d) or un.shape != (nchains, last + 1)):
            raise MCMCGPUError(E_ARG, "normals must be (nchains, last+1, d) and uniforms (nchains, last+1)")
        h = C.c_void_p()
        check(lib().mcmcgpu_run_create(model.h, C.byref(scfg), C.byref(r), dptr(init), dptr(sc), dptr(zn), dptr(un),
                                       C.byref(h)))
        self.h = h
        self._own("mcmcgpu_run_destroy", model)
        self.info = None

    def execute(self):
        info = RunInfo()
        rc = lib().mcmcgpu_run_execute(self.h, C.byref(info))
        self.info = info.as_dict()
        check(rc)
        return self.info

    def execute_steps(self, nsteps):
        info = RunInfo()
        rc = lib().mcmcgpu_run_execute_steps(self.h, int(nsteps), C.byref(info))
        self.info = info.as_dict()
        check(rc)
        return self.info

    def set_state(self, step0, leapstep=None, dual_leapstep=None, dualH=None):
        a, b, c = f64(leapstep), f64(dual_leapstep), f64(dualH)
        check(lib().mcmcgpu_run_set_state(self.h, int(step0), dptr(a), dptr(b), dptr(c)))

    def get_state(self):
        pars = np.empty((self.C, self.d))
        ls, du, dh = np.empty(self.C), np.empty(self.C), np.empty(self.C)
        check(lib().mcmcgpu_run_get_state(self.h, dptr(pars), dptr(ls), dptr(du), dptr(dh)))
        return dict(pars=pars, leapstep=ls, dual_leapstep=du, dualH=dh)

    def set_metric(self, inv_metric):
        """NUTS: diagonal inverse metric, (d,) for every chain or (nchains, d) per chain"""
        m = f64(inv_metric)
        if m.shape not in ((self.d,), (self.C, self.d)):
            raise MCMCGPUError(E_ARG, f"inv_metric must be (d,) or (nchains, d) = {(self.C, self.d)}, got {m.shape}")
        check(lib().mcmcgpu_run_set_metric(self.h, dptr(m), 1 if m.ndim == 2 else 0))

    def set_metric_adaptation(self, init_buffer=75, term_buffer=50, window=25):
        check(lib().mcmcgpu_run_set_metric_adaptation(self.h, int(init_buffer), int(term_buffer), int(window)))

    def get_metric(self):
        """(nchains, d) current inverse metric"""
        out = np.empty((self.C, self.d))
        check(lib().mcmcgpu_run_get_metric(self.h, dptr(out)))
        return out

    def set_dense_metric(self, inv_metric=None):
        """NUTS: dense inverse metric, (d, d) for every chain or (nchains, d, d) per chain; None = the identity"""
        if inv_metric is None:
            check(lib().mcmcgpu_run_set_dense_metric(self.h, None, 0))
            return
        m = f64(inv_metric)
        d = self.d
        if m.shape not in ((d, d), (self.C, d, d)):
            raise MCMCGPUError(E_ARG, f"inv_metric must be (d, d) or (nchains, d, d) = {(self.C, d, d)}, got {m.shape}")
        # (c, i, j) in C order is element (j, i) column-major; the library requires exact symmetry, so the two agree
        check(lib().mcmcgpu_run_set_dense_metric(self.h, dptr(m), 1 if m.ndim == 3 else 0))

    def get_dense_metric(self):
        """(nchains, d, d) current dense inverse metric"""
        out = np.empty((self.C, self.d, self.d))
        check(lib().mcmcgpu_run_get_dense_metric(self.h, dptr(out)))
        return np.ascontiguousarray(out.transpose(0, 2, 1))               # column-major blocks -> [c, i, j]

    def set_nuts_transition(self, transition):
        """NUTS, before the first execute: NUTS_SLICE (the default) or NUTS_MULTINOMIAL (Stan's transition)"""
        check(lib().mcmcgpu_run_set_nuts_transition(self.h, int(transition)))

    def fetch_nuts_stats(self):
        """multinomial NUTS: (nchains, S) accept_stat, energy and divergent (bool) of the kept steps"""
        acc, en = np.empty((self.C, self.S)), np.empty((self.C, self.S))
        div = np.empty((self.C, self.S), dtype=np.uint8)
        check(lib().mcmcgpu_run_fetch_nuts_stats(self.h, dptr(acc), dptr(en), div.ctypes.data_as(C.POINTER(C.c_uint8))))
        return dict(accept_stat=acc, energy=en, divergent=div.astype(bool))

    def fetch(self, samples=True, grads=None, accept=True, logtarget=None, out=None):
        grads = self.store_grad if grads is None else grads
        logtarget = self.store_logtarget if logtarget is None else logtarget
        out = out or {}
        res = {}
        res["samples"] = out.get("samples", np.empty((self.C, self.S, self.d))) if samples else None
        res["grads"] = out.get("grads", np.empty((self.C, self.S, self.d))) if grads else None
        res["accept"] = out.get("accept", np.empty((self.C, self.S), dtype=np.uint8)) if accept else None
        res["logtarget"] = out.get("logtarget", np.empty((self.C, self.S))) if logtarget else None
        acc = res["accept"]
        check(lib().mcmcgpu_run_fetch(self.h, dptr(res["samples"]), dptr(res["grads"]),
                                      None if acc is None else acc.ctypes.data_as(C.POINTER(C.c_uint8)),
                                      dptr(res["logtarget"])))
        return {k: v for k, v in res.items() if v is not None}

    def fetch_rb(self):
        rb = np.empty((self.C, self.S, self.d))
        check(lib().mcmcgpu_run_fetch_rb(self.h, dptr(rb)))
        return rb

    def fetch_diag(self):
        eps = np.empty((self.C, self.S))
        nl = np.empty((self.C, self.S), dtype=np.int64)
        check(lib().mcmcgpu_run_fetch_diag(self.h, dptr(eps), nl.ctypes.data_as(C.POINTER(C.c_int64))))
        return eps, nl

    def stats(self, vtype="imse", maxlag=-1, batchlen=100):
        names = ["mean", "var_iid", "var", "ess", "actime"]
        outs = {k: np.empty((self.C, self.d)) for k in names}
        if vtype == "iid":
            outs["ess"] = outs["actime"] = None
        rate = np.empty(self.C)
        check(lib().mcmcgpu_run_stats(self.h, VTYPE[vtype], maxlag, batchlen, dptr(outs["mean"]), dptr(outs["var_iid"]),
                                      dptr(outs["var"]), dptr(outs["ess"]), dptr(outs["actime"]), dptr(rate)))
        outs["accept_rate"] = rate
        return {k: v for k, v in outs.items() if v is not None}

    def zv(self, order=1, want_chain=True):
        k = self.d if order == 1 else self.d * (self.d + 3) // 2
        zv = np.empty((self.C, self.S, self.d)) if want_chain else None
        a = np.empty((self.C, k, self.d))
        check(lib().mcmcgpu_run_zv(self.h, order, dptr(zv), dptr(a)))
        return zv, a

