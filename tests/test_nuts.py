"""The No-U-Turn sampler (MCMCGPU_NUTS, mj.NUTS): the CPU restatement tests/nuts_oracle.c against exact targets and its
own invariants, the host API, and on the GPU the wave engine's nuts_kernel against the restatement, bit for bit on the
closed-form families and within the suite's draw-matched tolerances on the regression families."""
import ctypes as C
import math
import os
import subprocess
import tempfile
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest
from scipy import stats as sst

from conftest import make_regression, ou_series

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LEAF, TREE = 0x40000000, 0x80000000


# ---- the CPU restatement -----------------------------------------------------------------------------------------------
@pytest.fixture(scope="session")
def N(O):
    """tests/nuts_oracle.c compiled with the oracle (same flags as oracle/Makefile) into a temporary library"""
    tmp = tempfile.mkdtemp(prefix="nuts_oracle_")
    so = os.path.join(tmp, "libnuts_oracle.so")
    subprocess.check_call(["gcc", "-O3", "-std=gnu99", "-ffp-contract=off", "-fPIC", "-shared", "-o", so,
                           os.path.join(ROOT, "tests", "nuts_oracle.c"), os.path.join(ROOT, "oracle", "mcmc_oracle.c"), "-lm"])
    L = C.CDLL(so)
    dp, i64p = C.POINTER(C.c_double), C.POINTER(C.c_int64)
    L.orc_run_nuts.restype = C.c_int32
    L.orc_run_nuts.argtypes = [C.POINTER(O._Model), C.POINTER(O._Sampler), C.POINTER(O._Range), dp, C.c_uint64, C.c_uint64, dp,
                               dp, dp, C.POINTER(C.c_uint8), dp, dp, i64p, dp, i64p, i64p]
    L.orc_nuts_slot_uniform.restype = C.c_double
    L.orc_nuts_slot_uniform.argtypes = [C.c_uint64, C.c_uint64, C.c_uint32, C.c_uint32]
    return L


def run_nuts(O, N, om, rngt, init, seed, chain, maxd=10, rate=0.6, shrinkage=0.05, t0=10.0, step=0.75, force_eps=None,
             start_step=0, da_state=None, normals=None):
    """one oracle chain; rngt = (first, step, last); normals (last+1, d) or None (orc_draw_normals)"""
    first, stp, last = rngt
    d = om.d
    S = (last - first) // stp + 1
    smp = O.sampler("HMCDA", nleaps=maxd, rate=rate, shrinkage=shrinkage, t0=t0, step=step, force_eps=force_eps,
                    start_step=start_step, da_state=da_state)
    init = np.ascontiguousarray(np.broadcast_to(init, (d,)), dtype=np.float64)
    zn = None if normals is None else np.ascontiguousarray(normals[:last + 1], dtype=np.float64)
    out = dict(samples=np.full((S, d), np.nan), grads=np.full((S, d), np.nan), accept=np.zeros(S, np.uint8),
               logtarget=np.full(S, np.nan), eps=np.full(S, np.nan), leaps=np.zeros(S, np.int64), alpha=np.full(S, np.nan),
               ndoublings=np.zeros(S, np.int64))
    nev = C.c_int64(0)
    p = lambda a: a.ctypes.data_as(C.POINTER(C.c_double))
    rc = N.orc_run_nuts(C.byref(om._c), C.byref(smp), C.byref(O._Range(first, stp, last)), p(init), seed, chain,
                        None if zn is None else p(zn), p(out["samples"]), p(out["grads"]),
                        out["accept"].ctypes.data_as(C.POINTER(C.c_uint8)), p(out["logtarget"]), p(out["eps"]),
                        out["leaps"].ctypes.data_as(C.POINTER(C.c_int64)), p(out["alpha"]),
                        out["ndoublings"].ctypes.data_as(C.POINTER(C.c_int64)), C.byref(nev))
    out["rc"], out["n_grad_evals"] = rc, nev.value
    return out


def run_many(fn, jobs):
    with ThreadPoolExecutor(max_workers=min(32, os.cpu_count() or 1)) as ex:    # ctypes releases the GIL
        return list(ex.map(fn, jobs))


def u01(o):
    b = ((o[0] << 21) ^ (o[1] >> 11)) & ((1 << 53) - 1)
    return (b + 0.5) / 2.0 ** 53


def test_slot_uniforms_are_the_documented_philox_counters(O, N):
    seed, chain = (1 << 40) + 17, (1 << 33) + 5
    key = (seed & 0xFFFFFFFF, seed >> 32)
    for step in (1, 7, 123456):
        for block in (LEAF, LEAF + 1022, TREE, TREE + 1, TREE + 19, 0xFFFFFFFF):
            ref = u01(O.philox((chain & 0xFFFFFFFF, chain >> 32, step, block), key))
            assert N.orc_nuts_slot_uniform(seed, chain, step, block) == ref
        assert N.orc_nuts_slot_uniform(seed, chain, step, 0xFFFFFFFF) == O.draw_uniform(seed, chain, step)
    # no slot collides with a normal block (d <= 200: blocks 0..99) or with the Metropolis block
    normal = set(range(100))
    leaves = set(range(LEAF, LEAF + 2 ** 10 - 1))
    trees = set(range(TREE, TREE + 2 * 10))
    assert not (normal & leaves) and not (normal & trees) and not (leaves & trees) and 0xFFFFFFFF not in leaves | trees


@pytest.mark.parametrize("fam,d,hy,maxd", [("normal_dsl", 5, (1.0, 2.0), 10), ("normal_fn", 3, (), 3), ("abs_normal", 2, (1.0, 0.5), 4)])
def test_oracle_invariants(O, N, fam, d, hy, maxd):
    om = O.Model(fam, d, hyper=hy)
    rngt = (1, 1, 120)
    res = run_many(lambda c: run_nuts(O, N, om, rngt, np.ones(d), 11, c, maxd=maxd, rate=0.8), range(64))
    for r in res:
        assert r["rc"] == 0
        assert np.all(r["leaps"] >= 1) and np.all(r["leaps"] <= 2 ** maxd - 1)
        assert np.array_equal(np.floor(np.log2(r["leaps"])).astype(np.int64) + 1, r["ndoublings"])
        stay = r["accept"][1:] == 0
        assert np.array_equal(r["samples"][1:][stay], r["samples"][:-1][stay])
        assert np.array_equal(r["logtarget"][1:][stay], r["logtarget"][:-1][stay])
        assert r["n_grad_evals"] == 1 + r["leaps"].sum()
        assert np.all((r["alpha"] >= 0) & (r["alpha"] <= 1))
    assert np.mean([r["accept"].mean() for r in res]) > 0.2              # the trees move (eps = 1, no burn-in)


def _check_exact(x, mean, sd, label):
    """x (C, d) independent draws of N(mean, sd^2) per coordinate: KS (Bonferroni over d) and moments within 5 SE"""
    Cn, d = x.shape
    for j in range(d):
        p = sst.kstest(x[:, j], sst.norm(mean, sd).cdf).pvalue
        assert p * d > 1e-4, (label, j, p)
        m = x[:, j].mean()
        assert abs(m - mean) < 5 * x[:, j].std(ddof=1) / math.sqrt(Cn), (label, j, m)
        dev2 = (x[:, j] - m) ** 2
        assert abs(dev2.mean() - sd * sd) < 5 * dev2.std(ddof=1) / math.sqrt(Cn), (label, j, dev2.mean())


TARGETS = [("normal_dsl", 1, (1.0, 2.0), 1.0, 2.0), ("normal_dsl", 5, (1.0, 2.0), 1.0, 2.0), ("normal_fn", 4, (), 0.0, math.sqrt(0.5))]


@pytest.mark.parametrize("fam,d,hy,mu,sd", TARGETS, ids=lambda t: str(t))
def test_oracle_samples_exact_targets(O, N, fam, d, hy, mu, sd):
    om = O.Model(fam, d, hyper=hy)
    B, L, Cn = 100, 130, 2000
    res = run_many(lambda c: run_nuts(O, N, om, (B + 1, 1, L), np.full(d, 3.0), 2024, c), range(Cn))
    _check_exact(np.array([r["samples"][-1] for r in res]), mu, sd, fam)
    # the dual averaging reaches its target: the mean acceptance statistic of the post-burn-in steps
    a = np.mean([r["alpha"] for r in res])
    assert 0.55 < a < 0.8, a


# ---- host API --------------------------------------------------------------------------------------------------------
def test_nuts_constructor_and_config():
    import mcmc_jl_b200 as mj
    s = mj.NUTS()
    assert (s.rate, s.maxdoublings, s.shrinkage, s.t0, s.step) == (0.6, 10, 0.05, 10.0, 0.75)
    assert s.needs_gradient
    for bad in (lambda: mj.NUTS(rate=1.5), lambda: mj.NUTS(rate=0.0), lambda: mj.NUTS(maxdoublings=0), lambda: mj.NUTS(maxdoublings=11),
                lambda: mj.NUTS(maxdoublings=2.5), lambda: mj.NUTS(shrinkage=0.0), lambda: mj.NUTS(t0=-1.0)):
        with pytest.raises(AssertionError):
            bad()
    cfg = mj.NUTS(rate=0.7, maxdoublings=6, shrinkage=0.1, t0=5.0, step=0.5)._cfg()
    assert (cfg.kind, cfg.nleaps, cfg.rate, cfg.shrinkage, cfg.t0, cfg.step, cfg.tuner_on) == (5, 6, 0.7, 0.1, 5.0, 0.5, 0)


# ---- GPU: the kernel against the restatement -----------------------------------------------------------------------
def _device_and_oracle(O, N, capi, ctx, fam, d, X, y, hy, C, rngt, init, seed, maxd=10, s0=0, eps0=None, chains=None, run_kw=None):
    """Philox-mode device run and oracle chains replaying it with the device's normals.  s0 > 0: start after step s0 with
    the per-chain step size eps0 (set_state), burn-in over, so every kept step size is forced on the oracle one step ahead."""
    first, _, last = rngt
    om, dm = O.Model(fam, d, X, y, hy), capi.DeviceModel(ctx, fam, d, X, y, hy)
    run = capi.DeviceRun(dm, capi.sampler_cfg("NUTS", nleaps=maxd, rate=0.6), rngt, C, init, seed=seed, engine="wave", **(run_kw or {}))
    if s0:
        run.set_state(s0, eps0, eps0, np.zeros(C))
    info = run.execute(); out = run.fetch(); eps, leaps = run.fetch_diag()
    run.close(); dm.close()
    zn, _ = ctx.philox_draws(seed, 0, C, d, last)
    chains = range(C) if chains is None else chains
    ini = lambda c: init[c] if np.ndim(init) == 2 else init

    def one(c):
        kw = dict(maxd=maxd, normals=zn[c])
        if s0:
            kw.update(start_step=s0, da_state=[eps0[c], eps0[c], 0.0], force_eps=np.concatenate([np.full(s0 + 1, np.nan), eps[c]]))
        return c, run_nuts(O, N, om, rngt, ini(c), seed, c, **kw)
    refs = dict(run_many(one, list(chains)))
    return out, eps, leaps, refs, info


CLOSED = [("normal_fn", d, ()) for d in (1, 3, 9, 33)] + [("normal_dsl", d, (1.0, 2.0)) for d in (1, 3, 9, 33)] + \
         [("abs_normal", d, (1.0, 0.5)) for d in (1, 3, 9, 33)] + [("ou", 3, (100.0, 2.0, 20.0))]


@pytest.mark.gpu
@pytest.mark.parametrize("fam,d,hy", CLOSED, ids=lambda c: str(c))
def test_closed_form_parity_bit_exact(O, N, capi, ctx, fam, d, hy):
    C, s0, K = 70, 50, 25
    r = np.random.default_rng(d)
    if fam == "ou":
        y, init, maxd = ou_series(300, 4), np.array([20.0, 0.1, 10.0]), 7
        eps0 = 0.002 * np.exp(0.3 * r.standard_normal(C))
    else:
        y, init, maxd = None, 0.5 + r.standard_normal((C, d)), 10
        eps0 = {"normal_fn": 0.8, "normal_dsl": 1.2, "abs_normal": 0.25}[fam] * np.exp(0.4 * r.standard_normal(C))
    out, eps, leaps, refs, info = _device_and_oracle(O, N, capi, ctx, fam, d, None, y, hy, C, (s0 + 1, 1, s0 + K), init, 7, maxd, s0, eps0)
    for c in range(C):
        ref = refs[c]
        assert ref["rc"] == 0
        assert np.array_equal(ref["accept"], out["accept"][c]), c
        assert np.array_equal(ref["leaps"], leaps[c]), c
        assert np.array_equal(ref["eps"], eps[c]), c
        if fam == "ou":     # the OU likelihood itself agrees with the oracle to 1e-10, not bitwise (as for every sampler)
            assert np.allclose(ref["samples"], out["samples"][c], rtol=1e-10, atol=0), c
            assert np.allclose(ref["logtarget"], out["logtarget"][c], rtol=1e-10, atol=0), c
            continue
        assert np.array_equal(ref["samples"], out["samples"][c]), c
        assert np.array_equal(ref["logtarget"], out["logtarget"][c]), c
        assert np.array_equal(ref["grads"], out["grads"][c]), c
    assert info["n_grad_evals"] == C + int(leaps.sum())
    assert leaps.max() > 4 and out["accept"].mean() > 0.2                  # the trees are real


@pytest.mark.gpu
@pytest.mark.parametrize("burnin", (3, 12, 30))
def test_adaptation_parity(O, N, capi, ctx, burnin):
    """from eps = 1 with the dual averaging on: the step sizes (suite tolerance), leaps and decisions agree with the oracle"""
    d, C = 3, 64
    rngt = (burnin + 1, 1, burnin + 8)
    out, eps, leaps, refs, _ = _device_and_oracle(O, N, capi, ctx, "normal_dsl", d, None, None, (1.0, 2.0), C, rngt, np.ones(d), 3)
    for c in range(C):
        assert np.allclose(refs[c]["eps"], eps[c], rtol=1e-9, atol=0), c
        assert np.array_equal(refs[c]["leaps"], leaps[c]) and np.array_equal(refs[c]["accept"], out["accept"][c]), c
        assert np.allclose(refs[c]["samples"], out["samples"][c], rtol=1e-9, atol=1e-12), c


REGRESSION = [(f, d) for f in ("linear", "logistic", "probit") for d in (1, 20, 100, 200)]


@pytest.mark.gpu
@pytest.mark.parametrize("fam,d", REGRESSION, ids=lambda c: str(c))
def test_regression_parity(O, N, capi, ctx, fam, d):
    Nrows = 997                                                             # ragged: not a multiple of 32
    X, y, hy, b0 = make_regression(fam, Nrows, d, 5)
    ntiles = -(-Nrows // 32)
    s0, K = 40, 12
    r = np.random.default_rng(d)
    # step sizes of the adapted regime: the posterior sd is ~ 1 / sqrt(N) per coordinate
    base = (0.3 if fam == "probit" else 0.5) / math.sqrt(Nrows)
    gs = np.abs(X).sum(0)
    try:
        for C, splits in ((130, 1), (70, 3), (1, ntiles + 3)):
            ctx.set_option("force_splits", splits)
            init = b0 + 0.05 * r.standard_normal((C, d)) / math.sqrt(d)
            eps0 = base * np.exp(0.3 * r.standard_normal(C))
            chains = range(C) if d <= 10 else range(0, C, 5)
            out, eps, leaps, refs, info = _device_and_oracle(O, N, capi, ctx, fam, d, X, y, hy, C, (s0 + 1, 1, s0 + K), init, 9,
                                                             8, s0, eps0, chains)
            for c in chains:
                ref = refs[c]
                assert np.array_equal(ref["accept"], out["accept"][c]), (C, splits, c)
                assert np.array_equal(ref["leaps"], leaps[c]), (C, splits, c)
                assert np.allclose(ref["samples"], out["samples"][c], rtol=1e-9, atol=1e-12), (C, splits, c)
                assert np.allclose(ref["logtarget"], out["logtarget"][c], rtol=1e-11, atol=0), (C, splits, c)
                assert np.all(np.abs(ref["grads"] - out["grads"][c]) <= 1e-9 * gs), (C, splits, c)
            assert info["n_grad_evals"] == C + int(leaps.sum())
    finally:
        ctx.set_option("force_splits", 0)


# ---- GPU: statistical validity ----------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_many_chains_sample_normal_dsl(capi, ctx):
    d, C = 5, 16384
    dm = capi.DeviceModel(ctx, "normal_dsl", d, hyper=(1.0, 2.0))
    run = capi.DeviceRun(dm, capi.sampler_cfg("NUTS", nleaps=10), (201, 1, 260), C, np.full(d, 3.0), seed=31, store_grad=False)
    run.execute(); out = run.fetch(); eps, leaps = run.fetch_diag()
    _check_exact(out["samples"][:, -1], 1.0, 2.0, "normal_dsl")
    assert np.all(leaps >= 1) and np.all(leaps <= 1023)
    run.close(); dm.close()


@pytest.mark.gpu
def test_many_chains_sample_linear_posterior(capi, ctx):
    """linear regression with correlated columns against its closed-form Gaussian posterior"""
    d, Nr, C = 10, 300, 8192
    r = np.random.default_rng(8)
    A = np.eye(d) + 0.6 * np.tril(r.standard_normal((d, d)), -1)
    X = r.standard_normal((Nr, d)) @ A.T
    X[:, 0] = 1.0
    beta = r.standard_normal(d) / 2
    y = X @ beta + r.standard_normal(Nr)
    prec = X.T @ X + np.eye(d)                                              # noise sd 1, prior sd 1
    cov = np.linalg.inv(prec)
    mean = cov @ (X.T @ y)
    dm = capi.DeviceModel(ctx, "linear", d, X, y, (1.0, 1.0))
    run = capi.DeviceRun(dm, capi.sampler_cfg("NUTS", nleaps=10), (301, 1, 360), C, mean + 0.1, seed=5, store_grad=False, engine="wave")
    run.execute(); x = run.fetch()["samples"][:, -1]
    run.close(); dm.close()
    z = (x - mean) @ np.linalg.cholesky(prec)                              # whitened: iid N(0, 1) coordinates
    _check_exact(z, 0.0, 1.0, "linear")


# ---- GPU: bit-identity across execution paths ---------------------------------------------------------------------
def _path_run(capi, ctx, dm, C, rngt, init, seed, pieces=None, offset=0, nchains=None, state=None):
    run = capi.DeviceRun(dm, capi.sampler_cfg("NUTS", nleaps=8), rngt, nchains or C, init, seed=seed, chain_offset=offset, engine="wave")
    if state is not None:
        run.set_state(*state)
    infos = []
    if pieces:
        for p in pieces:
            infos.append(run.execute_steps(p))
    else:
        infos.append(run.execute())
    out = run.fetch(); eps, leaps = run.fetch_diag(); st = run.get_state()
    run.close()
    return dict(out=out, eps=eps, leaps=leaps, state=st, evals=sum(i["n_grad_evals"] for i in infos))


def _same(a, b, sl=slice(None)):
    for k in ("samples", "grads", "accept", "logtarget"):
        assert np.array_equal(a["out"][k][sl], b["out"][k]), k
    assert np.array_equal(a["eps"][sl], b["eps"]) and np.array_equal(a["leaps"][sl], b["leaps"])


@pytest.mark.gpu
@pytest.mark.parametrize("fam", ["normal_dsl", "logistic"])
def test_execution_paths_are_bit_identical(capi, ctx, fam):
    d, C, seed = (4, 200, 13) if fam == "normal_dsl" else (12, 96, 14)
    if fam == "normal_dsl":
        X = y = None; hy = (1.0, 2.0); init = np.ones(d)
    else:
        X, y, hy, b0 = make_regression(fam, 1500, d, 3); init = b0
    dm = capi.DeviceModel(ctx, fam, d, X, y, hy)
    rngt = (21, 1, 50)
    base = _path_run(capi, ctx, dm, C, rngt, init, seed)
    _same(base, _path_run(capi, ctx, dm, C, rngt, init, seed, pieces=(7, 13, 30)))
    for opt, vals in (("poll_every", (1, 8)), ("use_graphs", (0, 1)), ("time_eval", (1,))):
        for v in vals:
            ctx.set_option(opt, v)
            try:
                _same(base, _path_run(capi, ctx, dm, C, rngt, init, seed))
            finally:
                ctx.set_option(opt, {"poll_every": 0, "use_graphs": 1, "time_eval": 0}[opt])
    # chain sharding: global chain ids key the draws
    lo = _path_run(capi, ctx, dm, C, rngt, init, seed, nchains=C // 3)
    hi = _path_run(capi, ctx, dm, C, rngt, init, seed, offset=C // 3, nchains=C - C // 3)
    _same(base, lo, slice(0, C // 3)); _same(base, hi, slice(C // 3, C))
    # continuation: 25 steps, then get_state / set_state into a new run of the remaining steps
    first = _path_run(capi, ctx, dm, C, (21, 1, 25), init, seed)
    st = first["state"]
    cont = capi.DeviceRun(dm, capi.sampler_cfg("NUTS", nleaps=8), (26, 1, 50), C, st["pars"], seed=seed, engine="wave")
    cont.set_state(25, st["leapstep"], st["dual_leapstep"], st["dualH"])
    cont.execute(); o = cont.fetch(); e2, l2 = cont.fetch_diag(); cont.close()
    assert np.array_equal(base["out"]["samples"][:, 5:], o["samples"]) and np.array_equal(base["leaps"][:, 5:], l2)
    assert np.array_equal(base["eps"][:, 5:], e2) and np.array_equal(base["out"]["accept"][:, 5:], o["accept"])
    dm.close()


@pytest.mark.gpu
def test_gradient_count_is_one_per_leapfrog(capi, ctx):
    d, C = 3, 100
    dm = capi.DeviceModel(ctx, "normal_fn", d)
    run = capi.DeviceRun(dm, capi.sampler_cfg("NUTS", nleaps=10), (1, 1, 40), C, np.ones(d), seed=2)
    info = run.execute(); _, leaps = run.fetch_diag()
    assert info["n_grad_evals"] == C + int(leaps.sum())
    run.close(); dm.close()


@pytest.mark.gpu
def test_errors(capi, ctx):
    dm = capi.DeviceModel(ctx, "normal_fn", 2)
    bad = [capi.sampler_cfg("NUTS", nleaps=0), capi.sampler_cfg("NUTS", nleaps=11), capi.sampler_cfg("NUTS", rate=1.5),
           capi.sampler_cfg("NUTS", shrinkage=0.0), capi.sampler_cfg("NUTS", tuner=dict(target_rate=0.5))]
    for cfg in bad:
        with pytest.raises(capi.MCMCGPUError) as e:
            capi.DeviceRun(dm, cfg, (1, 1, 10), 4, np.ones(2))
        assert e.value.code == capi.E_ARG
    ok = capi.sampler_cfg("NUTS")
    for kw in (dict(engine="fused"), dict(store_rb=True),
               dict(normals=np.zeros((4, 11, 2)), uniforms=np.full((4, 11), 0.5))):
        with pytest.raises(capi.MCMCGPUError) as e:
            capi.DeviceRun(dm, ok, (1, 1, 10), 4, np.ones(2), **kw)
        assert e.value.code == capi.E_ARG
    dm.close()
    dm = capi.DeviceModel(ctx, "normal_dsl", 2, hyper=(0.0, 1.0))
    run = capi.DeviceRun(dm, capi.sampler_cfg("NUTS"), (1, 1, 10), 4, np.array([np.inf, 0.0]))
    with pytest.raises(capi.MCMCGPUError) as e:
        run.execute()
    assert e.value.code == capi.E_SUPPORT
    run.close(); dm.close()
    import mcmc_jl_b200 as mj
    with pytest.raises(AssertionError, match="requires model with gradient"):
        mj.run(mj.model("normal", init=np.ones(2), gradient=False) * mj.NUTS() * mj.SerialMC(steps=10))


@pytest.mark.gpu
def test_end_to_end(capi, ctx):
    import io
    import mcmc_jl_b200 as mj
    m = mj.model("normal", init=np.ones(3))
    t = m * mj.NUTS() * mj.GPUMC(steps=100, burnin=50, nchains=8)
    assert isinstance(t, mj.MCMCTask) and isinstance(t.sampler, mj.NUTS) and t.runner.nchains == 8
    ts = m * [mj.NUTS(), mj.HMC()] * mj.SerialMC(steps=10)
    assert isinstance(ts[0].sampler, mj.NUTS) and len(ts) == 2
    c = mj.run(m * mj.NUTS() * mj.SerialMC(steps=600, burnin=100))
    assert isinstance(c, mj.MCMCChain) and c.samples.shape == (500, 3)
    nd = c.diagnostics["ndoublings"]
    assert nd.shape == (500,) and nd.min() >= 1 and nd.max() <= 10 and c.diagnostics["epsilon"].shape == (500,)
    assert np.all(np.isfinite(mj.ess(c))) and np.all(mj.ess(c) > 50)
    buf = io.StringIO(); mj.describe(c, buf)
    assert buf.getvalue()
    batch = mj.run(m * mj.NUTS(maxdoublings=6) * mj.GPUMC(steps=300, burnin=100, nchains=256, seed=3))
    assert mj.ess(batch).shape == (256, 3) and batch[5].diagnostics["ndoublings"].max() <= 6
    assert abs(batch.arrays()["samples"][:, -1].var() - 0.5) < 0.1
    batch.close()
