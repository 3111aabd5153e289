"""NUTS with a diagonal metric (mcmcgpu_run_set_metric / _set_metric_adaptation / _get_metric, mj.NUTS(inv_metric=,
adapt_metric=)): the CPU restatement tests/nuts_metric_oracle.c (orc_run_nuts_metric) against Stan's window rule, the
identity-metric restatement tests/nuts_oracle.c, exact targets and its own invariants, the host API, and on the GPU nuts_kernel<true> against the restatement -- bit for bit on the
closed-form families, with the metric fixed or adapted through Stan's windows -- plus statistics, execution paths and
errors."""
import ctypes as C
import math
import os
import subprocess
import tempfile

import numpy as np
import pytest

from conftest import make_regression, ou_series
from test_nuts import CLOSED, REGRESSION, _check_exact, run_many, run_nuts

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

STAN = (75, 50, 25)


# ---- Stan's windows, restated from windowed_adaptation.hpp in Python ----------------------------------------------------
def stan_windows(W, init, term, window):
    """window-end STEPS (counter k = step - 1) and the steps lo..hi whose samples enter the estimate"""
    if W < 20:
        return [], (1, 0)
    if init + window + term > W:
        init, term = int(0.15 * W), int(0.1 * W)
        window = W - (init + term)
    size, nxt, ends = window, init + window - 1, []
    for k in range(W):
        if k == nxt and k != W:                                             # end_adaptation_window
            ends.append(k + 1)
            if nxt != W - term - 1:                                         # compute_next_window
                size *= 2
                nxt = k + size
                if nxt != W - term - 1 and nxt + 2 * size >= W - term:
                    nxt = W - term - 1
    return ends, (init + 1, W - term)


@pytest.fixture(scope="session")
def NM(O):
    """tests/nuts_metric_oracle.c and tests/nuts_oracle.c compiled with the oracle (same flags as oracle/Makefile) into a
    temporary library"""
    tmp = tempfile.mkdtemp(prefix="nuts_metric_oracle_")
    so = os.path.join(tmp, "libnuts_metric_oracle.so")
    subprocess.check_call(["gcc", "-O3", "-std=gnu99", "-ffp-contract=off", "-fPIC", "-shared", "-o", so,
                           os.path.join(ROOT, "tests", "nuts_metric_oracle.c"), os.path.join(ROOT, "tests", "nuts_oracle.c"),
                           os.path.join(ROOT, "oracle", "mcmc_oracle.c"), "-lm"])
    N = C.CDLL(so)
    dp, i64p = C.POINTER(C.c_double), C.POINTER(C.c_int64)
    N.orc_run_nuts.restype = C.c_int32
    N.orc_run_nuts.argtypes = [C.POINTER(O._Model), C.POINTER(O._Sampler), C.POINTER(O._Range), dp, C.c_uint64, C.c_uint64, dp,
                               dp, dp, C.POINTER(C.c_uint8), dp, dp, i64p, dp, i64p, i64p]
    N.orc_nuts_windows.restype = C.c_int32
    N.orc_nuts_windows.argtypes = [C.c_int64, C.c_int64, C.c_int64, C.c_int64, i64p, i64p, i64p]
    N.orc_run_nuts_metric.restype = C.c_int32
    N.orc_run_nuts_metric.argtypes = [C.POINTER(O._Model), C.POINTER(O._Sampler), C.POINTER(O._Range), dp, C.c_uint64, C.c_uint64,
                                      dp, dp, i64p, dp, dp, dp, C.POINTER(C.c_uint8), dp, dp, i64p, dp, i64p, i64p, dp, i64p, dp]
    return N


def oracle_windows(NM, W, init, term, window):
    ends, lo, hi = np.zeros(64, np.int64), C.c_int64(0), C.c_int64(0)
    n = NM.orc_nuts_windows(W, init, term, window, ends.ctypes.data_as(C.POINTER(C.c_int64)), C.byref(lo), C.byref(hi))
    return list(ends[:n]), (lo.value, hi.value)


def run_nuts_metric(O, NM, om, rngt, init, seed, chain, inv_metric=None, adapt=None, force_minv=None, maxd=10, rate=0.6,
                    force_eps=None, start_step=0, da_state=None, normals=None):
    """one restated chain with a metric; adapt = (init_buffer, term_buffer, window) or None; force_minv (last+1, d)"""
    first, stp, last = rngt
    d = om.d
    S = (last - first) // stp + 1
    smp = O.sampler("HMCDA", nleaps=maxd, rate=rate, force_eps=force_eps, start_step=start_step, da_state=da_state)
    f64 = lambda a: None if a is None else np.ascontiguousarray(a, dtype=np.float64)
    init = np.ascontiguousarray(np.broadcast_to(init, (d,)), dtype=np.float64)
    zn = None if normals is None else f64(normals[:last + 1])
    im, fm = f64(inv_metric), f64(force_minv)
    ad = None if adapt is None else np.ascontiguousarray(adapt, dtype=np.int64)
    out = dict(samples=np.full((S, d), np.nan), grads=np.full((S, d), np.nan), accept=np.zeros(S, np.uint8),
               logtarget=np.full(S, np.nan), eps=np.full(S, np.nan), leaps=np.zeros(S, np.int64), alpha=np.full(S, np.nan),
               ndoublings=np.zeros(S, np.int64), win_minv=np.full((64, d), np.nan), minv=np.full(d, np.nan))
    nev, nwin = C.c_int64(0), C.c_int64(0)
    p = lambda a: None if a is None else a.ctypes.data_as(C.POINTER(C.c_double))
    i64 = lambda a: a.ctypes.data_as(C.POINTER(C.c_int64))
    rc = NM.orc_run_nuts_metric(C.byref(om._c), C.byref(smp), C.byref(O._Range(first, stp, last)), p(init), seed, chain, p(zn),
                                p(im), None if ad is None else i64(ad), p(fm), p(out["samples"]), p(out["grads"]),
                                out["accept"].ctypes.data_as(C.POINTER(C.c_uint8)), p(out["logtarget"]), p(out["eps"]),
                                i64(out["leaps"]), p(out["alpha"]), i64(out["ndoublings"]), C.byref(nev), p(out["win_minv"]),
                                C.byref(nwin), p(out["minv"]))
    out["rc"], out["n_grad_evals"], out["n_win"] = rc, nev.value, nwin.value
    out["win_minv"] = out["win_minv"][:nwin.value]
    return out


# ---- CPU: the restatement ---------------------------------------------------------------------------------------------
def test_window_schedule_is_stans(NM):
    for bufs in (STAN, (5, 5, 5), (15, 10, 3), (0, 0, 1), (100, 100, 100), (10, 0, 7)):
        for W in range(0, 2501):
            assert oracle_windows(NM, W, *bufs) == stan_windows(W, *bufs), (W, bufs)
    assert stan_windows(19, *STAN)[0] == []
    assert stan_windows(100, *STAN) == ([90], (16, 90))                    # 15 / 70 / 10 % of W
    assert stan_windows(151, *STAN)[0] == [100, 101]                        # the last window holds one draw
    assert stan_windows(1000, *STAN)[0] == [100, 150, 250, 450, 950]
    assert stan_windows(2000, *STAN)[0] == [100, 150, 250, 450, 850, 1950]


def test_all_ones_metric_is_the_identity_bit_for_bit(O, NM):
    om = O.Model("normal_dsl", 5, hyper=(1.0, 2.0))
    rngt = (31, 1, 60)
    for c in range(16):
        ref = run_nuts(O, NM, om, rngt, np.full(5, 3.0), 4, c)
        one = run_nuts_metric(O, NM, om, rngt, np.full(5, 3.0), 4, c, inv_metric=np.ones(5))
        assert one["rc"] == 0
        for k in ("samples", "grads", "accept", "logtarget", "eps", "leaps", "alpha", "ndoublings"):
            assert np.array_equal(ref[k], one[k]), (c, k)
        assert one["n_grad_evals"] == ref["n_grad_evals"]


def test_fixed_metric_samples_exact_target(O, NM):
    """any positive metric leaves the target invariant: 2000 chains of N(1, 2^2), each with its own metric in [0.2, 5]"""
    om = O.Model("normal_dsl", 5, hyper=(1.0, 2.0))
    mets = np.random.default_rng(3).uniform(0.2, 5.0, (2000, 5))
    res = run_many(lambda c: run_nuts_metric(O, NM, om, (101, 1, 130), np.full(5, 3.0), 2024, c, inv_metric=mets[c]), range(2000))
    assert all(r["rc"] == 0 for r in res)
    _check_exact(np.array([r["samples"][-1] for r in res]), 1.0, 2.0, "normal_dsl, fixed metric")


def test_adapted_metric_estimates_the_variance(O, NM):
    """W = 1000 with Stan's buffers: five windows, and the median over chains of the final metric is within 15 % of 4"""
    om = O.Model("normal_dsl", 5, hyper=(1.0, 2.0))
    W = 1000
    res = run_many(lambda c: run_nuts_metric(O, NM, om, (W + 2, 1, W + 11), np.full(5, 3.0), 77, c, adapt=STAN), range(500))
    assert all(r["rc"] == 0 and r["n_win"] == 5 for r in res)
    med = np.median(np.array([r["minv"] for r in res]), axis=0)
    assert np.all(np.abs(med / 4.0 - 1.0) < 0.15), med
    _check_exact(np.array([r["samples"][-1] for r in res]), 1.0, 2.0, "normal_dsl, adapted")


def test_one_draw_window_keeps_the_metric_before_regularising(O, NM):
    """W = 151: the window ending at step 101 holds one draw, so the metric becomes (1/6) minv + 1e-3 (5/6)"""
    om = O.Model("normal_dsl", 2, hyper=(1.0, 2.0))
    r = run_nuts_metric(O, NM, om, (153, 1, 155), np.ones(2), 5, 0, adapt=STAN)
    assert r["rc"] == 0 and r["n_win"] == 2
    assert np.array_equal(r["win_minv"][1], (1.0 / 6.0) * r["win_minv"][0] + 1e-3 * (5.0 / 6.0))
    assert np.array_equal(r["minv"], r["win_minv"][1])


@pytest.mark.parametrize("fam,d,hy,maxd", [("normal_dsl", 5, (1.0, 2.0), 10), ("normal_fn", 3, (), 3), ("abs_normal", 2, (1.0, 0.5), 4)])
def test_invariants_hold_with_a_metric(O, NM, fam, d, hy, maxd):
    """odd chains: a fixed metric, every step kept; even chains: adapted (W = 60 with 5 / 5 / 5), the steps after it kept"""
    om = O.Model(fam, d, hyper=hy)
    mets = np.random.default_rng(d).uniform(0.2, 5.0, (64, d))
    jobs = [(c, (1, 1, 120), dict(inv_metric=mets[c])) if c % 2 else (c, (62, 1, 150), dict(adapt=(5, 5, 5))) for c in range(64)]
    res = run_many(lambda j: run_nuts_metric(O, NM, om, j[1], np.ones(d), 11, j[0], maxd=maxd, rate=0.8, **j[2]), jobs)
    for c, r in enumerate(res):
        assert r["rc"] == 0
        assert np.all(r["leaps"] >= 1) and np.all(r["leaps"] <= 2 ** maxd - 1)
        assert np.array_equal(np.floor(np.log2(r["leaps"])).astype(np.int64) + 1, r["ndoublings"])
        stay = r["accept"][1:] == 0
        assert np.array_equal(r["samples"][1:][stay], r["samples"][:-1][stay])
        assert np.array_equal(r["logtarget"][1:][stay], r["logtarget"][:-1][stay])
        assert r["n_grad_evals"] == 1 + r["leaps"].sum() if c % 2 else r["n_grad_evals"] > 61 + r["leaps"].sum()
        assert np.all(np.isfinite(r["minv"])) and np.all(r["minv"] > 0)
    assert all(res[c]["n_win"] == 3 for c in range(0, 64, 2))              # W = 60 with 5 / 5 / 5: steps 10, 20, 55


def test_nuts_constructor_metric_arguments():
    import mcmc_jl_b200 as mj
    s = mj.NUTS()
    assert (s.inv_metric, s.adapt_metric, s.init_buffer, s.term_buffer, s.window) == (None, False, 75, 50, 25)
    cfg = mj.NUTS(rate=0.7, maxdoublings=6, shrinkage=0.1, t0=5.0, step=0.5)._cfg()
    assert (cfg.kind, cfg.nleaps, cfg.rate, cfg.shrinkage, cfg.t0, cfg.step, cfg.tuner_on) == (5, 6, 0.7, 0.1, 5.0, 0.5, 0)
    calls = []

    class Rec:
        C = 4

        def set_metric(self, m):
            calls.append(("set_metric", np.array(m)))

        def set_metric_adaptation(self, *a):
            calls.append(("adapt", a))
    s._set_metric(Rec(), 0, 4)
    assert calls == []                                                      # the defaults make no metric call
    mj.NUTS(inv_metric=np.arange(1.0, 13.0).reshape(6, 2), adapt_metric=True, init_buffer=5, term_buffer=6, window=7)._set_metric(Rec(), 2, 6)
    assert np.array_equal(calls[0][1], np.arange(5.0, 13.0).reshape(4, 2)) and calls[1] == ("adapt", (5, 6, 7))
    assert np.array_equal(mj.NUTS(inv_metric=[1.0, 2.0]).inv_metric, [1.0, 2.0])
    for bad in (lambda: mj.NUTS(inv_metric=[1.0, 0.0]), lambda: mj.NUTS(inv_metric=[1.0, -2.0]), lambda: mj.NUTS(inv_metric=[np.nan]),
                lambda: mj.NUTS(inv_metric=[np.inf]), lambda: mj.NUTS(inv_metric=np.ones((2, 2, 2))), lambda: mj.NUTS(inv_metric=[]),
                lambda: mj.NUTS(init_buffer=-1), lambda: mj.NUTS(term_buffer=-1), lambda: mj.NUTS(window=0),
                lambda: mj.NUTS(window=2.5)):
        with pytest.raises(AssertionError):
            bad()


# ---- GPU ----------------------------------------------------------------------------------------------------------------
def _out(run):
    out = run.fetch(); eps, leaps = run.fetch_diag()
    return dict(out=out, eps=eps, leaps=leaps, minv=run.get_metric())


def _same(a, b, sl=slice(None)):
    for k in ("samples", "grads", "accept", "logtarget"):
        assert np.array_equal(a["out"][k][sl], b["out"][k]), k
    assert np.array_equal(a["eps"][sl], b["eps"]) and np.array_equal(a["leaps"][sl], b["leaps"])


@pytest.mark.gpu
@pytest.mark.parametrize("fam", ["normal_dsl", "logistic"])
def test_all_ones_metric_is_bit_identical_on_the_device(capi, ctx, fam):
    d, C = (5, 300) if fam == "normal_dsl" else (100, 256)
    if fam == "normal_dsl":
        X = y = None; hy = (1.0, 2.0); init = np.full(d, 3.0)
    else:
        X, y, hy, b0 = make_regression(fam, 2000, d, 6); init = b0
    dm = capi.DeviceModel(ctx, fam, d, X, y, hy)
    rngt = (31, 1, 45)                                                      # the step size adapts on steps 1..29

    def one(metric):
        run = capi.DeviceRun(dm, capi.sampler_cfg("NUTS", nleaps=8), rngt, C, init, seed=21, engine="wave")
        if metric is not None:
            run.set_metric(metric)
        run.execute(); o = _out(run); run.close()
        return o
    base = one(None)
    assert np.array_equal(base["minv"], np.ones((C, d)))
    for m in (np.ones(d), np.ones((C, d))):
        _same(base, one(m))
    dm.close()


def _device_and_oracle(O, NM, capi, ctx, fam, d, X, y, hy, C, rngt, init, seed, minv, maxd=10, s0=0, eps0=None, chains=None):
    """a device run with the per-chain metric minv and the restatement replaying it with the device's normals (as
    test_nuts._device_and_oracle: s0 > 0 starts after step s0 with step size eps0, forced one step ahead)"""
    first, _, last = rngt
    om, dm = O.Model(fam, d, X, y, hy), capi.DeviceModel(ctx, fam, d, X, y, hy)
    run = capi.DeviceRun(dm, capi.sampler_cfg("NUTS", nleaps=maxd, rate=0.6), rngt, C, init, seed=seed, engine="wave")
    run.set_state(s0, eps0, eps0, np.zeros(C))
    run.set_metric(minv)
    info = run.execute(); out = run.fetch(); eps, leaps = run.fetch_diag()
    run.close(); dm.close()
    zn, _ = ctx.philox_draws(seed, 0, C, d, last)
    chains = range(C) if chains is None else chains
    ini = lambda c: init[c] if np.ndim(init) == 2 else init

    def one(c):
        fe = np.concatenate([np.full(s0 + 1, np.nan), eps[c]])
        return c, run_nuts_metric(O, NM, om, rngt, ini(c), seed, c, inv_metric=minv[c], maxd=maxd, normals=zn[c], start_step=s0,
                                  da_state=[eps0[c], eps0[c], 0.0], force_eps=fe)
    return out, eps, leaps, dict(run_many(one, list(chains))), info


@pytest.mark.gpu
@pytest.mark.parametrize("fam,d,hy", CLOSED, ids=lambda c: str(c))
def test_closed_form_parity_with_a_fixed_metric(O, NM, capi, ctx, fam, d, hy):
    C, s0, K = 70, 50, 25
    r = np.random.default_rng(100 + d)
    minv = np.exp(r.uniform(np.log(0.2), np.log(5.0), (C, d)))
    if fam == "ou":
        y, init, maxd = ou_series(300, 4), np.array([20.0, 0.1, 10.0]), 7
        eps0 = 0.002 * np.exp(0.3 * r.standard_normal(C))
        minv = np.exp(r.uniform(np.log(0.5), np.log(2.0), (C, d)))
    else:
        y, init, maxd = None, 0.5 + r.standard_normal((C, d)), 10
        eps0 = {"normal_fn": 0.8, "normal_dsl": 1.2, "abs_normal": 0.25}[fam] * np.exp(0.4 * r.standard_normal(C)) / 2
    out, eps, leaps, refs, info = _device_and_oracle(O, NM, capi, ctx, fam, d, None, y, hy, C, (s0 + 1, 1, s0 + K), init, 7, minv,
                                                     maxd, s0, eps0)
    for c in range(C):
        ref = refs[c]
        assert ref["rc"] == 0
        assert np.array_equal(ref["accept"], out["accept"][c]), c
        assert np.array_equal(ref["leaps"], leaps[c]), c
        assert np.array_equal(ref["eps"], eps[c]), c
        if fam == "ou":
            assert np.allclose(ref["samples"], out["samples"][c], rtol=1e-10, atol=0), c
            assert np.allclose(ref["logtarget"], out["logtarget"][c], rtol=1e-10, atol=0), c
            continue
        assert np.array_equal(ref["samples"], out["samples"][c]), c
        assert np.array_equal(ref["logtarget"], out["logtarget"][c]), c
        assert np.array_equal(ref["grads"], out["grads"][c]), c
    assert info["n_grad_evals"] == C + int(leaps.sum())
    assert leaps.max() > 4 and out["accept"].mean() > 0.2


@pytest.mark.gpu
@pytest.mark.parametrize("fam,d,hy", [("normal_fn", 3, ()), ("normal_dsl", 3, (1.0, 2.0)), ("abs_normal", 3, (1.0, 0.5))])
def test_adaptation_parity_bit_exact(O, NM, capi, ctx, fam, d, hy):
    """W = 60 with 5 / 5 / 5: windows end at steps 10, 20 and 55.  Stepwise, the step size and the metric of every warm-up
    step are read back and forced on the restatement, whose own metrics after every window end must equal the device's bit
    for bit (its own step sizes to 1e-9); the metric changes at those steps and nowhere else; the draws are bit-identical
    and equal those of a one-call run."""
    C, seed, W = 64, 17, 60
    first, last = W + 2, W + 10
    rngt = (first, 1, last)
    init = 0.5 + np.random.default_rng(d).standard_normal((C, d))
    dm = capi.DeviceModel(ctx, fam, d, None, None, hy)
    mk = lambda: capi.DeviceRun(dm, capi.sampler_cfg("NUTS", nleaps=10, rate=0.6), rngt, C, init, seed=seed, engine="wave")
    one = mk(); one.set_metric_adaptation(5, 5, 5); one.execute(); o1 = _out(one); one.close()
    run = mk(); run.set_metric_adaptation(5, 5, 5)
    fe, fm = np.full((C, last + 1), np.nan), np.ones((C, last + 1, d))
    fe[:, 1] = 1.0
    changed = []
    for i in range(1, first):                                               # after step i: the step size and metric of step i + 1
        run.execute_steps(1)
        fe[:, i + 1] = run.get_state()["leapstep"]
        fm[:, i + 1] = run.get_metric()
        if not np.array_equal(fm[:, i + 1], fm[:, i]):
            changed.append(i)
    assert changed == [10, 20, 55]
    fe[:, first + 1:] = fe[:, first][:, None]
    fm[:, first + 1:] = fm[:, first][:, None]
    run.execute_steps(last - first + 1)
    o = _out(run); run.close(); dm.close()
    _same(o1, o)
    assert np.array_equal(o1["minv"], o["minv"]) and np.array_equal(o["minv"], fm[:, first])
    assert np.array_equal(o["eps"], fe[:, first:])
    zn, _ = ctx.philox_draws(seed, 0, C, d, last)
    om = O.Model(fam, d, hyper=hy)
    refs = run_many(lambda c: run_nuts_metric(O, NM, om, rngt, init[c], seed, c, adapt=(5, 5, 5), force_minv=fm[c], force_eps=fe[c],
                                              normals=zn[c]), range(C))
    for c, ref in enumerate(refs):
        assert ref["rc"] == 0 and ref["n_win"] == 3, c
        assert np.array_equal(ref["win_minv"], fm[c, [11, 21, 56]]), c
        assert np.array_equal(ref["minv"], o["minv"][c]), c
        for k in ("samples", "grads", "logtarget", "accept"):
            assert np.array_equal(ref[k], o["out"][k][c]), (c, k)
        assert np.array_equal(ref["leaps"], o["leaps"][c]), c
        assert np.allclose(ref["eps"], o["eps"][c], rtol=1e-9, atol=0), c
    assert np.any(np.abs(o["minv"] - 1.0) > 0.1)


@pytest.mark.gpu
@pytest.mark.parametrize("fam,d", REGRESSION, ids=lambda c: str(c))
def test_regression_parity_with_a_fixed_metric(O, NM, capi, ctx, fam, d):
    Nrows = 997
    X, y, hy, b0 = make_regression(fam, Nrows, d, 5)
    ntiles = -(-Nrows // 32)
    s0, K = 40, 12
    r = np.random.default_rng(d + 1)
    base = (0.3 if fam == "probit" else 0.5) / math.sqrt(Nrows)
    gs = np.abs(X).sum(0)
    try:
        for C, splits in ((130, 1), (70, 3), (1, ntiles + 3)):
            ctx.set_option("force_splits", splits)
            init = b0 + 0.05 * r.standard_normal((C, d)) / math.sqrt(d)
            minv = np.exp(r.uniform(np.log(0.5), np.log(2.0), (C, d)))
            eps0 = base * np.exp(0.3 * r.standard_normal(C)) / 1.5
            chains = range(C) if d <= 10 else range(0, C, 5)
            out, eps, leaps, refs, info = _device_and_oracle(O, NM, capi, ctx, fam, d, X, y, hy, C, (s0 + 1, 1, s0 + K), init, 9,
                                                             minv, 8, s0, eps0, chains)
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


def regularised_variance(W, var, bufs=STAN):
    """what Stan's estimator targets from the last window's n draws: (n / (n + 5)) var + 1e-3 (5 / (n + 5))"""
    ends = stan_windows(W, *bufs)[0]
    n = ends[-1] - ends[-2]
    return (n / (n + 5.0)) * var + 1e-3 * (5.0 / (n + 5.0))


def _scaled_linear(Nr=300, d=10, seed=8, top=2.0):
    """linear regression with columns scaled by 10**linspace(0, top, d) and correlated, and its Gaussian posterior"""
    r = np.random.default_rng(seed)
    A = np.eye(d) + 0.6 * np.tril(r.standard_normal((d, d)), -1)
    X = r.standard_normal((Nr, d)) @ A.T
    X[:, 0] = 1.0
    X = X * 10.0 ** np.linspace(0, top, d)
    beta = r.standard_normal(d) / 2 / 10.0 ** np.linspace(0, top, d)
    y = X @ beta + r.standard_normal(Nr)
    prec = X.T @ X + np.eye(d)                                              # noise sd 1, prior sd 1
    cov = np.linalg.inv(prec)
    return X, y, prec, cov, cov @ (X.T @ y)


@pytest.mark.gpu
def test_adapted_metric_on_a_badly_scaled_posterior(capi, ctx):
    d, C, W = 10, 4096, 1000
    X, y, prec, cov, mean = _scaled_linear(d=d)
    dm = capi.DeviceModel(ctx, "linear", d, X, y, (1.0, 1.0))
    run = capi.DeviceRun(dm, capi.sampler_cfg("NUTS", nleaps=10), (W + 2, 1, W + 61), C, mean, seed=5, store_grad=False, engine="wave")
    run.set_metric_adaptation(*STAN)
    run.execute(); x = run.fetch()["samples"]; _, leaps = run.fetch_diag(); minv = run.get_metric()
    run.close()
    z = (x[:, -1] - mean) @ np.linalg.cholesky(prec)                        # whitened: iid N(0, 1) coordinates
    _check_exact(z, 0.0, 1.0, "linear, adapted metric")
    # the narrowest coordinates' variances (~1e-7) are far below the regulariser 1e-3 * 5 / (n + 5): compare with what it targets
    ratio = np.median(minv / regularised_variance(W, np.diag(cov)), axis=0)
    assert np.all((ratio > 0.8) & (ratio < 1.25)), ratio
    ident = capi.DeviceRun(dm, capi.sampler_cfg("NUTS", nleaps=10), (202, 1, 221), 512, mean, seed=5, store_grad=False, engine="wave")
    ident.execute(); _, leaps_id = ident.fetch_diag(); ident.close(); dm.close()
    assert leaps.mean() <= 0.25 * leaps_id.mean(), (leaps.mean(), leaps_id.mean())


@pytest.mark.gpu
@pytest.mark.parametrize("fam", ["normal_dsl", "logistic"])
def test_execution_paths_are_bit_identical_with_adaptation(capi, ctx, fam):
    d, C, seed = (4, 200, 13) if fam == "normal_dsl" else (12, 96, 14)
    if fam == "normal_dsl":
        X = y = None; hy = (1.0, 2.0); init = np.ones(d)
    else:
        X, y, hy, b0 = make_regression(fam, 1500, d, 3); init = b0
    dm = capi.DeviceModel(ctx, fam, d, X, y, hy)
    rngt = (62, 1, 80)                                                      # W = 60, windows end at steps 10, 20, 55
    mets = np.random.default_rng(2).uniform(0.5, 2.0, (C, d))

    def path(pieces=None, offset=0, n=None, rng=rngt, state=None, metric=mets, adapt=True, x0=init):
        n = n or C
        run = capi.DeviceRun(dm, capi.sampler_cfg("NUTS", nleaps=8), rng, n, x0, seed=seed, chain_offset=offset, engine="wave")
        if state is not None:
            run.set_state(*state)
        run.set_metric(metric[offset:offset + n])
        if adapt:
            run.set_metric_adaptation(5, 5, 5)
        for p in (pieces or [None]):
            run.execute() if p is None else run.execute_steps(p)
        o = _out(run); o["state"] = run.get_state(); run.close()
        return o
    base = path()
    assert not np.array_equal(base["minv"], mets)
    for pieces in ((7, 13, 30, 30), (10, 10, 35, 1, 24)):                  # pieces that end at and cross the window ends
        o = path(pieces)
        _same(base, o); assert np.array_equal(base["minv"], o["minv"])
    for opt, vals in (("poll_every", (1, 8)), ("use_graphs", (0, 1)), ("time_eval", (1,))):
        for v in vals:
            ctx.set_option(opt, v)
            try:
                o = path()
                _same(base, o); assert np.array_equal(base["minv"], o["minv"])
            finally:
                ctx.set_option(opt, {"poll_every": 0, "use_graphs": 1, "time_eval": 0}[opt])
    lo, hi = path(n=C // 3), path(offset=C // 3, n=C - C // 3)              # each chain adapts alone: sharding changes nothing
    _same(base, lo, slice(0, C // 3)); _same(base, hi, slice(C // 3, C))
    assert np.array_equal(base["minv"], np.concatenate([lo["minv"], hi["minv"]]))
    # continuation: the warm-up run, then a new run from its state and metric gives the one-call run's later draws
    warm = path(rng=(62, 1, 65))
    st = warm["state"]
    cont = path(rng=(66, 1, 80), state=(65, st["leapstep"], st["dual_leapstep"], st["dualH"]), metric=warm["minv"], adapt=False,
                x0=st["pars"])
    assert np.array_equal(cont["minv"], base["minv"])
    for k in ("samples", "grads", "accept", "logtarget"):
        assert np.array_equal(base["out"][k][:, 4:], cont["out"][k]), k
    assert np.array_equal(base["eps"][:, 4:], cont["eps"]) and np.array_equal(base["leaps"][:, 4:], cont["leaps"])
    dm.close()


@pytest.mark.gpu
def test_metric_errors(capi, ctx):
    dm = capi.DeviceModel(ctx, "normal_dsl", 2, hyper=(0.0, 1.0))
    ok = np.ones(2)
    for cfg, kw in ((capi.sampler_cfg("HMC"), {}), (capi.sampler_cfg("HMCDA"), dict(engine="wave")), (capi.sampler_cfg("HMC"), dict(engine="fused"))):
        run = capi.DeviceRun(dm, cfg, (1, 1, 10), 4, ok, **kw)
        for call in (lambda: run.set_metric(ok), lambda: run.set_metric_adaptation(), lambda: run.get_metric()):
            with pytest.raises(capi.MCMCGPUError) as e:
                call()
            assert e.value.code == capi.E_ARG
        run.close()
    run = capi.DeviceRun(dm, capi.sampler_cfg("NUTS"), (30, 1, 40), 4, ok)
    for bad in (np.array([1.0, np.nan]), np.array([0.0, 1.0]), np.array([1.0, -1.0]), np.array([np.inf, 1.0]), np.full((4, 2), -1.0)):
        with pytest.raises(capi.MCMCGPUError) as e:
            run.set_metric(bad)
        assert e.value.code == capi.E_ARG
    for bufs in ((-1, 5, 5), (5, -1, 5), (5, 5, 0)):
        with pytest.raises(capi.MCMCGPUError) as e:
            run.set_metric_adaptation(*bufs)
        assert e.value.code == capi.E_ARG
    run.set_metric(np.array([2.0, 3.0]))
    assert np.array_equal(run.get_metric(), np.tile([2.0, 3.0], (4, 1)))  # before execute: the starting metric
    run.set_metric_adaptation(5, 5, 5)
    with pytest.raises(capi.MCMCGPUError) as e:                             # adaptation needs the whole warm-up
        run.set_state(10)
    assert e.value.code == capi.E_ARG
    run.execute_steps(3)
    for call in (lambda: run.set_metric(ok), lambda: run.set_metric_adaptation()):
        with pytest.raises(capi.MCMCGPUError) as e:
            call()
        assert e.value.code == capi.E_STATE
    run.close()
    run = capi.DeviceRun(dm, capi.sampler_cfg("NUTS"), (30, 1, 40), 4, ok)
    run.set_state(10)
    with pytest.raises(capi.MCMCGPUError) as e:
        run.set_metric_adaptation()
    assert e.value.code == capi.E_ARG
    run.close()
    run = capi.DeviceRun(dm, capi.sampler_cfg("NUTS"), (30, 1, 40), 4, ok)  # step0 after the warm-up is allowed
    run.set_state(28); run.set_metric_adaptation(); run.execute(); run.close()
    dm.close()


@pytest.mark.gpu
def test_end_to_end(capi, ctx):
    import mcmc_jl_b200 as mj
    d = 6
    X, y, prec, cov, mean = _scaled_linear(Nr=300, d=d, seed=4, top=1.5)
    m = mj.model("linear", X=X, Y=y, vars=mean)
    batch = mj.run(m * mj.NUTS(adapt_metric=True) * mj.GPUMC(steps=700, burnin=601, nchains=512, seed=2))
    minv = batch.inv_metric()
    assert minv.shape == (512, d)
    ratio = np.median(minv / regularised_variance(600, np.diag(cov)), axis=0)
    assert np.all((ratio > 0.7) & (ratio < 1.4)), ratio
    assert np.array_equal(batch[3].diagnostics["inv_metric"], minv[3])
    batch.close()
    plain = mj.run(m * mj.NUTS() * mj.GPUMC(steps=50, burnin=20, nchains=8))
    assert "inv_metric" not in plain[0].diagnostics and np.array_equal(plain.inv_metric(), np.ones((8, d)))
    plain.close()
    fixed = np.diag(cov)
    c = mj.run(m * mj.NUTS(inv_metric=fixed) * mj.SerialMC(steps=300, burnin=100))
    assert np.array_equal(c.diagnostics["inv_metric"], fixed) and c.samples.shape == (200, d)
    per = np.tile(fixed, (8, 1)) * np.linspace(0.5, 2.0, 8)[:, None]
    b = mj.run(m * mj.NUTS(inv_metric=per) * mj.GPUMC(steps=60, burnin=20, nchains=8))
    assert np.array_equal(b.inv_metric(), per)
    b.close()
    with pytest.raises(AssertionError, match="inv_metric"):                # (nchains, d) must match the runner's chains
        mj.run(m * mj.NUTS(inv_metric=per) * mj.GPUMC(steps=60, burnin=20, nchains=4))
