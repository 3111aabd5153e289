"""NUTS with a dense metric (mcmcgpu_run_set_dense_metric / _get_dense_metric, mj.NUTS(metric="dense")): the CPU
restatement tests/nuts_dense_oracle.c (orc_run_nuts_dense) against the diagonal- and identity-metric restatements, numpy
and an exact Gaussian posterior, the host API, and on the GPU nuts_kernel's dense instantiation against the restatement --
bit for bit on the closed-form families, with the metric fixed or adapted through Stan's windows -- plus statistics,
execution paths and errors."""
import ctypes as C
import math
import os
import subprocess
import tempfile

import numpy as np
import pytest
from scipy import stats as sst

from conftest import make_regression, ou_series
from test_nuts import CLOSED, REGRESSION, run_many, run_nuts
from test_nuts_metric import STAN, run_nuts_metric, stan_windows

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="session")
def ND(O):
    """tests/nuts_dense_oracle.c with tests/nuts_metric_oracle.c, tests/nuts_oracle.c and the oracle (same flags as
    oracle/Makefile) in a temporary library"""
    tmp = tempfile.mkdtemp(prefix="nuts_dense_oracle_")
    so = os.path.join(tmp, "libnuts_dense_oracle.so")
    subprocess.check_call(["gcc", "-O3", "-std=gnu99", "-ffp-contract=off", "-fPIC", "-shared", "-o", so,
                           os.path.join(ROOT, "tests", "nuts_dense_oracle.c"), os.path.join(ROOT, "tests", "nuts_metric_oracle.c"),
                           os.path.join(ROOT, "tests", "nuts_oracle.c"), os.path.join(ROOT, "oracle", "mcmc_oracle.c"), "-lm"])
    N = C.CDLL(so)
    dp, i64p = C.POINTER(C.c_double), C.POINTER(C.c_int64)
    N.orc_run_nuts.restype = C.c_int32
    N.orc_run_nuts.argtypes = [C.POINTER(O._Model), C.POINTER(O._Sampler), C.POINTER(O._Range), dp, C.c_uint64, C.c_uint64, dp,
                               dp, dp, C.POINTER(C.c_uint8), dp, dp, i64p, dp, i64p, i64p]
    N.orc_run_nuts_metric.restype = C.c_int32
    N.orc_run_nuts_metric.argtypes = [C.POINTER(O._Model), C.POINTER(O._Sampler), C.POINTER(O._Range), dp, C.c_uint64, C.c_uint64,
                                      dp, dp, i64p, dp, dp, dp, C.POINTER(C.c_uint8), dp, dp, i64p, dp, i64p, i64p, dp, i64p, dp]
    N.orc_run_nuts_dense.restype = C.c_int32
    N.orc_run_nuts_dense.argtypes = N.orc_run_nuts_metric.argtypes
    N.orc_dense_cholesky.restype = C.c_int32
    N.orc_dense_cholesky.argtypes = [dp, dp, C.c_int64]
    N.orc_dense_backsub.restype = None
    N.orc_dense_backsub.argtypes = [dp, dp, dp, C.c_int64]
    N.orc_welford_covar.restype = None
    N.orc_welford_covar.argtypes = [dp, C.c_int64, C.c_int64, dp, dp]
    return N


def _p(a):
    return None if a is None else a.ctypes.data_as(C.POINTER(C.c_double))


def run_nuts_dense(O, ND, om, rngt, init, seed, chain, inv_metric=None, adapt=None, force_A=None, maxd=10, rate=0.6,
                   force_eps=None, start_step=0, da_state=None, normals=None):
    """one restated chain with a dense metric (d, d) (None: the identity); adapt = (init, term, window); force_A (last+1, d, d)"""
    first, stp, last = rngt
    d = om.d
    S = (last - first) // stp + 1
    smp = O.sampler("HMCDA", nleaps=maxd, rate=rate, force_eps=force_eps, start_step=start_step, da_state=da_state)
    f64 = lambda a: None if a is None else np.ascontiguousarray(a, dtype=np.float64)
    init = np.ascontiguousarray(np.broadcast_to(init, (d,)), dtype=np.float64)
    zn = None if normals is None else f64(normals[:last + 1])
    im, fa = f64(inv_metric), f64(force_A)
    ad = None if adapt is None else np.ascontiguousarray(adapt, dtype=np.int64)
    out = dict(samples=np.full((S, d), np.nan), grads=np.full((S, d), np.nan), accept=np.zeros(S, np.uint8),
               logtarget=np.full(S, np.nan), eps=np.full(S, np.nan), leaps=np.zeros(S, np.int64), alpha=np.full(S, np.nan),
               ndoublings=np.zeros(S, np.int64), win_A=np.full((64, d, d), np.nan), A=np.full((d, d), np.nan))
    nev, nwin = C.c_int64(0), C.c_int64(0)
    i64 = lambda a: a.ctypes.data_as(C.POINTER(C.c_int64))
    rc = ND.orc_run_nuts_dense(C.byref(om._c), C.byref(smp), C.byref(O._Range(first, stp, last)), _p(init), seed, chain, _p(zn),
                               _p(im), None if ad is None else i64(ad), _p(fa), _p(out["samples"]), _p(out["grads"]),
                               out["accept"].ctypes.data_as(C.POINTER(C.c_uint8)), _p(out["logtarget"]), _p(out["eps"]),
                               i64(out["leaps"]), _p(out["alpha"]), i64(out["ndoublings"]), C.byref(nev), _p(out["win_A"]),
                               C.byref(nwin), _p(out["A"]))
    out["rc"], out["n_grad_evals"], out["n_win"] = rc, nev.value, nwin.value
    out["win_A"] = out["win_A"][:nwin.value]
    return out


def random_spd(r, d, lo=0.3, hi=3.0):
    """a symmetric positive definite matrix with eigenvalues in [lo, hi] and random eigenvectors, exactly symmetric"""
    Q, _ = np.linalg.qr(r.standard_normal((d, d)))
    A = (Q * r.uniform(lo, hi, d)) @ Q.T
    return (A + A.T) / 2


def correlated_linear(Nr=200, d=3, seed=5):
    """linear regression (noise sd 1, prior sd 1) whose first two features are nearly collinear: an exact Gaussian posterior
    with precision X'X + I and a correlation near -0.98 between the first two coefficients"""
    r = np.random.default_rng(seed)
    Z = r.standard_normal((Nr, d))
    X = Z.copy()
    X[:, 1] = Z[:, 0] + 0.2 * Z[:, 1]
    beta = r.standard_normal(d) / 2
    y = X @ beta + r.standard_normal(Nr)
    prec = X.T @ X + np.eye(d)
    cov = np.linalg.inv(prec)
    cov = (cov + cov.T) / 2                                                 # exactly symmetric, to be usable as a metric
    return X, y, prec, cov, cov @ (X.T @ y)


def regularised(n, cov):
    """what Stan's estimator targets from a window of n draws: (n / (n + 5)) cov + 1e-3 (5 / (n + 5)) I"""
    return (n / (n + 5.0)) * cov + 1e-3 * (5.0 / (n + 5.0)) * np.eye(cov.shape[0])


# ---- CPU: the restatement ---------------------------------------------------------------------------------------------
FAMS = [("normal_dsl", 5, (1.0, 2.0)), ("normal_fn", 3, ()), ("abs_normal", 4, (1.0, 0.5))]


@pytest.mark.parametrize("fam,d,hy", FAMS)
def test_diagonal_and_identity_as_dense_are_bit_identical(O, ND, fam, d, hy):
    om = O.Model(fam, d, hyper=hy)
    rngt = (31, 1, 60)
    r = np.random.default_rng(d)
    keys = ("samples", "grads", "accept", "logtarget", "eps", "leaps", "alpha", "ndoublings")
    for c in range(12):
        minv = np.exp(r.uniform(np.log(0.2), np.log(5.0), d))
        ref = run_nuts_metric(O, ND, om, rngt, np.full(d, 1.5), 4, c, inv_metric=minv)
        den = run_nuts_dense(O, ND, om, rngt, np.full(d, 1.5), 4, c, inv_metric=np.diag(minv))
        assert ref["rc"] == 0 and den["rc"] == 0
        for k in keys:
            assert np.array_equal(ref[k], den[k]), (c, k)
        assert den["n_grad_evals"] == ref["n_grad_evals"]
        ident = run_nuts(O, ND, om, rngt, np.full(d, 1.5), 4, c)
        for A in (None, np.eye(d)):
            den = run_nuts_dense(O, ND, om, rngt, np.full(d, 1.5), 4, c, inv_metric=A)
            for k in keys:
                assert np.array_equal(ident[k], den[k]), (c, k)


def test_linear_algebra_helpers_agree_with_numpy(ND):
    r = np.random.default_rng(0)
    for d in (1, 2, 5, 17, 60):
        A = random_spd(r, d, 0.1, 10.0)
        L = np.zeros((d, d))
        assert ND.orc_dense_cholesky(_p(A), _p(L), d) == 0
        Lr = np.linalg.cholesky(A)
        assert np.max(np.abs(L - Lr)) <= 1e-13 * np.max(np.abs(Lr)) * d, d
        z = r.standard_normal(d)
        p = np.zeros(d)
        ND.orc_dense_backsub(_p(L), _p(z), _p(p), d)
        pr = np.linalg.solve(Lr.T, z)
        assert np.allclose(p, pr, rtol=1e-11, atol=1e-13 * np.abs(pr).max()), d
        # p = L^-T z has covariance A^-1, and p' A p = z' z
        assert abs(p @ A @ p - z @ z) <= 1e-11 * (z @ z), d
        x = r.standard_normal((200, d)) @ np.linalg.cholesky(A).T + 3.0
        mean, m2 = np.zeros(d), np.zeros((d, d))
        ND.orc_welford_covar(_p(x), 200, d, _p(mean), _p(m2))
        assert np.allclose(mean, x.mean(0), rtol=1e-13, atol=1e-13)
        cov = np.atleast_2d(np.cov(x.T))
        assert np.max(np.abs(m2 / 199 - cov)) <= 1e-13 * np.max(np.abs(cov)) * 10, d
    bad = np.array([[1.0, 2.0], [2.0, 1.0]])                                # indefinite
    assert ND.orc_dense_cholesky(_p(bad), _p(np.zeros((2, 2))), 2) == -1
    nan = np.array([[1.0, np.nan], [np.nan, 1.0]])
    assert ND.orc_dense_cholesky(_p(nan), _p(np.zeros((2, 2))), 2) == -1


def _check_gaussian(x, mean, cov, label):
    """x (C, d) independent draws of N(mean, cov): whitened moments within 5 SE, KS of a projection"""
    Cn, d = x.shape
    z = (x - mean) @ np.linalg.inv(np.linalg.cholesky(cov)).T               # iid N(0, 1) coordinates
    se = 1.0 / math.sqrt(Cn)
    assert np.all(np.abs(z.mean(0)) < 5 * se), (label, z.mean(0))
    S = np.cov(z.T)
    assert np.all(np.abs(S - np.eye(d)) < 5 * math.sqrt(2.0) * se), (label, S)
    w = np.random.default_rng(1).standard_normal(d)
    w /= np.linalg.norm(w)
    p = sst.kstest(z @ w, sst.norm().cdf).pvalue
    assert p > 1e-4, (label, p)


def test_fixed_dense_metric_samples_the_exact_posterior(O, ND):
    d = 3
    X, y, prec, cov, mean = correlated_linear(d=d)
    om = O.Model("linear", d, X, y, (1.0, 1.0))
    A = 0.02 * (0.4 * np.eye(d) + 0.6 * np.ones((d, d))) + np.diag([0.0, 0.01, 0.005])   # correlation 0.6 .. 0.75
    res = run_many(lambda c: run_nuts_dense(O, ND, om, (101, 1, 130), mean + 0.1, 2024, c, inv_metric=A), range(2000))
    assert all(r["rc"] == 0 for r in res)
    _check_gaussian(np.array([r["samples"][-1] for r in res]), mean, cov, "linear, fixed dense metric")


def test_dense_adaptation_learns_the_posterior_covariance(O, ND):
    """W = 500 with Stan's buffers (windows end at steps 100, 150, 250, 450): the final A of every chain is close to the
    regularised covariance of the last window's 200 draws, and dense-adapted trees are far shorter than diagonal-adapted
    ones on a posterior with correlation -0.98"""
    d, W = 3, 500
    X, y, prec, cov, mean = correlated_linear(d=d)
    corr = cov[0, 1] / math.sqrt(cov[0, 0] * cov[1, 1])
    assert corr < -0.95, corr
    om = O.Model("linear", d, X, y, (1.0, 1.0))
    rngt = (W + 2, 1, W + 101)
    ends = stan_windows(W, *STAN)[0]
    assert ends == [100, 150, 250, 450]
    n = ends[-1] - ends[-2]
    dense = run_many(lambda c: run_nuts_dense(O, ND, om, rngt, mean, 31, c, adapt=STAN), range(200))
    diag = run_many(lambda c: run_nuts_metric(O, ND, om, rngt, mean, 31, c, adapt=STAN), range(200))
    assert all(r["rc"] == 0 and r["n_win"] == 4 for r in dense + diag)
    target = regularised(n, cov)
    err = np.array([np.linalg.norm(r["A"] - target) for r in dense]) / np.linalg.norm(target)
    # the Wishart spread of a sample covariance of n draws: E|S - cov|_F^2 = (tr(cov)^2 + |cov|_F^2) / (n - 1)
    sd = math.sqrt((np.trace(cov) ** 2 + np.sum(cov ** 2)) / (n - 1)) / np.linalg.norm(cov)
    assert np.median(err) < 1.5 * sd and np.max(err) < 6 * sd, (np.median(err), np.max(err), sd)
    assert all(np.array_equal(r["A"], r["win_A"][-1]) for r in dense)
    ld, lg = np.mean([r["leaps"].mean() for r in dense]), np.mean([r["leaps"].mean() for r in diag])
    assert ld < 0.5 * lg, (ld, lg)


def test_one_draw_window_keeps_the_metric_before_regularising(O, ND):
    """W = 151: the window ending at step 101 holds one draw, so A becomes (1/6) A + 1e-3 (5/6) I"""
    om = O.Model("normal_dsl", 2, hyper=(1.0, 2.0))
    r = run_nuts_dense(O, ND, om, (153, 1, 155), np.ones(2), 5, 0, adapt=STAN)
    assert r["rc"] == 0 and r["n_win"] == 2
    assert np.array_equal(r["win_A"][1], (1.0 / 6.0) * r["win_A"][0] + 1e-3 * (5.0 / 6.0) * np.eye(2))


def test_nuts_constructor_dense_arguments():
    import mcmc_jl_b200 as mj
    s = mj.NUTS()
    assert (s.metric, s.inv_metric, s.adapt_metric) == ("diag", None, False)
    calls = []

    class Rec:
        C = 2

        def set_metric(self, m):
            calls.append(("set_metric", np.array(m)))

        def set_dense_metric(self, m=None):
            calls.append(("dense", None if m is None else np.array(m)))

        def set_metric_adaptation(self, *a):
            calls.append(("adapt", a))
    s._set_metric(Rec(), 0, 2)
    assert calls == []
    A = random_spd(np.random.default_rng(0), 3)
    per = np.stack([A, 2 * A, 3 * A, 4 * A])
    mj.NUTS(metric="dense", inv_metric=per, adapt_metric=True, window=7)._set_metric(Rec(), 1, 4)
    assert calls[0][0] == "dense" and np.array_equal(calls[0][1], per[1:3]) and calls[1] == ("adapt", (75, 50, 7))
    calls.clear()
    mj.NUTS(metric="dense")._set_metric(Rec(), 0, 2)
    assert calls[0] == ("dense", None) and len(calls) == 1
    calls.clear()
    mj.NUTS(metric="dense", inv_metric=A)._set_metric(Rec(), 0, 2)
    assert np.array_equal(calls[0][1], A)
    assert np.array_equal(mj.NUTS(inv_metric=np.ones((2, 2))).inv_metric, np.ones((2, 2)))   # (d, d) is per-chain diagonal by default
    asym = A.copy(); asym[0, 1] += 1e-12
    indef = np.array([[1.0, 2.0], [2.0, 1.0]])
    for bad in (lambda: mj.NUTS(metric="full"), lambda: mj.NUTS(metric="dense", inv_metric=np.ones(3)),
                lambda: mj.NUTS(metric="dense", inv_metric=np.ones((2, 3))), lambda: mj.NUTS(metric="dense", inv_metric=asym),
                lambda: mj.NUTS(metric="dense", inv_metric=indef), lambda: mj.NUTS(metric="dense", inv_metric=np.full((2, 2), np.nan)),
                lambda: mj.NUTS(metric="dense", inv_metric=np.ones((2, 2, 2, 2)))):
        with pytest.raises(AssertionError):
            bad()
    with pytest.raises(AssertionError, match="matrices"):
        mj.NUTS(metric="dense", inv_metric=per)._set_metric(Rec(), 0, 3)


# ---- GPU ----------------------------------------------------------------------------------------------------------------
def _out(run, dense=True):
    out = run.fetch(); eps, leaps = run.fetch_diag()
    return dict(out=out, eps=eps, leaps=leaps, A=run.get_dense_metric() if dense else None)


def _same(a, b, sl=slice(None)):
    for k in ("samples", "grads", "accept", "logtarget"):
        assert np.array_equal(a["out"][k][sl], b["out"][k]), k
    assert np.array_equal(a["eps"][sl], b["eps"]) and np.array_equal(a["leaps"][sl], b["leaps"])


@pytest.mark.gpu
@pytest.mark.parametrize("fam", ["normal_dsl", "logistic", "linear"])
def test_diagonal_and_identity_as_dense_are_bit_identical_on_the_device(capi, ctx, fam):
    d, C = (5, 300) if fam == "normal_dsl" else (40, 256)
    if fam == "normal_dsl":
        X = y = None; hy = (1.0, 2.0); init = np.full(d, 3.0)
    else:
        X, y, hy, b0 = make_regression(fam, 2000, d, 6); init = b0
    dm = capi.DeviceModel(ctx, fam, d, X, y, hy)
    rngt = (31, 1, 45)                                                      # the step size adapts on steps 1..29
    r = np.random.default_rng(3)
    minv = np.exp(r.uniform(np.log(0.5), np.log(2.0), (C, d)))

    def one(setup):
        run = capi.DeviceRun(dm, capi.sampler_cfg("NUTS", nleaps=8), rngt, C, init, seed=21, engine="wave")
        setup(run)
        run.execute(); o = _out(run, False); run.close()
        return o
    _same(one(lambda run: None), one(lambda run: run.set_dense_metric(None)))
    _same(one(lambda run: None), one(lambda run: run.set_dense_metric(np.eye(d))))
    _same(one(lambda run: run.set_metric(minv[0])), one(lambda run: run.set_dense_metric(np.diag(minv[0]))))
    _same(one(lambda run: run.set_metric(minv)), one(lambda run: run.set_dense_metric(np.stack([np.diag(m) for m in minv]))))
    dm.close()


def _device_and_oracle(O, ND, capi, ctx, fam, d, X, y, hy, C, rngt, init, seed, A, maxd=10, s0=0, eps0=None, chains=None):
    """a device run with the dense metric A ((d, d) shared or (C, d, d)) and the restatement replaying it with the device's
    normals; s0 > 0 starts after step s0 with step size eps0, forced one step ahead"""
    first, _, last = rngt
    om, dm = O.Model(fam, d, X, y, hy), capi.DeviceModel(ctx, fam, d, X, y, hy)
    run = capi.DeviceRun(dm, capi.sampler_cfg("NUTS", nleaps=maxd, rate=0.6), rngt, C, init, seed=seed, engine="wave")
    run.set_state(s0, eps0, eps0, np.zeros(C))
    run.set_dense_metric(A)
    info = run.execute(); out = run.fetch(); eps, leaps = run.fetch_diag()
    assert np.array_equal(run.get_dense_metric(), np.broadcast_to(A, (C, d, d)))
    run.close(); dm.close()
    zn, _ = ctx.philox_draws(seed, 0, C, d, last)
    chains = range(C) if chains is None else chains
    ini = lambda c: init[c] if np.ndim(init) == 2 else init

    def one(c):
        fe = np.concatenate([np.full(s0 + 1, np.nan), eps[c]])
        return c, run_nuts_dense(O, ND, om, rngt, ini(c), seed, c, inv_metric=A if A.ndim == 2 else A[c], maxd=maxd,
                                 normals=zn[c], start_step=s0, da_state=[eps0[c], eps0[c], 0.0], force_eps=fe)
    return out, eps, leaps, dict(run_many(one, list(chains))), info


@pytest.mark.gpu
@pytest.mark.parametrize("shared", [True, False], ids=["shared", "per_chain"])
@pytest.mark.parametrize("fam,d,hy", CLOSED, ids=lambda c: str(c))
def test_closed_form_parity_with_a_dense_metric(O, ND, capi, ctx, fam, d, hy, shared):
    C, s0, K = 70, 50, 25
    r = np.random.default_rng(100 + d)
    lo, hi = (0.5, 2.0) if fam == "ou" else (0.2, 5.0)
    A = random_spd(r, d, lo, hi) if shared else np.stack([random_spd(r, d, lo, hi) for _ in range(C)])
    if fam == "ou":
        y, init, maxd = ou_series(300, 4), np.array([20.0, 0.1, 10.0]), 7
        eps0 = 0.002 * np.exp(0.3 * r.standard_normal(C))
    else:
        y, init, maxd = None, 0.5 + r.standard_normal((C, d)), 10
        eps0 = {"normal_fn": 0.8, "normal_dsl": 1.2, "abs_normal": 0.25}[fam] * np.exp(0.4 * r.standard_normal(C)) / 2
    out, eps, leaps, refs, info = _device_and_oracle(O, ND, capi, ctx, fam, d, None, y, hy, C, (s0 + 1, 1, s0 + K), init, 7, A,
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
def test_dense_adaptation_parity_bit_exact(O, ND, capi, ctx, fam, d, hy):
    """W = 60 with 5 / 5 / 5: windows end at steps 10, 20 and 55.  Stepwise, the step size and the metric of every warm-up
    step are read back and forced on the restatement, whose own metric after every window end must equal the device's bit
    for bit; the metric changes at those steps and nowhere else; the draws equal those of a one-call run."""
    C, seed, W = 64, 17, 60
    first, last = W + 2, W + 10
    rngt = (first, 1, last)
    init = 0.5 + np.random.default_rng(d).standard_normal((C, d))
    A0 = random_spd(np.random.default_rng(9), d, 0.5, 2.0)
    dm = capi.DeviceModel(ctx, fam, d, None, None, hy)

    def mk():
        run = capi.DeviceRun(dm, capi.sampler_cfg("NUTS", nleaps=10, rate=0.6), rngt, C, init, seed=seed, engine="wave")
        run.set_dense_metric(A0); run.set_metric_adaptation(5, 5, 5)
        return run
    one = mk(); one.execute(); o1 = _out(one); one.close()
    run = mk()
    fe, fA = np.full((C, last + 1), np.nan), np.tile(A0, (C, last + 1, 1, 1))
    fe[:, 1] = 1.0
    changed = []
    for i in range(1, first):                                               # after step i: the step size and metric of step i + 1
        run.execute_steps(1)
        fe[:, i + 1] = run.get_state()["leapstep"]
        fA[:, i + 1] = run.get_dense_metric()
        if not np.array_equal(fA[:, i + 1], fA[:, i]):
            changed.append(i)
    assert changed == [10, 20, 55]
    fe[:, first + 1:] = fe[:, first][:, None]
    fA[:, first + 1:] = fA[:, first][:, None]
    run.execute_steps(last - first + 1)
    o = _out(run); run.close(); dm.close()
    _same(o1, o)
    assert np.array_equal(o1["A"], o["A"]) and np.array_equal(o["A"], fA[:, first])
    assert np.array_equal(o["eps"], fe[:, first:])
    zn, _ = ctx.philox_draws(seed, 0, C, d, last)
    om = O.Model(fam, d, hyper=hy)
    refs = run_many(lambda c: run_nuts_dense(O, ND, om, rngt, init[c], seed, c, inv_metric=A0, adapt=(5, 5, 5), force_A=fA[c],
                                             force_eps=fe[c], normals=zn[c]), range(C))
    for c, ref in enumerate(refs):
        assert ref["rc"] == 0 and ref["n_win"] == 3, c
        assert np.array_equal(ref["win_A"], fA[c, [11, 21, 56]]), c
        assert np.array_equal(ref["A"], o["A"][c]), c
        for k in ("samples", "grads", "logtarget", "accept"):
            assert np.array_equal(ref[k], o["out"][k][c]), (c, k)
        assert np.array_equal(ref["leaps"], o["leaps"][c]), c
        assert np.allclose(ref["eps"], o["eps"][c], rtol=1e-9, atol=0), c
    offd = o["A"][:, 0, 1]
    assert np.any(np.abs(offd - A0[0, 1]) > 0.05)


@pytest.mark.gpu
@pytest.mark.parametrize("fam,d", REGRESSION, ids=lambda c: str(c))
def test_regression_parity_with_a_dense_metric(O, ND, capi, ctx, fam, d):
    Nrows = 997
    X, y, hy, b0 = make_regression(fam, Nrows, d, 5)
    ntiles = -(-Nrows // 32)
    s0, K = 40, 12
    r = np.random.default_rng(d + 1)
    base = (0.3 if fam == "probit" else 0.5) / math.sqrt(Nrows)
    gs = np.abs(X).sum(0)
    try:
        for C, splits, shared in ((130, 1, False), (70, 3, True), (1, ntiles + 3, False)):
            ctx.set_option("force_splits", splits)
            init = b0 + 0.05 * r.standard_normal((C, d)) / math.sqrt(d)
            A = random_spd(r, d, 0.5, 2.0) if shared else np.stack([random_spd(r, d, 0.5, 2.0) for _ in range(C)])
            eps0 = base * np.exp(0.3 * r.standard_normal(C)) / 1.5
            chains = range(C) if d <= 20 else range(0, C, 5)
            out, eps, leaps, refs, info = _device_and_oracle(O, ND, capi, ctx, fam, d, X, y, hy, C, (s0 + 1, 1, s0 + K), init, 9,
                                                             A, 8, s0, eps0, chains)
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


@pytest.mark.gpu
def test_dense_adaptation_on_a_correlated_posterior(capi, ctx):
    d, C, W = 3, 8192, 500
    X, y, prec, cov, mean = correlated_linear(d=d)
    dm = capi.DeviceModel(ctx, "linear", d, X, y, (1.0, 1.0))
    run = capi.DeviceRun(dm, capi.sampler_cfg("NUTS", nleaps=10), (W + 2, 1, W + 61), C, mean, seed=5, store_grad=False, engine="wave")
    run.set_dense_metric(None); run.set_metric_adaptation(*STAN)
    run.execute(); x = run.fetch()["samples"]; _, leaps = run.fetch_diag(); A = run.get_dense_metric()
    run.close(); dm.close()
    _check_gaussian(x[:, -1], mean, cov, "linear, adapted dense metric")
    ends = stan_windows(W, *STAN)[0]
    n = ends[-1] - ends[-2]
    target = regularised(n, cov)
    assert np.allclose(np.median(A, axis=0), target, rtol=0.1, atol=0.02 * np.abs(target).max()), (np.median(A, axis=0), target)
    err = np.linalg.norm(A - target, axis=(1, 2)) / np.linalg.norm(target)
    sd = math.sqrt((np.trace(cov) ** 2 + np.sum(cov ** 2)) / (n - 1)) / np.linalg.norm(cov)
    assert np.median(err) < 1.5 * sd, (np.median(err), sd)
    assert leaps.mean() < 8, leaps.mean()


@pytest.mark.gpu
@pytest.mark.parametrize("fam", ["normal_dsl", "logistic"])
def test_execution_paths_are_bit_identical_with_a_dense_metric(capi, ctx, fam):
    d, C, seed = (4, 200, 13) if fam == "normal_dsl" else (12, 96, 14)
    if fam == "normal_dsl":
        X = y = None; hy = (1.0, 2.0); init = np.ones(d)
    else:
        X, y, hy, b0 = make_regression(fam, 1500, d, 3); init = b0
    dm = capi.DeviceModel(ctx, fam, d, X, y, hy)
    rngt = (62, 1, 80)                                                      # W = 60, windows end at steps 10, 20, 55
    r = np.random.default_rng(2)
    mets = np.stack([random_spd(r, d, 0.5, 2.0) for _ in range(C)])

    def path(pieces=None, offset=0, n=None, rng=rngt, state=None, metric=mets, adapt=True, x0=init):
        n = n or C
        run = capi.DeviceRun(dm, capi.sampler_cfg("NUTS", nleaps=8), rng, n, x0, seed=seed, chain_offset=offset, engine="wave")
        if state is not None:
            run.set_state(*state)
        run.set_dense_metric(metric[offset:offset + n])
        if adapt:
            run.set_metric_adaptation(5, 5, 5)
        for p in (pieces or [None]):
            run.execute() if p is None else run.execute_steps(p)
        o = _out(run); o["state"] = run.get_state(); run.close()
        return o
    base = path()
    assert not np.array_equal(base["A"], mets)
    for pieces in ((7, 13, 30, 30), (10, 10, 35, 1, 24)):                  # pieces that end at and cross the window ends
        o = path(pieces)
        _same(base, o); assert np.array_equal(base["A"], o["A"])
    for opt, vals in (("poll_every", (1, 8)), ("use_graphs", (0, 1)), ("time_eval", (1,))):
        for v in vals:
            ctx.set_option(opt, v)
            try:
                o = path()
                _same(base, o); assert np.array_equal(base["A"], o["A"])
            finally:
                ctx.set_option(opt, {"poll_every": 0, "use_graphs": 1, "time_eval": 0}[opt])
    lo, hi = path(n=C // 3), path(offset=C // 3, n=C - C // 3)              # each chain adapts alone: sharding changes nothing
    _same(base, lo, slice(0, C // 3)); _same(base, hi, slice(C // 3, C))
    assert np.array_equal(base["A"], np.concatenate([lo["A"], hi["A"]]))
    # continuation with a fixed metric: a run to step 65, then a new run from its state gives the one-call run's later draws
    fixed = path(adapt=False)
    warm = path(rng=(62, 1, 65), adapt=False)
    st = warm["state"]
    cont = path(rng=(66, 1, 80), state=(65, st["leapstep"], st["dual_leapstep"], st["dualH"]), adapt=False, x0=st["pars"])
    for k in ("samples", "grads", "accept", "logtarget"):
        assert np.array_equal(fixed["out"][k][:, 4:], cont["out"][k]), k
    assert np.array_equal(fixed["eps"][:, 4:], cont["eps"]) and np.array_equal(fixed["leaps"][:, 4:], cont["leaps"])
    # a shared fixed metric equals the same matrix given per chain
    sh = path(metric=np.broadcast_to(mets[0], mets.shape).copy(), adapt=False)
    run = capi.DeviceRun(dm, capi.sampler_cfg("NUTS", nleaps=8), rngt, C, init, seed=seed, engine="wave")
    run.set_dense_metric(mets[0]); run.execute(); o = _out(run); run.close()
    _same(sh, o)
    dm.close()


@pytest.mark.gpu
def test_dense_metric_errors(capi, ctx):
    dm = capi.DeviceModel(ctx, "normal_dsl", 2, hyper=(0.0, 1.0))
    ok, I2 = np.ones(2), np.eye(2)
    for cfg, kw in ((capi.sampler_cfg("HMC"), {}), (capi.sampler_cfg("HMCDA"), dict(engine="wave")), (capi.sampler_cfg("HMC"), dict(engine="fused"))):
        run = capi.DeviceRun(dm, cfg, (1, 1, 10), 4, ok, **kw)
        for call in (lambda: run.set_dense_metric(I2), lambda: run.set_dense_metric(None), lambda: run.get_dense_metric()):
            with pytest.raises(capi.MCMCGPUError) as e:
                call()
            assert e.value.code == capi.E_ARG
        run.close()
    mk = lambda: capi.DeviceRun(dm, capi.sampler_cfg("NUTS"), (30, 1, 40), 4, ok)
    run = mk()
    with pytest.raises(capi.MCMCGPUError) as e:                             # no dense metric yet
        run.get_dense_metric()
    assert e.value.code == capi.E_ARG
    per = np.stack([I2] * 3 + [np.array([[1.0, 2.0], [2.0, 1.0]])])         # one chain's matrix is indefinite
    for bad in (np.array([[1.0, 0.5], [0.4, 1.0]]), np.array([[1.0, np.nan], [np.nan, 1.0]]), np.array([[np.inf, 0], [0, 1.0]]),
                np.array([[1.0, 2.0], [2.0, 1.0]]), np.array([[0.0, 0.0], [0.0, 1.0]]), -I2, per, np.ones((3, 2, 2)), np.ones(2)):
        with pytest.raises(capi.MCMCGPUError) as e:
            run.set_dense_metric(bad)
        assert e.value.code == capi.E_ARG
    A = np.array([[2.0, 0.5], [0.5, 1.0]])
    run.set_dense_metric(A)
    assert np.array_equal(run.get_dense_metric(), np.tile(A, (4, 1, 1)))   # before execute: the starting metric
    for call in (lambda: run.set_metric(ok), lambda: run.get_metric()):    # the diagonal calls on a dense run
        with pytest.raises(capi.MCMCGPUError) as e:
            call()
        assert e.value.code == capi.E_ARG
    run.set_metric_adaptation(5, 5, 5)
    with pytest.raises(capi.MCMCGPUError) as e:                             # adaptation needs the whole warm-up
        run.set_state(10)
    assert e.value.code == capi.E_ARG
    run.execute_steps(3)
    for call in (lambda: run.set_dense_metric(A), lambda: run.set_metric_adaptation()):
        with pytest.raises(capi.MCMCGPUError) as e:
            call()
        assert e.value.code == capi.E_STATE
    run.close()
    run = mk(); run.set_metric(ok)                                          # a diagonal run takes no dense metric
    with pytest.raises(capi.MCMCGPUError) as e:
        run.set_dense_metric(A)
    assert e.value.code == capi.E_ARG
    run.close()
    run = mk(); run.set_metric_adaptation()                                 # nor after the diagonal adaptation
    with pytest.raises(capi.MCMCGPUError) as e:
        run.set_dense_metric(A)
    assert e.value.code == capi.E_ARG
    run.close()
    run = mk(); run.set_state(10); run.set_dense_metric(A)
    with pytest.raises(capi.MCMCGPUError) as e:
        run.set_metric_adaptation()
    assert e.value.code == capi.E_ARG
    run.close()
    dm.close()


@pytest.mark.gpu
def test_end_to_end(capi, ctx):
    import mcmc_jl_b200 as mj
    d = 3
    X, y, prec, cov, mean = correlated_linear(d=d, seed=4)
    m = mj.model("linear", X=X, Y=y, vars=mean)
    batch = mj.run(m * mj.NUTS(metric="dense", adapt_metric=True) * mj.GPUMC(steps=700, burnin=601, nchains=512, seed=2))
    A = batch.inv_metric()
    assert A.shape == (512, d, d)
    n = np.diff(stan_windows(600, *STAN)[0])[-1]
    assert np.allclose(np.median(A, axis=0), regularised(n, cov), rtol=0.2, atol=0.05 * cov.max())
    assert np.array_equal(batch[3].diagnostics["inv_metric"], A[3]) and batch[3].diagnostics["inv_metric"].shape == (d, d)
    batch.close()
    c = mj.run(m * mj.NUTS(metric="dense", inv_metric=cov) * mj.SerialMC(steps=300, burnin=100))
    assert np.array_equal(c.diagnostics["inv_metric"], cov) and c.samples.shape == (200, d)
    per = np.stack([cov * s for s in np.linspace(0.5, 2.0, 8)])
    b = mj.run(m * mj.NUTS(metric="dense", inv_metric=per) * mj.GPUMC(steps=60, burnin=20, nchains=8))
    assert np.array_equal(b.inv_metric(), per)
    b.close()
    with pytest.raises(AssertionError, match="matrices"):                   # (nchains, d, d) must match the runner's chains
        mj.run(m * mj.NUTS(metric="dense", inv_metric=per) * mj.GPUMC(steps=60, burnin=20, nchains=4))
