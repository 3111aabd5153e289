"""Multinomial NUTS (mcmcgpu_run_set_nuts_transition, mj.NUTS(transition="multinomial")): the C restatement
tests/nuts_multinomial_oracle.c against a second, scalar Python restatement, its invariants, exact targets, the dual
averaging and divergences on the CPU; the host API; and on the GPU nuts_kernel's multinomial instantiations against the C
restatement -- bit for bit on the closed-form families for every metric, through adaptation windows, on the regression
families within the suite's draw-matched tolerances -- plus statistics, execution paths, errors and an end-to-end run."""
import ctypes as C
import math
import os
import subprocess
import tempfile

import numpy as np
import pytest
from scipy import stats as sst

from conftest import make_regression, ou_series
from test_nuts import CLOSED, LEAF, REGRESSION, TARGETS, TREE, _check_exact, run_many, u01
from test_nuts_dense import _check_gaussian, correlated_linear, random_spd, regularised
from test_nuts_metric import stan_windows

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
UNIT, DIAG, DENSE = 0, 1, 2


@pytest.fixture(scope="session")
def NMN(O):
    """tests/nuts_multinomial_oracle.c with the other NUTS restatements and the oracle (same flags as oracle/Makefile)"""
    tmp = tempfile.mkdtemp(prefix="nuts_multinomial_oracle_")
    so = os.path.join(tmp, "libnuts_multinomial_oracle.so")
    src = ["nuts_multinomial_oracle.c", "nuts_dense_oracle.c", "nuts_metric_oracle.c", "nuts_oracle.c"]
    subprocess.check_call(["gcc", "-O3", "-std=gnu99", "-ffp-contract=off", "-fPIC", "-shared", "-o", so] +
                          [os.path.join(ROOT, "tests", f) for f in src] + [os.path.join(ROOT, "oracle", "mcmc_oracle.c"), "-lm"])
    L = C.CDLL(so)
    dp, i64p, u8p = C.POINTER(C.c_double), C.POINTER(C.c_int64), C.POINTER(C.c_uint8)
    L.orc_run_nuts_multinomial.restype = C.c_int32
    L.orc_run_nuts_multinomial.argtypes = [C.POINTER(O._Model), C.POINTER(O._Sampler), C.POINTER(O._Range), dp, C.c_uint64,
                                           C.c_uint64, dp, C.c_int32, dp, dp, dp, dp, u8p, dp, dp, i64p, dp, dp, u8p, i64p]
    L.orc_nuts_slot_uniform.restype = C.c_double
    L.orc_nuts_slot_uniform.argtypes = [C.c_uint64, C.c_uint64, C.c_uint32, C.c_uint32]
    L.orc_log_sum_exp.restype = C.c_double
    L.orc_log_sum_exp.argtypes = [C.c_double, C.c_double]
    return L


def _p(a):
    return None if a is None else a.ctypes.data_as(C.POINTER(C.c_double))


def run_mn(O, NMN, om, rngt, init, seed, chain, metric=UNIT, inv_metric=None, force_metric=None, maxd=10, rate=0.6,
           force_eps=None, start_step=0, da_state=None, normals=None):
    """one restated multinomial chain; inv_metric (d,) or (d, d); force_metric (last+1, d) or (last+1, d, d)"""
    first, stp, last = rngt
    d = om.d
    S = (last - first) // stp + 1
    smp = O.sampler("HMCDA", nleaps=maxd, rate=rate, force_eps=force_eps, start_step=start_step, da_state=da_state)
    f64 = lambda a: None if a is None else np.ascontiguousarray(a, dtype=np.float64)
    init = np.ascontiguousarray(np.broadcast_to(init, (d,)), dtype=np.float64)
    zn, im, fm = (None if normals is None else f64(normals[:last + 1])), f64(inv_metric), f64(force_metric)
    out = dict(samples=np.full((S, d), np.nan), grads=np.full((S, d), np.nan), accept=np.zeros(S, np.uint8),
               logtarget=np.full(S, np.nan), eps=np.full(S, np.nan), leaps=np.zeros(S, np.int64),
               accept_stat=np.full(S, np.nan), energy=np.full(S, np.nan), divergent=np.zeros(S, np.uint8))
    nev = C.c_int64(0)
    u8 = lambda a: a.ctypes.data_as(C.POINTER(C.c_uint8))
    rc = NMN.orc_run_nuts_multinomial(C.byref(om._c), C.byref(smp), C.byref(O._Range(first, stp, last)), _p(init), seed, chain,
                                      _p(zn), metric, _p(im), _p(fm), _p(out["samples"]), _p(out["grads"]), u8(out["accept"]),
                                      _p(out["logtarget"]), _p(out["eps"]), out["leaps"].ctypes.data_as(C.POINTER(C.c_int64)),
                                      _p(out["accept_stat"]), _p(out["energy"]), u8(out["divergent"]), C.byref(nev))
    out["rc"], out["n_grad_evals"] = rc, nev.value
    return out


# ---- a second restatement: recursive scalar Python with the C library's exp / log1p -------------------------------------
def _lse(a, b):
    l1pe = lambda x: x + math.log1p(math.exp(-x)) if x > 0.0 else math.log1p(math.exp(x))
    if a == -math.inf:
        return b
    if a == math.inf and b == math.inf:
        return math.inf
    return a + l1pe(b - a) if a > b else b + l1pe(a - b)


def _dot(a, b):
    s = 0.0
    for x, y in zip(a, b):
        s += x * y
    return s


def py_multinomial(O, om, init, seed, chain, normals, eps, nsteps, maxd, metric=UNIT, minv=None, A=None):
    """nsteps steps at the fixed step size eps from init: per step (sample, moved, leaps, accept_stat, energy, divergent)
    and the choices made at every merge (slot, chosen side)"""
    d = om.d
    if metric == DENSE:                                                     # L = chol(A), the pinned order
        L = [[0.0] * d for _ in range(d)]
        for j in range(d):
            s = A[j][j]
            for k in range(j):
                s -= L[j][k] * L[j][k]
            L[j][j] = math.sqrt(s)
            for i in range(j + 1, d):
                t = A[i][j]
                for k in range(j):
                    t -= L[i][k] * L[j][k]
                L[i][j] = t / L[j][j]

    def sharp(p):
        if metric == UNIT:
            return list(p)
        if metric == DIAG:
            return [minv[j] * p[j] for j in range(d)]
        out = []
        for j in range(d):
            s = 0.0
            for k in range(d):
                s += A[j][k] * p[k]
            out.append(s)
        return out

    def evalg(th):
        lt, g = om.evalallg(np.array(th))
        return float(lt), [float(x) for x in g]

    crit = lambda sm, sp, rho: _dot(sm, rho) > 0.0 and _dot(sp, rho) > 0.0
    uslot = lambda step, block: u01(O.philox((chain & 0xFFFFFFFF, chain >> 32, step, block), (seed & 0xFFFFFFFF, seed >> 32)))
    pars = [float(x) for x in init]
    lt, grad = evalg(pars)
    steps, choices = [], []
    for i in range(1, nsteps + 1):
        z = [float(x) for x in normals[i]]
        if metric == UNIT:
            p0 = z
        elif metric == DIAG:
            p0 = [z[j] / math.sqrt(minv[j]) for j in range(d)]
        else:
            p0 = [0.0] * d
            for j in range(d - 1, -1, -1):
                s = z[j]
                for k in range(j + 1, d):
                    s -= L[k][j] * p0[k]
                p0[j] = s / L[j][j]
        H0 = -lt + 0.5 * _dot(sharp(p0), p0)
        st = dict(n=0, sm=0.0, div=False)

        def build(end, depth, e):
            """(valid, block) of 2^depth leaves from end = [th, p, g, lt], which it advances"""
            if depth == 0:
                th, p, g = end[0], end[1], end[2]
                p = [p[j] + (0.5 * g[j]) * e for j in range(d)]
                sp = sharp(p)
                th = [th[j] + e * sp[j] for j in range(d)]
                lt1, g = evalg(th)
                p = [p[j] + (0.5 * g[j]) * e for j in range(d)]
                sp = sharp(p)
                h = -lt1 + 0.5 * _dot(sp, p)
                end[:] = [th, p, g, lt1]
                st["n"] += 1
                if math.isnan(h):
                    h = math.inf
                if h - H0 > 1000.0:
                    st["div"] = True
                st["sm"] += 1.0 if H0 - h > 0.0 else math.exp(H0 - h)
                return not st["div"], dict(lsw=H0 - h, rho=list(p), pb=p, sb=sp, pe=p, se=sp, prop=(th, g, lt1, h))
            ok, Lb = build(end, depth - 1, e)
            if not ok:
                return False, None
            kL = st["n"] - 1
            ok, Rb = build(end, depth - 1, e)
            if not ok:
                return False, None
            lsw = _lse(Lb["lsw"], Rb["lsw"])
            take = Rb["lsw"] > lsw or uslot(i, LEAF + kL) < math.exp(Rb["lsw"] - lsw)
            choices.append((i, LEAF + kL, take))
            rho = [Lb["rho"][j] + Rb["rho"][j] for j in range(d)]
            ok = crit(Lb["sb"], Rb["se"], rho) and crit(Lb["sb"], Rb["sb"], [Lb["rho"][j] + Rb["pb"][j] for j in range(d)]) \
                and crit(Lb["se"], Rb["se"], [Rb["rho"][j] + Lb["pe"][j] for j in range(d)])
            return ok, dict(lsw=lsw, rho=rho, pb=Lb["pb"], sb=Lb["sb"], pe=Rb["pe"], se=Rb["se"],
                            prop=Rb["prop"] if take else Lb["prop"])

        s0 = sharp(p0)
        fwd_end, bck_end = [pars, p0, grad, lt], [pars, p0, grad, lt]
        B = dict(rho=p0, pm=p0, sm=s0, pp=p0, sp=s0)                         # backward part: - and + ends
        F = dict(rho=p0, pm=p0, sm=s0, pp=p0, sp=s0)
        rho, lsw, sample, sh, moved = p0, 0.0, (pars, grad, lt), H0, False
        for j in range(maxd):
            fwd = uslot(i, TREE + 2 * j) >= 0.5
            if fwd:
                B = dict(rho=rho, pm=B["pm"], sm=B["sm"], pp=F["pp"], sp=F["sp"])
                ok, sub = build(fwd_end, j, eps)
                if ok:
                    F = dict(rho=sub["rho"], pm=sub["pb"], sm=sub["sb"], pp=sub["pe"], sp=sub["se"])
            else:
                F = dict(rho=rho, pm=B["pm"], sm=B["sm"], pp=F["pp"], sp=F["sp"])
                ok, sub = build(bck_end, j, -eps)
                if ok:
                    B = dict(rho=sub["rho"], pm=sub["pe"], sm=sub["se"], pp=sub["pb"], sp=sub["sb"])
            if not ok:
                break
            take = sub["lsw"] > lsw or uslot(i, TREE + 2 * j + 1) < math.exp(sub["lsw"] - lsw)
            choices.append((i, TREE + 2 * j + 1, take))
            if take:
                th, g, ltp, h = sub["prop"]
                sample, sh, moved = (th, g, ltp), h, True
            lsw = _lse(lsw, sub["lsw"])
            rho = [B["rho"][q] + F["rho"][q] for q in range(d)]
            if not (crit(B["sm"], F["sp"], rho) and crit(B["sm"], F["sm"], [B["rho"][q] + F["pm"][q] for q in range(d)])
                    and crit(B["sp"], F["sp"], [F["rho"][q] + B["pp"][q] for q in range(d)])):
                break
        pars, grad, lt = sample
        steps.append(dict(sample=list(pars), moved=moved, leaps=st["n"], accept_stat=st["sm"] / st["n"], energy=sh,
                          divergent=st["div"], H0=H0))
    return steps, choices


# ---- CPU: the two restatements, invariants, slots ------------------------------------------------------------------------
PY_CASES = [("normal_dsl", 1, (1.0, 2.0), UNIT, 1.3), ("normal_fn", 2, (), UNIT, 0.9), ("abs_normal", 2, (1.0, 0.5), DIAG, 0.4),
            ("normal_dsl", 2, (1.0, 2.0), DENSE, 1.1), ("normal_fn", 2, (), UNIT, 40.0)]


@pytest.mark.parametrize("fam,d,hy,metric,eps", PY_CASES, ids=lambda c: str(c))
def test_c_restatement_equals_python_restatement(O, NMN, fam, d, hy, metric, eps):
    om = O.Model(fam, d, hyper=hy)
    K = 6
    minv = [0.5, 2.0][:d] if metric == DIAG else None
    A = [[1.5, 0.6], [0.6, 0.8]] if metric == DENSE else None
    inv = minv if metric == DIAG else A
    nchoice, ndiv = 0, 0
    for c in range(8):
        zn = np.random.default_rng(100 + c).standard_normal((K + 1, d))
        init = np.full(d, 0.7)
        ref = run_mn(O, NMN, om, (1, 1, K), init, 5, c, metric=metric, inv_metric=inv, maxd=6, normals=zn,
                     force_eps=np.full(K + 1, eps))
        assert ref["rc"] == 0
        py, choices = py_multinomial(O, om, init, 5, c, zn, eps, K, 6, metric, minv, A)
        nchoice += len(choices)
        for s, st in enumerate(py):
            assert ref["samples"][s].tolist() == st["sample"], (c, s)
            assert ref["accept"][s] == st["moved"] and ref["leaps"][s] == st["leaps"], (c, s)
            assert ref["divergent"][s] == st["divergent"], (c, s)
            assert ref["accept_stat"][s] == st["accept_stat"] and ref["energy"][s] == st["energy"], (c, s)
            ndiv += st["divergent"]
    if eps > 10:                                                            # far past stability: the first leaves diverge
        assert ndiv > 0
    else:
        assert nchoice > 20


def test_log_sum_exp_rule(NMN):
    inf = math.inf
    for a, b in ((-inf, 3.0), (-inf, -inf), (inf, inf), (2.0, -1.0), (-1.0, 2.0), (0.5, 0.5), (700.0, -800.0), (-1e-300, 1e-300)):
        assert NMN.orc_log_sum_exp(a, b) == _lse(a, b), (a, b)
    assert NMN.orc_log_sum_exp(-inf, 3.0) == 3.0 and NMN.orc_log_sum_exp(inf, inf) == inf
    assert abs(NMN.orc_log_sum_exp(1.0, 2.0) - math.log(math.e + math.e ** 2)) < 1e-15


@pytest.mark.parametrize("fam,d,hy,maxd,metric", [("normal_dsl", 5, (1.0, 2.0), 10, UNIT), ("normal_fn", 3, (), 3, DIAG),
                                                  ("abs_normal", 2, (1.0, 0.5), 4, DENSE)])
def test_oracle_invariants(O, NMN, fam, d, hy, maxd, metric):
    om = O.Model(fam, d, hyper=hy)
    K = 120
    inv = None if metric == UNIT else (np.linspace(0.5, 2.0, d) if metric == DIAG else random_spd(np.random.default_rng(1), d, 0.5, 2.0))
    res = run_many(lambda c: (c, run_mn(O, NMN, om, (1, 1, K), np.ones(d), 11, c, metric=metric, inv_metric=inv, maxd=maxd, rate=0.8)),
                   range(64))
    for c, r in res:
        assert r["rc"] == 0
        assert np.all(r["leaps"] >= 1) and np.all(r["leaps"] <= 2 ** maxd - 1)
        assert r["n_grad_evals"] == 1 + r["leaps"].sum()
        assert np.all((r["accept_stat"] >= 0) & (r["accept_stat"] <= 1))
        stay = r["accept"][1:] == 0
        assert np.array_equal(r["samples"][1:][stay], r["samples"][:-1][stay])
        assert np.array_equal(r["logtarget"][1:][stay], r["logtarget"][:-1][stay])
        if metric == UNIT:                                                  # no move: the energy is H0 = -lt + 0.5 z.z
            z = np.stack([O.draw_normals(11, c, i, d) for i in range(2, K + 1)])
            H0 = -r["logtarget"][:-1] + 0.5 * np.array([sum(x * x for x in zi) for zi in z])
            assert np.allclose(r["energy"][1:][stay], H0[stay], rtol=1e-15, atol=1e-15)
    assert np.mean([r["accept"].mean() for _, r in res]) > 0.2


def test_internal_node_slots_are_distinct_and_clear_of_other_blocks():
    """every internal node of a full tree of 10 doublings draws from LEAF + (the step's index of its left half's last
    leaf): all distinct, inside the LEAF range, and clear of the normal blocks and the TREE blocks"""
    slots = []
    first = 0                                                               # the step's index of the subtree's first leaf

    def nodes(lo, n):                                                       # internal nodes of leaves lo .. lo + n - 1
        if n == 1:
            return
        nodes(lo, n // 2)
        slots.append(LEAF + lo + n // 2 - 1)
        nodes(lo + n // 2, n // 2)
    for j in range(10):
        nodes(first, 2 ** j)
        first += 2 ** j
    assert first == 1023 and len(slots) == sum(2 ** j - 1 for j in range(10))
    assert len(set(slots)) == len(slots)
    assert min(slots) >= LEAF and max(slots) < LEAF + 2 ** 10 - 1
    normal, trees = set(range(100)), set(range(TREE, TREE + 2 * 10))
    assert not (set(slots) & normal) and not (set(slots) & trees) and 0xFFFFFFFF not in slots


@pytest.mark.parametrize("fam,d,hy,mu,sd", TARGETS, ids=lambda t: str(t))
def test_oracle_samples_exact_targets(O, NMN, fam, d, hy, mu, sd):
    om = O.Model(fam, d, hyper=hy)
    B, L, Cn = 100, 130, 2000
    res = run_many(lambda c: run_mn(O, NMN, om, (B + 1, 1, L), np.full(d, 3.0), 2024, c), range(Cn))
    assert all(r["rc"] == 0 for r in res)
    _check_exact(np.array([r["samples"][-1] for r in res]), mu, sd, fam)
    assert not any(r["divergent"].any() for r in res)                     # none at an adapted step size


def test_oracle_samples_a_correlated_gaussian_with_a_dense_metric(O, NMN):
    d = 3
    X, y, prec, cov, mean = correlated_linear(d=d)
    om = O.Model("linear", d, X, y, (1.0, 1.0))
    res = run_many(lambda c: run_mn(O, NMN, om, (101, 1, 130), mean + 0.1, 2024, c, metric=DENSE, inv_metric=cov), range(2000))
    assert all(r["rc"] == 0 for r in res)
    _check_gaussian(np.array([r["samples"][-1] for r in res]), mean, cov, "linear, dense metric = the posterior covariance")


@pytest.mark.parametrize("rate", [0.6, 0.8])
def test_dual_averaging_reaches_the_target_accept_stat(O, NMN, rate):
    """the adaptation drives Stan's accept_stat to the target; at the averaged step size kept afterwards the mean sits
    somewhat above it (the average of log eps lies below the iterates), as for slice NUTS"""
    om = O.Model("normal_dsl", 5, hyper=(1.0, 2.0))
    res = run_many(lambda c: run_mn(O, NMN, om, (501, 1, 540), np.full(5, 3.0), 7, c, rate=rate), range(200))
    a = np.mean([r["accept_stat"] for r in res])
    assert rate - 0.02 < a < rate + 0.15, a


def test_divergences(O, NMN):
    """none at a stable step size; at a step size far past stability most steps diverge, a divergent step's last subtree
    stopped at that leaf, and a step whose first leaf diverged does not move"""
    om = O.Model("normal_fn", 3)
    K = 30
    ok = run_many(lambda c: run_mn(O, NMN, om, (1, 1, K), np.ones(3), 3, c, force_eps=np.full(K + 1, 0.5)), range(64))
    assert not any(r["divergent"].any() for r in ok)
    bad = run_many(lambda c: run_mn(O, NMN, om, (1, 1, K), np.ones(3), 3, c, force_eps=np.full(K + 1, 1e3)), range(64))
    div = np.array([r["divergent"] for r in bad]).astype(bool)
    leaps = np.array([r["leaps"] for r in bad])
    assert div.mean() > 0.9
    first = div & (leaps == 1)
    assert first.sum() > 0
    assert not np.array([r["accept"] for r in bad])[first].any()
    assert np.all(np.array([r["accept_stat"] for r in bad])[div] < 1.0)


# ---- host API ----------------------------------------------------------------------------------------------------------
def test_nuts_constructor_transition():
    import mcmc_jl_b200 as mj
    from mcmc_jl_b200 import _capi as capi
    assert mj.NUTS().transition == "slice" and mj.NUTS().rate == 0.6
    assert mj.NUTS(transition="multinomial").transition == "multinomial"
    for bad in ("stan", "Multinomial", None, 1):
        with pytest.raises(AssertionError):
            mj.NUTS(transition=bad)
    calls = []

    class Rec:
        C = 2

        def set_nuts_transition(self, t):
            calls.append(("transition", t))

        def set_dense_metric(self, m=None):
            calls.append(("dense", m))

        def set_metric_adaptation(self, *a):
            calls.append(("adapt", a))
    mj.NUTS()._set_metric(Rec(), 0, 2)
    assert calls == []
    mj.NUTS(transition="multinomial", metric="dense", adapt_metric=True)._set_metric(Rec(), 0, 2)
    assert calls == [("transition", capi.NUTS_MULTINOMIAL), ("dense", None), ("adapt", (75, 50, 25))]
    assert (capi.NUTS_SLICE, capi.NUTS_MULTINOMIAL) == (0, 1)


# ---- GPU ----------------------------------------------------------------------------------------------------------------
def _out(run, metric=UNIT):
    out = run.fetch(); eps, leaps = run.fetch_diag()
    o = dict(out=out, eps=eps, leaps=leaps, stats=run.fetch_nuts_stats())
    o["M"] = run.get_dense_metric() if metric == DENSE else (run.get_metric() if metric == DIAG else None)
    return o


def _same(a, b, sl=slice(None)):
    for k in ("samples", "grads", "accept", "logtarget"):
        assert np.array_equal(a["out"][k][sl], b["out"][k]), k
    assert np.array_equal(a["eps"][sl], b["eps"]) and np.array_equal(a["leaps"][sl], b["leaps"])
    for k in ("accept_stat", "energy", "divergent"):
        assert np.array_equal(a["stats"][k][sl], b["stats"][k]), k


def _set_metric(run, metric, M):
    if metric == DIAG:
        run.set_metric(M)
    elif metric == DENSE:
        run.set_dense_metric(M)


def _device_and_oracle(O, NMN, capi, ctx, fam, d, X, y, hy, C, rngt, init, seed, metric=UNIT, M=None, maxd=10, s0=0, eps0=None,
                       chains=None):
    first, _, last = rngt
    om, dm = O.Model(fam, d, X, y, hy), capi.DeviceModel(ctx, fam, d, X, y, hy)
    run = capi.DeviceRun(dm, capi.sampler_cfg("NUTS", nleaps=maxd, rate=0.6), rngt, C, init, seed=seed, engine="wave")
    run.set_nuts_transition(capi.NUTS_MULTINOMIAL)
    if s0:
        run.set_state(s0, eps0, eps0, np.zeros(C))
    _set_metric(run, metric, M)
    info = run.execute(); o = _out(run)
    run.close(); dm.close()
    zn, _ = ctx.philox_draws(seed, 0, C, d, last)
    chains = range(C) if chains is None else chains
    ini = lambda c: init[c] if np.ndim(init) == 2 else init
    per = M is not None and np.ndim(M) == (2 if metric == DIAG else 3)

    def one(c):
        kw = dict(maxd=maxd, normals=zn[c], metric=metric, inv_metric=(M[c] if per else M))
        if s0:
            kw.update(start_step=s0, da_state=[eps0[c], eps0[c], 0.0], force_eps=np.concatenate([np.full(s0 + 1, np.nan), o["eps"][c]]))
        return c, run_mn(O, NMN, om, rngt, ini(c), seed, c, **kw)
    return o, dict(run_many(one, list(chains))), info


def _check_stats(ref, o, c):
    assert np.array_equal(ref["divergent"], o["stats"]["divergent"][c]), c
    assert np.allclose(ref["accept_stat"], o["stats"]["accept_stat"][c], rtol=1e-13, atol=1e-300), c
    assert np.allclose(ref["energy"], o["stats"]["energy"][c], rtol=1e-13, atol=0), c


METRICS = [(UNIT, False), (DIAG, True), (DIAG, False), (DENSE, True), (DENSE, False)]


@pytest.mark.gpu
@pytest.mark.parametrize("metric,shared", METRICS, ids=["unit", "diag_shared", "diag_per_chain", "dense_shared", "dense_per_chain"])
@pytest.mark.parametrize("fam,d,hy", CLOSED, ids=lambda c: str(c))
def test_closed_form_parity_bit_exact(O, NMN, capi, ctx, fam, d, hy, metric, shared):
    C, s0, K = 70, 50, 25
    r = np.random.default_rng(200 + d)
    lo, hi = (0.5, 2.0) if fam == "ou" else (0.2, 5.0)
    M = None
    if metric == DIAG:
        M = np.exp(r.uniform(np.log(lo), np.log(hi), d if shared else (C, d)))
    elif metric == DENSE:
        M = random_spd(r, d, lo, hi) if shared else np.stack([random_spd(r, d, lo, hi) for _ in range(C)])
    if fam == "ou":
        y, init, maxd = ou_series(300, 4), np.array([20.0, 0.1, 10.0]), 7
        eps0 = 0.002 * np.exp(0.3 * r.standard_normal(C))
    else:
        y, init, maxd = None, 0.5 + r.standard_normal((C, d)), 10
        eps0 = {"normal_fn": 0.8, "normal_dsl": 1.2, "abs_normal": 0.25}[fam] * np.exp(0.4 * r.standard_normal(C))
        if metric != UNIT:
            eps0 = eps0 / 2
    o, refs, info = _device_and_oracle(O, NMN, capi, ctx, fam, d, None, y, hy, C, (s0 + 1, 1, s0 + K), init, 7, metric, M, maxd, s0, eps0)
    out, leaps = o["out"], o["leaps"]
    for c in range(C):
        ref = refs[c]
        assert ref["rc"] == 0
        assert np.array_equal(ref["accept"], out["accept"][c]), c
        assert np.array_equal(ref["leaps"], leaps[c]), c
        assert np.array_equal(ref["eps"], o["eps"][c]), c
        if fam == "ou":     # the OU likelihood itself agrees with the oracle to 1e-10, not bitwise (as for every sampler)
            assert np.allclose(ref["samples"], out["samples"][c], rtol=1e-10, atol=0), c
            assert np.allclose(ref["logtarget"], out["logtarget"][c], rtol=1e-10, atol=0), c
            assert np.array_equal(ref["divergent"], o["stats"]["divergent"][c]), c
            continue
        assert np.array_equal(ref["samples"], out["samples"][c]), c
        assert np.array_equal(ref["logtarget"], out["logtarget"][c]), c
        assert np.array_equal(ref["grads"], out["grads"][c]), c
        _check_stats(ref, o, c)
    assert info["n_grad_evals"] == C + int(leaps.sum())
    assert leaps.max() > 4 and out["accept"].mean() > 0.2


@pytest.mark.gpu
@pytest.mark.parametrize("metric", [DIAG, DENSE], ids=["diag", "dense"])
def test_adaptation_windows_parity(O, NMN, capi, ctx, metric):
    """W = 60 with 5 / 5 / 5 (windows end at steps 10, 20, 55), read back stepwise: the step size, metric and position
    after every warm-up step.  The metric changes exactly at the window ends, equals the regularised Welford estimate of
    the chain's window draws, and the restatement fed the step sizes and metrics reproduces every draw"""
    fam, d, hy, C, seed, W = "normal_dsl", 3, (1.0, 2.0), 64, 17, 60
    first, last = W + 2, W + 10
    rngt = (first, 1, last)
    init = 0.5 + np.random.default_rng(d).standard_normal((C, d))
    M0 = random_spd(np.random.default_rng(9), d, 0.5, 2.0) if metric == DENSE else np.linspace(0.5, 2.0, d)
    dm = capi.DeviceModel(ctx, fam, d, None, None, hy)

    def mk():
        run = capi.DeviceRun(dm, capi.sampler_cfg("NUTS", nleaps=10, rate=0.6), rngt, C, init, seed=seed, engine="wave")
        run.set_nuts_transition(capi.NUTS_MULTINOMIAL)
        _set_metric(run, metric, M0); run.set_metric_adaptation(5, 5, 5)
        return run
    one = mk(); one.execute(); o1 = _out(one, metric); one.close()
    run = mk()
    fe = np.full((C, last + 1), np.nan)
    fM = np.tile(M0, (C, last + 1) + (1,) * M0.ndim)
    pos = np.zeros((C, first, d))
    fe[:, 1] = 1.0
    changed = []
    for i in range(1, first):
        run.execute_steps(1)
        st = run.get_state()
        fe[:, i + 1], pos[:, i] = st["leapstep"], st["pars"]
        fM[:, i + 1] = run.get_dense_metric() if metric == DENSE else run.get_metric()
        if not np.array_equal(fM[:, i + 1], fM[:, i]):
            changed.append(i)
    assert changed == [10, 20, 55]
    fe[:, first + 1:] = fe[:, first][:, None]
    fM[:, first + 1:] = fM[:, first][:, None]
    run.execute_steps(last - first + 1)
    o = _out(run, metric); run.close(); dm.close()
    _same(o1, o)
    assert np.array_equal(o1["M"], o["M"])
    ends, (lo, hi) = stan_windows(W, 5, 5, 5)
    assert ends == [10, 20, 55]
    for a, b in zip([lo - 1] + ends[:-1], ends):                            # window (a, b]: its draws are steps max(a+1, lo) .. b
        x = pos[:, max(a + 1, lo):b + 1]
        n = x.shape[1]
        for c in range(C):
            cov = np.cov(x[c].T, ddof=1)
            want = regularised(n, cov) if metric == DENSE else (n / (n + 5.0)) * np.diag(cov) + 1e-3 * (5.0 / (n + 5.0))
            assert np.allclose(fM[c, b + 1], want, rtol=1e-12, atol=1e-15), (b, c)
    zn, _ = ctx.philox_draws(seed, 0, C, d, last)
    om = O.Model(fam, d, hyper=hy)
    refs = run_many(lambda c: run_mn(O, NMN, om, rngt, init[c], seed, c, metric=metric, force_metric=fM[c], force_eps=fe[c],
                                     normals=zn[c]), range(C))
    for c, ref in enumerate(refs):
        assert ref["rc"] == 0, c
        for k in ("samples", "grads", "logtarget", "accept"):
            assert np.array_equal(ref[k], o["out"][k][c]), (c, k)
        assert np.array_equal(ref["leaps"], o["leaps"][c]), c
        _check_stats(ref, o, c)


@pytest.mark.gpu
@pytest.mark.parametrize("fam,d", REGRESSION, ids=lambda c: str(c))
def test_regression_parity(O, NMN, capi, ctx, fam, d):
    Nrows = 997
    X, y, hy, b0 = make_regression(fam, Nrows, d, 5)
    ntiles = -(-Nrows // 32)
    s0, K = 40, 12
    r = np.random.default_rng(d + 7)
    base = (0.3 if fam == "probit" else 0.5) / math.sqrt(Nrows)
    gs = np.abs(X).sum(0)
    try:
        for C, splits in ((130, 1), (70, 3), (1, ntiles + 3)):
            ctx.set_option("force_splits", splits)
            init = b0 + 0.05 * r.standard_normal((C, d)) / math.sqrt(d)
            eps0 = base * np.exp(0.3 * r.standard_normal(C))
            chains = range(C) if d <= 10 else range(0, C, 5)
            o, refs, info = _device_and_oracle(O, NMN, capi, ctx, fam, d, X, y, hy, C, (s0 + 1, 1, s0 + K), init, 9, UNIT, None, 8,
                                               s0, eps0, chains)
            out, leaps = o["out"], o["leaps"]
            for c in chains:
                ref = refs[c]
                assert np.array_equal(ref["accept"], out["accept"][c]), (C, splits, c)
                assert np.array_equal(ref["leaps"], leaps[c]), (C, splits, c)
                assert np.array_equal(ref["divergent"], o["stats"]["divergent"][c]), (C, splits, c)
                assert np.allclose(ref["samples"], out["samples"][c], rtol=1e-9, atol=1e-12), (C, splits, c)
                assert np.allclose(ref["logtarget"], out["logtarget"][c], rtol=1e-11, atol=0), (C, splits, c)
                assert np.all(np.abs(ref["grads"] - out["grads"][c]) <= 1e-9 * gs), (C, splits, c)
            assert info["n_grad_evals"] == C + int(leaps.sum())
    finally:
        ctx.set_option("force_splits", 0)


@pytest.mark.gpu
def test_many_chains_sample_exact_targets(capi, ctx):
    d, C = 5, 8192
    dm = capi.DeviceModel(ctx, "normal_dsl", d, hyper=(1.0, 2.0))
    run = capi.DeviceRun(dm, capi.sampler_cfg("NUTS", nleaps=10), (201, 1, 260), C, np.full(d, 3.0), seed=31, store_grad=False)
    run.set_nuts_transition(capi.NUTS_MULTINOMIAL)
    run.execute(); out = run.fetch(); st = run.fetch_nuts_stats()
    run.close(); dm.close()
    _check_exact(out["samples"][:, -1], 1.0, 2.0, "normal_dsl")
    assert not st["divergent"].any() and 0.55 < st["accept_stat"].mean() < 0.8
    X, y, prec, cov, mean = correlated_linear(d=3)
    dm = capi.DeviceModel(ctx, "linear", 3, X, y, (1.0, 1.0))
    run = capi.DeviceRun(dm, capi.sampler_cfg("NUTS", nleaps=10), (502, 1, 561), C, mean, seed=5, store_grad=False, engine="wave")
    run.set_nuts_transition(capi.NUTS_MULTINOMIAL); run.set_dense_metric(None); run.set_metric_adaptation(75, 50, 25)
    run.execute(); x = run.fetch()["samples"]; _, leaps = run.fetch_diag()
    run.close(); dm.close()
    _check_gaussian(x[:, -1], mean, cov, "linear, multinomial, adapted dense metric")
    assert leaps.mean() < 8, leaps.mean()


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

    def path(pieces=None, offset=0, n=None, rng=rngt, state=None, x0=init):
        n = n or C
        run = capi.DeviceRun(dm, capi.sampler_cfg("NUTS", nleaps=8), rng, n, x0, seed=seed, chain_offset=offset, engine="wave")
        run.set_nuts_transition(capi.NUTS_MULTINOMIAL)
        if state is not None:
            run.set_state(*state)
        for p in (pieces or [None]):
            run.execute() if p is None else run.execute_steps(p)
        o = _out(run); o["state"] = run.get_state(); run.close()
        return o
    base = path()
    assert base["out"]["accept"].mean() > 0.3
    _same(base, path((7, 13, 30)))
    for opt, vals in (("poll_every", (1, 8)), ("use_graphs", (0, 1)), ("time_eval", (1,))):
        for v in vals:
            ctx.set_option(opt, v)
            try:
                _same(base, path())
            finally:
                ctx.set_option(opt, {"poll_every": 0, "use_graphs": 1, "time_eval": 0}[opt])
    lo, hi = path(n=C // 3), path(offset=C // 3, n=C - C // 3)
    _same(base, lo, slice(0, C // 3)); _same(base, hi, slice(C // 3, C))
    st = path(rng=(21, 1, 25))["state"]
    cont = path(rng=(26, 1, 50), state=(25, st["leapstep"], st["dual_leapstep"], st["dualH"]), x0=st["pars"])
    for k in ("samples", "grads", "accept", "logtarget"):
        assert np.array_equal(base["out"][k][:, 5:], cont["out"][k]), k
    assert np.array_equal(base["eps"][:, 5:], cont["eps"]) and np.array_equal(base["leaps"][:, 5:], cont["leaps"])
    for k in ("accept_stat", "energy", "divergent"):
        assert np.array_equal(base["stats"][k][:, 5:], cont["stats"][k]), k
    dm.close()


@pytest.mark.gpu
def test_slice_is_unchanged_by_setting_it(capi, ctx):
    d, C = 4, 128
    dm = capi.DeviceModel(ctx, "normal_dsl", d, hyper=(1.0, 2.0))
    outs = []
    for setit in (False, True):
        run = capi.DeviceRun(dm, capi.sampler_cfg("NUTS", nleaps=8), (21, 1, 50), C, np.ones(d), seed=4, engine="wave")
        if setit:
            run.set_nuts_transition(capi.NUTS_SLICE)
        run.execute(); out = run.fetch(); eps, leaps = run.fetch_diag(); run.close()
        outs.append(dict(out=out, eps=eps, leaps=leaps))
    for k in ("samples", "grads", "accept", "logtarget"):
        assert np.array_equal(outs[0]["out"][k], outs[1]["out"][k]), k
    assert np.array_equal(outs[0]["eps"], outs[1]["eps"]) and np.array_equal(outs[0]["leaps"], outs[1]["leaps"])
    dm.close()


@pytest.mark.gpu
def test_transition_errors(capi, ctx):
    dm = capi.DeviceModel(ctx, "normal_dsl", 2, hyper=(0.0, 1.0))
    ok = np.ones(2)

    def code(call):
        with pytest.raises(capi.MCMCGPUError) as e:
            call()
        return e.value.code
    for cfg, kw in ((capi.sampler_cfg("HMC"), {}), (capi.sampler_cfg("HMCDA"), dict(engine="wave"))):
        run = capi.DeviceRun(dm, cfg, (1, 1, 10), 4, ok, **kw)
        assert code(lambda: run.set_nuts_transition(capi.NUTS_MULTINOMIAL)) == capi.E_ARG
        run.execute()
        assert code(lambda: run.fetch_nuts_stats()) == capi.E_ARG
        run.close()
    run = capi.DeviceRun(dm, capi.sampler_cfg("NUTS"), (5, 1, 10), 4, ok)
    for bad in (2, -1, 7):
        assert code(lambda: run.set_nuts_transition(bad)) == capi.E_ARG
    run.execute()
    assert code(lambda: run.fetch_nuts_stats()) == capi.E_ARG                # a slice run keeps no statistics
    run.close()
    run = capi.DeviceRun(dm, capi.sampler_cfg("NUTS"), (5, 1, 10), 4, ok)
    run.set_nuts_transition(capi.NUTS_MULTINOMIAL)
    assert code(lambda: run.fetch_nuts_stats()) == capi.E_STATE              # nothing executed yet
    run.execute_steps(2)
    for t in (capi.NUTS_SLICE, capi.NUTS_MULTINOMIAL):
        assert code(lambda: run.set_nuts_transition(t)) == capi.E_STATE
    run.execute()
    st = run.fetch_nuts_stats()
    assert st["accept_stat"].shape == (4, 6) and st["divergent"].dtype == bool
    run.close(); dm.close()


@pytest.mark.gpu
def test_end_to_end(capi, ctx):
    import mcmc_jl_b200 as mj
    d = 3
    X, y, prec, cov, mean = correlated_linear(d=d, seed=4)
    m = mj.model("linear", X=X, Y=y, vars=mean)
    batch = mj.run(m * mj.NUTS(transition="multinomial", metric="dense", adapt_metric=True) *
                   mj.GPUMC(steps=700, burnin=601, nchains=512, seed=2))
    st = batch.nuts_stats()
    S = batch.arrays()["samples"].shape[1]
    assert set(st) == {"accept_stat", "energy", "divergent"} and all(v.shape == (512, S) for v in st.values())
    assert st["divergent"].dtype == bool and not st["divergent"].any()
    assert 0.5 < st["accept_stat"].mean() < 0.9 and np.all(np.isfinite(st["energy"]))
    n = np.diff(stan_windows(600, 75, 50, 25)[0])[-1]
    assert np.allclose(np.median(batch.inv_metric(), axis=0), regularised(n, cov), rtol=0.2, atol=0.05 * cov.max())
    ch = batch[7]
    for k in ("accept_stat", "energy", "divergent"):
        assert np.array_equal(ch.diagnostics[k], st[k][7]), k
    assert abs(np.mean(batch.arrays()["samples"][:, -1] @ np.linalg.inv(cov) @ np.ones(d)) - mean @ np.linalg.inv(cov) @ np.ones(d)) < 1.0
    batch.close()
    c = mj.run(m * mj.NUTS() * mj.SerialMC(steps=60, burnin=20))                # slice runs keep today's keys
    assert "accept_stat" not in c.diagnostics and "divergent" not in c.diagnostics
    c = mj.run(m * mj.NUTS(transition="multinomial") * mj.SerialMC(steps=60, burnin=20))
    assert c.diagnostics["energy"].shape == (40,) and c.diagnostics["divergent"].dtype == bool
