"""K1 (csrc/k1_regress.cu) at every compiled variant against an extended-precision reference.

`launch_f` instantiates the likelihood kernel for 18 feature-block counts DK (d <= 8 DK) in each of the three regression
families, and the variants differ in compile-time constants: resident CTAs and ring depth, the width of the shared-memory
copy of the probit link table (|z| < 8, |z| < 4 or none, `k1_probit_half`), the unrolled DK x 2 gradient accumulators and the
fused-leapfrog epilogue.  The reference below is independent of the oracle (oracle/mcmc_oracle.c, a double-precision
restatement) and more precise than the kernel: eta = X beta and X'r in long double (64-bit mantissa), the links in long
double or from erfcx.  The tests compare every chain of a ragged problem at the smallest and largest d of every compiled
DK, pin down the reference itself on the CPU, and check invariants that need no reference at all: a chain's numbers do not
depend on which copy of the probit table its warp reads, nor on where in the chain tiles it sits.
"""
import math
import os
import re
from functools import lru_cache

import numpy as np
import pytest
from scipy.special import erfcx

from conftest import ROOT, make_regression

FAMS = ("linear", "logistic", "probit")
HYPER = {"linear": (3.0, 0.7), "logistic": (1.0, -1.0), "probit": (10.0,)}
U = 2.0 ** -53                  # unit roundoff of binary64
EPS = np.finfo(float).eps       # 2 U
# K1's sums (eta over <= 200 features, the link terms and X'r over <= 2100 rows, then the split fold) accumulate one
# rounding per addition; such errors grow like a random walk, ~sqrt(n) ulp of the summed magnitudes: 64 = sqrt(4096).
C_U = 64
LEGACY = 1e-12                  # the suite's criterion against the oracle (_lt_grad_check); no tolerance here is looser
PROBIT_W_ABS = 1.8e-15          # absolute error of the table's phi/Phi for z >= 0 (tools/gen_probit_table.py, k1_regress.cu)
PI = np.longdouble("3.14159265358979323846264338327950288")
LOG2PI = np.log(2 * PI)
LN_SQRT_2PI = LOG2PI / 2

# compiled feature-block counts (k1_round_dk) and the d range each one serves
COMPILED_DK = tuple(range(1, 17)) + (20, 25)


def _d_range(dk):
    lo = {20: 129, 25: 161}.get(dk, 8 * dk - 7)
    return lo, {20: 160, 25: 200}.get(dk, 8 * dk)


def _dk(d):
    return next(k for k in COMPILED_DK if _d_range(k)[0] <= d <= _d_range(k)[1])


SWEEP_D = sorted({x for k in COMPILED_DK for x in _d_range(k)})
# probit: which copy of the link table the variant keeps in shared memory (k1_probit_half from k1_smem_base)
PSH = {k: (4 if 8 <= k <= 10 else 0 if (11 <= k <= 13 or k == 25) else 8) for k in COMPILED_DK}
# one d per resident-CTA class (DK <= 4: 3 CTAs, or 2 with a 4-deep ring for probit; 5..13: 2; >= 14: 1)
CTA_CLASS_D = (29, 75, 161)


# ---- the extended-precision reference ---------------------------------------------------------------------------------
def _log_ndtr_w(z):
    """log Phi(z) and W(z) = phi(z)/Phi(z) for long-double z, from one scaled complementary error function:
    z < 0:  Phi = exp(-v^2) erfcx(v) / 2, v = -z/sqrt2  ->  log Phi = -v^2 + log(erfcx(v)/2),  W = sqrt(2/pi)/erfcx(v)
    z >= 0: Phi = 1 - c, c = exp(-v^2) erfcx(v) / 2, v = z/sqrt2  ->  log Phi = log1p(-c),  W = phi(z)/(1 - c)
    erfcx is SciPy's double-precision one (Faddeeva package, ~1e-15 relative; rounding v to double moves it by at most
    2^-53 relative, since |v d log erfcx / dv| <= 1); v^2, exp, log and the division are long double."""
    z = np.asarray(z, dtype=np.longdouble)
    v = np.abs(z) / np.sqrt(np.longdouble(2))
    ex = erfcx(v.astype(np.float64)).astype(np.longdouble)
    e2 = np.exp(-v * v)
    c = np.longdouble(0.5) * e2 * ex
    neg = z < 0
    with np.errstate(divide="ignore", invalid="ignore"):
        lphi = np.where(neg, -v * v + np.log(np.longdouble(0.5) * ex), np.log1p(-c))
        phi = e2 / np.sqrt(2 * PI)
        w = np.where(neg, np.sqrt(2 / PI) / ex, phi / (1 - c))
    return lphi, w


def _link(fam, eta, y, hyper):
    """elementwise log-likelihood term l, r = dl/deta, r' = dr/deta, in long double (eta: rows x chains)"""
    y = np.asarray(y, dtype=np.longdouble)
    one = np.longdouble(1)
    with np.errstate(over="ignore", invalid="ignore", divide="ignore"):
        if fam == "linear":
            nsd = np.longdouble(hyper[1])
            resid = y - eta
            ll = -(LN_SQRT_2PI + resid * resid / (2 * nsd * nsd) + np.log(nsd))
            return ll, resid / (nsd * nsd), np.full_like(eta, -one / (nsd * nsd))
        if fam == "logistic":
            # prob = 1 / (1 + exp(sign eta)) (examples/logistic_regression.jl:18); Bernoulli: log p if y != 0 else log(1 - p)
            x = np.longdouble(hyper[1]) * eta
            p, q = one / (one + np.exp(x)), one / (one + np.exp(-x))            # p and 1 - p, neither by subtraction
            y1 = y != 0
            ll = np.where(y1, -np.logaddexp(np.longdouble(0), x), -np.logaddexp(np.longdouble(0), -x))
            sgn = np.longdouble(hyper[1])
            return ll, np.where(y1, -sgn * q, sgn * p), -p * q
        # probit, examples/probit_regression.jl:29,39-40: l = y log Phi(eta) + (1 - y) log Phi(-eta)
        lp, wp = _log_ndtr_w(eta)
        lm, wm = _log_ndtr_w(-eta)
        lp = np.where(np.isneginf(lp.astype(np.float64)), -np.inf, lp)       # where binary64's log Phi is -Inf: 0 * -Inf = NaN
        lm = np.where(np.isneginf(lm.astype(np.float64)), -np.inf, lm)
        ll = lp * y + lm * (one - y)
        r = y * wp - (one - y) * wm
        dr = -y * wp * (eta + wp) - (one - y) * wm * (wm - eta)                # W' = -W (z + W)
        return ll, r, dr


def _reference(fam, X, y, hyper, B):
    """log-target, gradient and the per-chain tolerances of a K1 evaluation (see ref_logtarget_grad and _tolerances)"""
    X, B = np.asarray(X, dtype=np.float64), np.atleast_2d(np.asarray(B, dtype=np.float64))
    XL, BL = X.astype(np.longdouble), B.astype(np.longdouble)
    y = np.asarray(y, dtype=np.float64)
    eta = XL @ BL.T                                                           # rows x chains
    ll, r, dr = _link(fam, eta, y[:, None], hyper)
    psd = np.longdouble(hyper[0])
    with np.errstate(over="ignore", invalid="ignore"):
        if fam == "probit":                                                   # logpdf(MvNormal(0, psd^2 I), beta)
            d = B.shape[1]
            prior = -0.5 * (d * LOG2PI + d * np.log(psd * psd)) - 0.5 * (BL * BL).sum(1) / (psd * psd)
        else:                                                                 # sum_j logpdf(Normal(0, psd), beta_j)
            prior = -(LN_SQRT_2PI + BL * BL / (2 * psd * psd) + np.log(psd)).sum(1)
        lt = prior + ll.sum(0)
        g = (XL.T @ r).T - BL / (psd * psd)
    bad = np.zeros(B.shape[0], dtype=bool)
    with np.errstate(over="ignore", invalid="ignore"):                      # support as binary64 decides it
        if fam == "linear":
            bad = ~np.all(np.isfinite(ll.astype(np.float64)), axis=0)
        elif fam == "logistic":
            # log of p = 1/(1 + exp(x)), or of 1 - p formed by subtraction: -Inf where that is 0 (or NaN)
            xd = (hyper[1] * eta).astype(np.float64)
            pd = 1.0 / (1.0 + np.exp(xd))
            arg = np.where(y[:, None] != 0, pd, 1.0 - pd)
            bad = ~np.all(arg > 0, axis=0)
        if fam != "probit":
            bad |= ~np.isfinite(prior.astype(np.float64))
        lt = np.where(bad, -np.inf, lt)
        g = np.where(bad[:, None], 0, g)
    return dict(X=X, y=y, eta=eta, ll=ll, r=r, dr=dr, prior_terms=BL, lt=lt, g=g, bad=bad, fam=fam, hyper=hyper)


def ref_logtarget_grad(fam, X, y, hyper, B):
    """log-target (C,) and gradient (C, d) of the regression family at each row of B, in long double.

    Same model, prior, sign conventions and out-of-support semantics as the oracle (oracle/mcmc_oracle.c:98-248):
    linear and logistic give (-Inf, zeros) where binary64's likelihood is not finite; probit propagates NaN from 0 * -Inf.
    Error bound: eta and X'r carry long-double rounding, ~n 2^-64 of the summed magnitudes (<= 2.2e-16 of them at
    n <= 2000); the linear and logistic links are long double (a few 2^-64 relative); probit's log Phi and phi/Phi come from
    SciPy's double erfcx, <= 1.2e-15 relative in erfcx, hence <= 1.2e-15 absolute in log Phi (z < 0, where |log Phi| >= log 2),
    <= 1.2e-15 relative in log Phi for z >= 0 and <= 1.2e-15 relative in phi/Phi; the sums add ~1e-16 of their magnitudes."""
    ref = _reference(fam, X, y, hyper, B)
    return ref["lt"], ref["g"]


def _tolerances(ref, general_probit=False):
    """per-chain bounds on |K1 - reference|, written from the reference's own terms:
       lt:   C_U U (sum_i |l_i| + |r_i| a_i + 1, + the prior terms)    a_i = sum_j |X_ij b_j| bounds eta's rounding, r_i carries
                                                                       it into l_i; the 1 per row is the tables' absolute error
             + 4 sum_{y_i = 0} eps p_i / (1 - p_i)                      logistic: 1 - p is formed by subtraction (the reference
                                                                       Julia code and K1 alike), so a last-bit change of p moves
                                                                       log(1 - p) by eps p / (1 - p)
       grad: C_U U (sum_i |X_ij| (|r_i| k_i + |r'_i| a_i) + |b_j| / psd^2) + PROBIT_W_ABS sum_i |X_ij| (probit)
             k_i = 1, or 1 + 2 eta_i^2 on probit's general-response path, whose exp(-(eta^2 + log 2 pi)/2 - log Phi)
             (probit_regression.jl:39) cancels terms of size eta^2 / 2
    Each is capped at the suite's criterion against the oracle (1e-12 |lt|, 1e-12 sum_i |X_ij|), so none is looser."""
    X, fam = ref["X"], ref["fam"]
    ax = np.abs(X)
    a = ax @ np.abs(ref["prior_terms"].astype(np.float64)).T                 # rows x chains
    ll, r, dr = (np.abs(np.nan_to_num(v.astype(np.float64))) for v in (ref["ll"], ref["r"], ref["dr"]))
    psd2 = float(ref["hyper"][0]) ** 2
    bt = np.abs(ref["prior_terms"].astype(np.float64))
    prior_mag = (LN_SQRT_2PI + bt * bt / (2 * psd2) + abs(math.log(math.sqrt(psd2)))).sum(1)
    lt_abs = np.abs(ref["lt"].astype(np.float64))
    tol_lt = np.minimum(C_U * U * ((ll + r * a + 1.0).sum(0) + prior_mag), LEGACY * lt_abs)
    if fam == "logistic":
        x = (ref["hyper"][1] * ref["eta"]).astype(np.float64)
        with np.errstate(over="ignore"):
            odds = np.exp(-x)                                                 # p / (1 - p), p = 1/(1 + exp(x))
        tol_lt = tol_lt + 4 * EPS * np.where(ref["y"][:, None] == 0, odds, 0.0).sum(0)
    k = 1.0 + 2.0 * ref["eta"].astype(np.float64) ** 2 if general_probit else 1.0
    tol_g = C_U * U * ((ax.T @ (r * k + dr * a)).T + bt / psd2)
    if fam == "probit":
        tol_g = tol_g + PROBIT_W_ABS * ax.sum(0)[None, :]
    tol_g = np.minimum(tol_g, LEGACY * ax.sum(0)[None, :])
    return tol_lt, tol_g


def _check_against_reference(ref, lt, g, general_probit=False, label=()):
    tol_lt, tol_g = _tolerances(ref, general_probit)
    rlt, rg = ref["lt"], ref["g"]
    for c in range(len(lt)):
        if ref["bad"][c]:
            assert lt[c] == -np.inf and np.all(g[c] == 0), (*label, c)
            continue
        assert np.isfinite(lt[c]) and np.all(np.isfinite(g[c])), (*label, c)
        err = abs(np.longdouble(lt[c]) - rlt[c])
        assert err <= tol_lt[c], (*label, c, float(err), tol_lt[c])
        gerr = np.abs(g[c].astype(np.longdouble) - rg[c]).astype(np.float64)
        assert np.all(gerr <= tol_g[c]), (*label, c, int(np.argmax(gerr / tol_g[c])), float(np.max(gerr / tol_g[c])))


# ---- problems ---------------------------------------------------------------------------------------------------------
def _rows(d):
    return 32 * (31 + d // 6) + 17                # 1009 .. 2065 rows: the last 32-row tile is always partial


# |eta| reach of the chains, one value per 8-chain warp (cycled), so that whole warps sit inside or straddle the probit
# table's shared copy (|z| < 4, < 8) and reach the libm paths (probit |z| >= 36.9; logistic |x| >= 700 in chain 5)
SCALES = {"linear": (0.01, 0.1, 0.5, 2.0), "logistic": (0.5, 3.0, 10.0, 25.0, 40.0), "probit": (0.3, 2.0, 3.5, 6.0, 9.0, 12.0, 40.0)}


@lru_cache(maxsize=None)
def sweep_problem(fam, d, C=130):
    """X = [1, linspace(-1, 1), uniform(-1, 1) ...], N not a multiple of 32; chain c reaches |eta| ~ SCALES[c // 8]"""
    rng = np.random.default_rng(1000 * d + FAMS.index(fam))
    N = _rows(d)
    s = np.linspace(-1.0, 1.0, N)
    X = np.column_stack([np.ones(N), s, rng.uniform(-1.0, 1.0, (N, max(d - 2, 0)))])[:, :d]
    reach = np.array(SCALES[fam])[(np.arange(C) // 8) % len(SCALES[fam])] * rng.uniform(0.8, 1.0, C)
    B = np.zeros((C, d))
    if fam == "linear":
        bt = rng.uniform(-1.0, 1.0, d)
        y = X @ bt + HYPER[fam][1] * rng.standard_normal(N)
        B[:] = bt + reach[:, None] * rng.standard_normal((C, d)) / math.sqrt(d)
        return X, y, B
    if d == 1:
        # logistic: eta <= 0, so that no y = 0 row has 1 - p near 0 (out of support past eta = 36.7)
        B[:, 0] = -reach if fam == "logistic" else reach * rng.choice([-1.0, 1.0], C)
    else:
        B[:, 0] = rng.uniform(-0.3, 0.3, C)
        B[:, 1] = reach if fam == "logistic" else reach * rng.choice([-1.0, 1.0], C)
        B[:, 2:] = rng.standard_normal((C, d - 2)) * (0.5 / math.sqrt(d))
    if fam == "logistic":
        # y = 1 wherever eta can be large (s > 0), and on 30 % of the other rows: y = 0 rows keep eta < ~1.5, so the
        # subtraction 1 - p stays well conditioned while y = 1 rows reach log p ~ -40
        y = ((s > 0) | (rng.random(N) < 0.3)).astype(float)
        # chain 5: x = -eta in [675, 705] (d = 1: 702), in support; the elements with |x| >= 700 take link<> and libm
        B[5] = 0.0
        B[5, 0] = -702.0 if d == 1 else -690.0
        if d > 1:
            B[5, 1] = 15.0
    else:
        y = (rng.random(N) < 0.5).astype(float)
    return X, y, B


@lru_cache(maxsize=None)
def sweep_reference(fam, d, C=130):
    X, y, B = sweep_problem(fam, d, C)
    return _reference(fam, X, y, HYPER[fam], B)


# ---- CPU: the reference itself ----------------------------------------------------------------------------------------
@pytest.mark.parametrize("fam", FAMS)
@pytest.mark.parametrize("N,d,C", [(257, 3, 4), (1009, 40, 3), (513, 113, 2), (70, 1, 3)])
def test_reference_matches_the_oracle(O, fam, N, d, C):
    X, y, hy, b0 = make_regression(fam, N, d, N + d)
    if fam == "linear":
        hy = HYPER["linear"]
    B = b0 + 0.3 * np.random.default_rng(d).standard_normal((C, d)) / math.sqrt(d)
    om = O.Model(fam, d, X, y, hy)
    lt, g = ref_logtarget_grad(fam, X, y, hy, B)
    gs = np.abs(X).sum(0)
    for c in range(C):
        olt, og = om.evalallg(B[c])
        assert abs(float(lt[c]) - olt) <= 1e-12 * abs(olt), (fam, c, float(lt[c]), olt)
        assert np.all(np.abs(g[c].astype(np.float64) - og) <= 1e-12 * gs), (fam, c)


def test_reference_out_of_support_semantics(O):
    X, y, hy, _ = make_regression("logistic", 50, 3, 1)
    B = np.array([[0.0, 800.0, 0.0], [np.nan, 0.0, 0.0], [0.1, 0.2, 0.3]])
    lt, g = ref_logtarget_grad("logistic", X, y, hy, B)
    assert lt[0] == -np.inf and np.all(g[0] == 0) and lt[1] == -np.inf and np.all(g[1] == 0) and np.isfinite(lt[2])
    Xl, yl, _, _ = make_regression("linear", 70, 3, 4)
    Bl = np.array([[np.nan, 0.0, 0.0], [1e200, 0.0, 0.0], [0.0, np.inf, 0.0], [0.3, -0.2, 0.1]])
    lt, g = ref_logtarget_grad("linear", Xl, yl, (1.0, 1.0), Bl)
    assert np.all(lt[:3] == -np.inf) and np.all(g[:3] == 0) and np.isfinite(lt[3])
    om = O.Model("linear", 3, Xl, yl, (1.0, 1.0))
    assert abs(float(lt[3]) - om.evalallg(Bl[3])[0]) <= 1e-12 * abs(float(lt[3]))
    Xp, yp, hyp, _ = make_regression("probit", 30, 2, 2)
    lt, _ = ref_logtarget_grad("probit", Xp, yp, hyp, np.array([[1e200, 1e200]]))
    assert np.isnan(lt[0]) and np.isnan(O.Model("probit", 2, Xp, yp, hyp).evalallg(np.array([1e200, 1e200]))[0])
    # the sweep's logistic chain 5 (|x| >= 700 on part of its rows) is in support
    ref = sweep_reference("logistic", 33)
    assert not ref["bad"].any() and np.isfinite(float(ref["lt"][5]))
    assert np.abs(ref["eta"][:, 5].astype(np.float64)).max() > 700


def _mpf(x):
    """a long double as an mpmath number, exactly (two doubles hold its 64-bit mantissa)"""
    import mpmath as mp
    hi = float(x)
    return mp.mpf(hi) + mp.mpf(float(np.longdouble(x) - np.longdouble(hi)))


def test_reference_links_against_mpmath():
    """element by element at 40 digits, including the far tails: long-double links to 1e-17 relative (logistic: both
    responses, both sign conventions; linear), probit's log Phi and phi/Phi within the erfcx bound of ref_logtarget_grad"""
    import mpmath as mp
    mp.mp.dps = 40
    eta = np.array([0.0, 1e-300, -1e-17, 0.3, -0.3, 1.7, -2.5, 3.99, -4.01, 7.99, -8.01, 12.0, -12.0, 20.0, -30.0,
                    36.89, -36.95, 39.0, -40.0, 150.0, -300.0, 690.0, -705.0, 720.0])
    for fam, hys in (("linear", [(1.0, 0.7)]), ("logistic", [(1.0, -1.0), (1.0, 1.0)]), ("probit", [(10.0,)])):
        for hy in hys:
            for yv in ((0.0, 1.0, 0.25) if fam == "probit" else (0.0, 1.0, 2.5) if fam == "linear" else (0.0, 1.0)):
                ll, r, _ = _link(fam, eta.astype(np.longdouble), np.full(eta.shape, yv), hy)
                for i, e in enumerate(eta):
                    z = mp.mpf(float(e))
                    if fam == "linear":
                        res = mp.mpf(yv) - z
                        tl, tr = -(mp.log(mp.sqrt(2 * mp.pi)) + res ** 2 / (2 * mp.mpf(hy[1]) ** 2) + mp.log(hy[1])), res / mp.mpf(hy[1]) ** 2
                        tol_l, tol_r = 1e-17 * abs(tl), 1e-17 * abs(tr)
                    elif fam == "logistic":
                        x = hy[1] * z                                  # p = 1/(1 + exp(x)), 1 - p = 1/(1 + exp(-x))
                        tl = -mp.log1p(mp.exp(x)) if yv != 0 else -mp.log1p(mp.exp(-x))
                        tr = -hy[1] / (1 + mp.exp(-x)) if yv != 0 else hy[1] / (1 + mp.exp(x))
                        tol_l, tol_r = 1e-17 * abs(tl), 1e-17 * abs(tr)
                    else:
                        if abs(e) > 40 and yv not in (0.0, 1.0):
                            continue
                        lP, lM = mp.log(mp.ncdf(z)), mp.log(mp.ncdf(-z))
                        tl = yv * lP + (1 - yv) * lM
                        tr = yv * mp.npdf(z) / mp.ncdf(z) - (1 - yv) * mp.npdf(z) / mp.ncdf(-z)
                        # 1.2e-15 absolute (z < 0) or relative (z >= 0) on each log Phi, relative on each phi/Phi
                        tol_l = 1.3e-15 * (yv * max(1, abs(lP)) + (1 - yv) * max(1, abs(lM)))
                        tol_r = 1.3e-15 * (yv * abs(mp.npdf(z) / mp.ncdf(z)) + (1 - yv) * abs(mp.npdf(z) / mp.ncdf(-z)))
                    assert abs(_mpf(ll[i]) - tl) <= max(tol_l, 1e-300), (fam, hy, yv, e, float(ll[i]), tl)
                    assert abs(_mpf(r[i]) - tr) <= max(tol_r, 1e-300), (fam, hy, yv, e, float(r[i]), tr)


def test_sweep_covers_every_compiled_variant():
    """the DK labels of launch_f in k1_regress.cu are exactly the sweep's: a variant added later without a test fails here"""
    src = open(os.path.join(ROOT, "mcmc.jl_b200", "csrc", "k1_regress.cu")).read()
    body = src[src.index("static cudaError_t launch_f("):]
    body = body[:body.index("\n}\n")]
    compiled = {int(m) for m in re.findall(r"case\s+(\d+)\s*:", body)}
    assert compiled == set(COMPILED_DK)
    assert {_dk(d) for d in SWEEP_D} == compiled
    for k in COMPILED_DK:                                     # the smallest and the largest d of every block
        assert set(_d_range(k)) <= set(SWEEP_D)
    assert {PSH[_dk(d)] for d in SWEEP_D} == {0, 4, 8}


def test_sweep_problems_reach_the_link_ranges():
    """the sweep's data do what its tests rely on: probit |eta| crosses 4, 8 and 36.9 with some 32-row groups wholly
    inside |z| < 4; logistic reaches |eta| ~ 40 in support and one chain |x| >= 700"""
    for d in (1, 64, 200):
        eta = np.abs(sweep_reference("probit", d)["eta"].astype(np.float64))
        assert eta.max() > 36.9 and (eta > 8).any() and ((eta > 4) & (eta < 8)).any()
        n32 = eta.shape[0] // 32 * 32
        groups = eta[:n32, :8].reshape(-1, 32, 8).max(axis=(1, 2))           # first warp's 32-row groups
        assert (groups < 4).any()
        ref = sweep_reference("logistic", d)
        assert not ref["bad"].any()
        eta = ref["eta"].astype(np.float64)
        assert np.abs(np.delete(eta, 5, axis=1)).max() > 30 and np.abs(eta[:, 5]).max() >= 700


# ---- GPU: the variant sweep -------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("d", SWEEP_D)
@pytest.mark.parametrize("fam", FAMS)
def test_every_variant_against_the_reference(capi, ctx, fam, d):
    X, y, B = sweep_problem(fam, d)
    ref = sweep_reference(fam, d)
    dm = capi.DeviceModel(ctx, fam, d, X, y, HYPER[fam])
    try:
        lt, g = dm.logtarget_grad(B)
        lt_only, none = dm.logtarget_grad(B, grad=False)
        if d in (1, 64, 113):                                  # one chain: a 64-chain tile holding a single chain
            lt1, g1 = dm.logtarget_grad(B[7:8])
    finally:
        dm.close()
    assert none is None and np.allclose(lt, lt_only, rtol=1e-13, atol=0)
    _check_against_reference(ref, lt, g, label=(fam, d))
    if d in (1, 64, 113):
        sub = {k: (v[:, 7:8] if k in ("eta", "ll", "r", "dr") else v[7:8] if k in ("prior_terms", "lt", "g", "bad") else v)
               for k, v in ref.items()}
        _check_against_reference(sub, lt1, g1, label=(fam, d, "C=1"))


@pytest.mark.gpu
@pytest.mark.parametrize("d", (8, 56, 80, 104, 120, 200))
def test_probit_general_response_against_the_reference(capi, ctx, d):
    """a response that is neither 0 nor 1 sends the whole model down link<>'s log_ndtr path, in every CTA class"""
    X, y, B = sweep_problem("probit", d, 70)
    y = y.copy()
    y[::7] = 0.25
    B = B.copy()
    B[:, 1] = np.clip(B[:, 1], -5.0, 5.0)                   # |eta| <= ~6.5: exp(base - log Phi) stays well conditioned
    ref = _reference("probit", X, y, HYPER["probit"], B)
    dm = capi.DeviceModel(ctx, "probit", d, X, y, HYPER["probit"])
    try:
        lt, g = dm.logtarget_grad(B)
        lt_only, _ = dm.logtarget_grad(B, grad=False)
    finally:
        dm.close()
    assert np.allclose(lt, lt_only, rtol=1e-13, atol=0)
    _check_against_reference(ref, lt, g, general_probit=True, label=("probit-general", d))


# ---- GPU: bit-identity invariants -------------------------------------------------------------------------------------
def _central_probit(d, C, seed):
    """probit chains with |z| < 4 on every row: bounded X, sum_j |beta_j| = 3"""
    X, y, _ = sweep_problem("probit", d)
    rng = np.random.default_rng(seed)
    B = rng.uniform(-1.0, 1.0, (C, d))
    B *= 3.0 / np.abs(B).sum(1, keepdims=True)
    return X, y, B


@pytest.mark.gpu
@pytest.mark.parametrize("dk", COMPILED_DK)
def test_probit_table_copy_never_changes_a_number(capi, ctx, dk):
    """a warp reads the shared-memory copy of the link table only when all its elements of a 32-row group lie inside it.
    Replacing one warp-mate by beta = (5, 0, ...) (|z| = 5 everywhere: global table in |z| < 4 variants) or (10, 0, ...)
    (global table in |z| < 8 variants too) must leave every other chain's numbers bit for bit unchanged."""
    d = _d_range(dk)[1]
    C, c, mate = 24, 13, 10                                    # chain 13 and its warp-mates 8..15
    X, y, B = _central_probit(d, C, dk)
    assert np.abs(X @ B.T).max() < 4
    dm = capi.DeviceModel(ctx, "probit", d, X, y, HYPER["probit"])
    ctx.set_option("force_splits", 2)
    try:
        outs = []
        for out_b in (None, 5.0, 10.0):
            Bk = B.copy()
            if out_b is not None:
                Bk[mate] = 0.0
                Bk[mate, 0] = out_b
            outs.append(dm.logtarget_grad(Bk))
    finally:
        ctx.set_option("force_splits", 0)
        dm.close()
    keep = np.array([k for k in range(C) if k != mate])
    for lt, g in outs[1:]:
        assert np.array_equal(lt[keep], outs[0][0][keep]) and np.array_equal(g[keep], outs[0][1][keep]), (dk, PSH[dk])
    assert np.isfinite(outs[0][0][c])


def _tile_position_cases():
    cases = [("probit", _d_range(k)[1]) for k in COMPILED_DK]
    return cases + [(f, d) for f in ("linear", "logistic") for d in CTA_CLASS_D]


@pytest.mark.gpu
@pytest.mark.parametrize("fam,d", _tile_position_cases())
def test_chain_tile_position_never_changes_a_number(capi, ctx, fam, d):
    """one chain placed at chain index 0, 8, 64 (same DMMA fragment row, g = index mod 8), 63 and 129 (other fragment
    rows; 129 is in the last, partial chain tile of C = 130) gives the same bits at a pinned split count"""
    X, y, B = sweep_problem(fam, d)
    target = B[3 * 8 + 2].copy()                               # a chain of a wide-reach warp
    rng = np.random.default_rng(d)
    C = 130
    filler = B[0] + 0.01 * rng.standard_normal((C, d)) / math.sqrt(d)    # chains of the smallest reach
    dm = capi.DeviceModel(ctx, fam, d, X, y, HYPER[fam])
    ctx.set_option("force_splits", 3)
    try:
        res = {}
        for pos in (0, 8, 64, 63, 129):
            Bk = filler.copy()
            Bk[pos] = target
            lt, g = dm.logtarget_grad(Bk)
            res[pos] = (lt[pos], g[pos])
    finally:
        ctx.set_option("force_splits", 0)
        dm.close()
    for pos in (8, 64, 63, 129):
        assert res[pos][0] == res[0][0] and np.array_equal(res[pos][1], res[0][1]), (fam, d, pos)
    assert np.isfinite(res[0][0])


# ---- GPU: row splits and the split fold -------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("fam,d", [("linear", 17), ("logistic", 32), ("probit", 24), ("probit", 72), ("logistic", 100),
                                   ("linear", 104), ("probit", 113), ("logistic", 200)])
def test_row_splits_against_the_reference(capi, ctx, fam, d):
    """force_splits in {1, 2, 3, 5, ntiles, ntiles + 3}: beyond 4 splits the partial sums are folded by a separate kernel
    (launch_reduce_splits); beyond ntiles the last splits are empty.  N is not a multiple of 32, so the last non-empty
    split ends in a partial tile."""
    X, y, B = sweep_problem(fam, d)
    ref = sweep_reference(fam, d)
    ntiles = -(-X.shape[0] // 32)
    dm = capi.DeviceModel(ctx, fam, d, X, y, HYPER[fam])
    try:
        for splits in (1, 2, 3, 5, ntiles, ntiles + 3):
            ctx.set_option("force_splits", splits)
            try:
                lt, g = dm.logtarget_grad(B)
            finally:
                ctx.set_option("force_splits", 0)
            _check_against_reference(ref, lt, g, label=(fam, d, splits))
    finally:
        dm.close()
