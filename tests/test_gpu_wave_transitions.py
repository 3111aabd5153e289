"""The sampler transition kernels (csrc/transition.cu), the wave loop (execute_impl, csrc/engine.cu) and the fused chain
kernel (csrc/fused_chain.cu) at every dimension class, row-split path and loop option they choose between.

transition_coop_kernel (regression families) splits a chain's parameters into CO_GROUPS groups of Philox pairs and makes the
interior leapfrog CO_GROUPS * CO_UNROLL elements per pass; transition_kernel (closed-form families on the wave engine, and
storeLeaps) makes it TR_GROUPS * TR_UNROLL elements per pass; the likelihood's row splits reach the transition as preloaded
partial sums with the fused interior leapfrog (1 split), a serial sum (2..4) or a separate fold (> 4).  The dimensions below
put every one of those loops at its boundary (a second pass, a half pair, a one-element tail), and a CPU guard re-reads the
constants from the sources so that retuning one cannot leave a class untested.

Regression runs are draw-matched with the oracle (oracle/mcmc_oracle.c) at the criteria of test_regression_runs_draw_matched,
and every kept draw is checked against the extended-precision reference of test_gpu_k1_variants.py; closed-form runs go
through the same IEEE operations on both sides and are compared bit for bit.  The wave loop's options (graphs, timed
evaluations, poll interval, stepwise execution, the fused leapfrog, Philox vs injected draws) must not change a bit."""
import math
import os
import re
from concurrent.futures import ThreadPoolExecutor
from functools import lru_cache

import numpy as np
import pytest

from conftest import ROOT, make_regression
from test_gpu_k1_variants import _check_against_reference, _reference, _tolerances

CSRC = os.path.join(ROOT, "mcmc.jl_b200", "csrc")

FAMS = ("linear", "logistic", "probit")
COOP_D = (7, 16, 17, 25, 49, 200)         # odd d under 8 pairs; 8 pairs; a half pair in a second pass; a 1-element second
                                          # stage-A pass; several passes with tails; K1's maximum
SPLITS = (1, 3, 6)                        # fused interior leapfrog; serial sum_part; reduce_splits_kernel fold
SAMPLERS = ("RWM", "MALA", "MALA-tuned", "HMC", "HMC-tuned", "HMCDA")
PSD = (1.0, 0.5, 3.0)                     # prior sd: 1 and 0.5 take div_by_var's power-of-two path, 3 the division
CLOSED_FAMS = ("normal_fn", "normal_dsl", "abs_normal")
CLOSED_D = (9, 20, 21, 41)                # wave engine above FUSED_MAX_D; 21 and 41: a second (and third) stage-A pass
CLOSED_SAMPLERS = ("RWM", "MALA", "HMC", "HMC-tuned", "HMCDA")
FUSED_D = tuple(range(1, 9))
CLOSED_HYPER = {"normal_fn": (), "normal_dsl": (0.5, 2.0), "abs_normal": (0.5, 1.0)}
CLOSED_SD = {"normal_fn": math.sqrt(0.5), "normal_dsl": 2.0, "abs_normal": 1.0}


def _coop_cases():
    """18 cases: every sampler x split class, every d x split class and every family x sampler"""
    cases = []
    for i in range(18):
        b, s = divmod(i, 6)
        cases.append((FAMS[(b + s) % 3], COOP_D[(s + 2 * b) % 6], SAMPLERS[s], SPLITS[b], PSD[(i + b) % 3], (130, 70, 130, 1)[i % 4]))
    return cases


COOP_CASES = _coop_cases()


def _oracle(O, om, jobs):
    """oracle chains on a thread pool (ctypes releases the GIL): jobs = [(sampler, range, init, scale, normals, uniforms)]"""
    with ThreadPoolExecutor(max_workers=min(32, os.cpu_count() or 1)) as ex:
        return list(ex.map(lambda j: O.run_chain(om, *j), jobs))


@lru_cache(maxsize=None)
def _problem(fam, d, psd):
    """ragged regression problem (N never a multiple of 32, >= 6 row tiles) and the curvature its step sizes follow"""
    N = 32 * (6 + d // 16) + 13
    X, y, hy, b0 = make_regression(fam, N, d, 7 * d + FAMS.index(fam))
    hy = (psd,) + tuple(hy[1:])
    w = {"linear": 1.0, "logistic": 0.25, "probit": 0.64}[fam]          # Fisher weight of a row at eta ~ 0
    H = w * X.T @ X + np.eye(d) / psd ** 2
    return X, y, hy, b0, H


def _inits(b0, H, C, seed):
    """per-chain inits around the data's beta, spread by half the approximate posterior sd"""
    z = np.random.default_rng(seed).standard_normal((C, len(b0)))
    return b0[None, :] + 0.5 * np.linalg.solve(np.linalg.cholesky(H).T, z.T).T


def _spec(label, H, d):
    """(oracle/device sampler kind, keywords, range, model scale, HMCDA step size base) of a labelled sampler"""
    lmax = np.linalg.eigvalsh(H)[-1]
    eps = 1.6 * d ** -0.25 / math.sqrt(lmax)                              # leapfrog step inside the stability limit
    if label == "RWM":
        sc = 0.5 + 0.5 * (np.arange(d) % 3)                               # non-uniform model scale (RWM.jl:52)
        return "RWM", dict(scale=2.0 / math.sqrt(np.sum(np.diag(H) * sc * sc))), (31, 2, 70), sc, None
    if label.startswith("MALA"):
        h = (2.0 * d ** (-1 / 6) / math.sqrt(lmax)) ** 2
        kw = dict(scale=h, tuner=dict(target_rate=0.6, adapt_step=10)) if label == "MALA-tuned" else dict(scale=h)
        return "MALA", kw, (31, 2, 70), None, None
    if label == "HMC":
        return "HMC", dict(scale=eps, nleaps=4), (31, 2, 70), None, None
    if label == "HMC-tuned":
        return "HMC", dict(scale=eps, nleaps=3, tuner=dict(target_rate=0.8, adapt_step=10, target_path=4 * eps, max_step=8)), (31, 2, 70), None, None
    assert label == "HMCDA"
    return "HMCDA", dict(len=5 * eps, max_leaps=64), (1, 1, 40), None, eps


def _draws(C, last, d, seed):
    rng = np.random.default_rng(seed)
    return rng.standard_normal((C, last + 1, d)), rng.random((C, last + 1))


def _run_regression(O, capi, ctx, fam, d, psd, label, C, splits, chains, seed=1, store_rb=False):
    """GPU run at a forced split count and the oracle chains `chains`, with injected draws"""
    X, y, hy, b0, H = _problem(fam, d, psd)
    kind, skw, rngt, sc, eps = _spec(label, H, d)
    init = _inits(b0, H, C, seed)
    zn, un = _draws(C, rngt[2], d, seed + 1)
    da = None if eps is None else eps * np.random.default_rng(seed + 2).uniform(0.7, 1.3, C)
    dm = capi.DeviceModel(ctx, fam, d, X, y, hy)
    ctx.set_option("force_splits", splits)
    try:
        run = capi.DeviceRun(dm, capi.sampler_cfg(kind, **skw), rngt, C, init, scale=sc, normals=zn, uniforms=un, engine="wave", store_rb=store_rb)
    finally:
        ctx.set_option("force_splits", 0)
    try:
        if da is not None:
            run.set_state(0, da, da, np.zeros(C))
        info = run.execute()
        out = run.fetch()
        diag = run.fetch_diag() if run.has_diag else None
        rb = run.fetch_rb() if store_rb else None
    finally:
        run.close(); dm.close()
    S = out["samples"].shape[1]
    orb = {c: np.full((S, d), np.nan) for c in chains} if store_rb else {}
    jobs = [(O.sampler(kind, rb_out=orb.get(c), da_state=None if da is None else [da[c], da[c], 0.0], **skw), rngt, init[c], sc, zn[c], un[c])
            for c in chains]
    refs = dict(zip(chains, _oracle(O, O.Model(fam, d, X, y, hy), jobs)))
    return dict(out=out, diag=diag, rb=rb, orb=orb, refs=refs, info=info, X=X, y=y, hy=hy, kind=kind, tuned="tuner" in skw)


def _checked(C, d):
    """oracle chains: all of them, or every fifth at d >= 49 -- always with the last, in the last (partial) chain tile"""
    return sorted(set(range(0, C, 1 if d < 49 else 5)) | {C - 1})


def _assert_draw_matched(r, chains, label):
    out, diag, refs = r["out"], r["diag"], r["refs"]
    gs = np.abs(r["X"]).sum(0)
    for c in chains:
        ref = refs[c]
        assert ref["rc"] == 0, (*label, c)
        assert np.array_equal(ref["accept"], out["accept"][c]), (*label, c)
        assert np.allclose(ref["samples"], out["samples"][c], rtol=1e-9, atol=1e-12), (*label, c)
        assert np.allclose(ref["logtarget"], out["logtarget"][c], rtol=1e-11, atol=0), (*label, c)
        if r["kind"] == "RWM":
            assert np.all(np.isnan(out["grads"][c])), (*label, c)
        else:
            assert np.all(np.abs(ref["grads"] - out["grads"][c]) <= 1e-9 * gs), (*label, c)
        if r["kind"] == "HMCDA":
            assert np.array_equal(diag[0][c], ref["eps"]) and np.array_equal(diag[1][c], ref["nleaps"]), (*label, c)
        elif r["tuned"]:
            assert np.allclose(diag[0][c], ref["eps"], rtol=1e-12, atol=0), (*label, c)
            if r["kind"] == "HMC":
                assert np.array_equal(diag[1][c], ref["nleaps"]), (*label, c)


# ---- 1 + 2: the cooperative kernel against the oracle and every kept draw against the reference -------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("fam,d,label,splits,psd,C", COOP_CASES,
                         ids=[f"{f}-d{d}-{s}-split{k}-psd{p:g}-C{c}" for f, d, s, k, p, c in COOP_CASES])
def test_coop_kernel_draw_matched(O, capi, ctx, fam, d, label, splits, psd, C):
    chains = _checked(C, d)
    r = _run_regression(O, capi, ctx, fam, d, psd, label, C, splits, chains)
    _assert_draw_matched(r, chains, (fam, d, label, splits))
    if C > 1:
        assert 0.1 < r["out"]["accept"].mean() < 1.0             # a real mix of accepts and rejects
    # every kept triple (sample, stored log-target, stored gradient) of a chain subset against the extended-precision
    # reference, at K1's bounds: a stale gradient kept on a reject, a prior summed from the wrong group or a log-target
    # of the wrong pair would hide inside the oracle's 1e-9
    out = r["out"]
    for c in chains[:3] + chains[-1:]:
        ref = _reference(fam, r["X"], r["y"], r["hy"], out["samples"][c])
        if r["kind"] == "RWM":
            tol_lt, _ = _tolerances(ref)
            err = np.abs(out["logtarget"][c].astype(np.longdouble) - ref["lt"]).astype(np.float64)
            assert not ref["bad"].any() and np.all(err <= tol_lt), (fam, d, label, c, float(np.max(err / tol_lt)))
        else:
            _check_against_reference(ref, out["logtarget"][c], out["grads"][c], label=(fam, d, label, splits, "chain", c))


@pytest.mark.gpu
def test_forced_split_counts_take_effect(O, capi, ctx):
    """the same run at 1, 3 and 6 row splits: K1 sums the rows in another order, so the log-targets differ in the last bits
    somewhere, and everything agrees within the draw-matched criteria"""
    fam, d, C = "logistic", 49, 130
    runs = {k: _run_regression(O, capi, ctx, fam, d, 1.0, "HMC", C, k, [])["out"] for k in SPLITS}
    gs = np.abs(_problem(fam, d, 1.0)[0]).sum(0)
    for a, b in ((1, 3), (1, 6), (3, 6)):
        ra, rb = runs[a], runs[b]
        assert not np.array_equal(ra["logtarget"], rb["logtarget"]), (a, b)
        assert np.array_equal(ra["accept"], rb["accept"]), (a, b)
        assert np.allclose(ra["samples"], rb["samples"], rtol=1e-9, atol=1e-12), (a, b)
        assert np.allclose(ra["logtarget"], rb["logtarget"], rtol=1e-11, atol=0), (a, b)
        assert np.all(np.abs(ra["grads"] - rb["grads"]) <= 1e-9 * gs), (a, b)


# ---- 3: transition_kernel (closed-form families on the wave engine) and the fused kernel, bit for bit -------------------
def _closed_init(C, d, seed):
    """both signs, and exact zeros (abs_normal's gradient takes sign(0) = 0 there)"""
    init = np.random.default_rng(seed).uniform(-1.5, 1.5, (C, d))
    init[(np.arange(C)[:, None] + np.arange(d)[None, :]) % 4 == 0] = 0.0
    return init


def _closed_spec(label, fam, d):
    sd = CLOSED_SD[fam]
    eps = 0.9 * sd * d ** -0.25
    if label == "RWM":
        sc = 0.5 + 0.5 * (np.arange(d) % 3)
        return "RWM", dict(scale=2.0 * sd / math.sqrt(np.sum(sc * sc))), (21, 1, 120), sc
    if label == "MALA":
        return "MALA", dict(scale=(1.1 * sd * d ** (-1 / 6)) ** 2), (21, 1, 120), None
    if label == "HMC":
        return "HMC", dict(scale=eps, nleaps=5), (21, 1, 120), None
    if label == "HMC-tuned":
        return "HMC", dict(scale=eps, nleaps=3, tuner=dict(target_rate=0.8, adapt_step=10, target_path=5 * eps, max_step=10)), (41, 1, 120), None
    return "HMCDA", dict(len=5 * eps, max_leaps=64), None, None


def _assert_bit_exact(out, diag, refs, chains, label):
    for c in chains:
        r = refs[c]
        assert np.array_equal(r["accept"], out["accept"][c]), (*label, c)
        assert np.array_equal(r["samples"], out["samples"][c]), (*label, c)
        assert np.array_equal(r["grads"], out["grads"][c], equal_nan=True), (*label, c)
        assert np.array_equal(r["logtarget"], out["logtarget"][c]), (*label, c)
        if diag is not None:
            assert np.array_equal(diag[0][c], r["eps"]) and np.array_equal(diag[1][c], r["nleaps"]), (*label, c)


def _hmcda_teacher_forced(O, capi, dm, om, skw, C, d, init, seed):
    """HMCDA continued at step 100 from restored step sizes with a consistent dualH, 6 adapting burn-in steps, then 14 kept
    ones.  The dual averaging amplifies last-bit libm differences (exp / log / pow, CUDA vs glibc), so the oracle replays
    every trajectory with the GPU's step size (read back after every burn-in step) and reports its own adapted one."""
    s0, B, last = 100, 106, 120
    eps0 = skw["len"] / 5 * np.random.default_rng(seed).uniform(0.7, 1.3, C)
    dualH = (math.log(10.0) - np.log(eps0)) * 0.05 / math.sqrt(s0)
    zn, un = _draws(C, last, d, seed + 1)
    run = capi.DeviceRun(dm, capi.sampler_cfg("HMCDA", **skw), (B + 1, 1, last), C, init, normals=zn, uniforms=un, engine="wave")
    try:
        run.set_state(s0, eps0, eps0, dualH)
        fe = np.full((C, last + 1), np.nan)
        fe[:, s0 + 1] = eps0
        for i in range(s0 + 1, B + 1):                  # after step i the state holds the step size of step i + 1
            run.execute_steps(1)
            fe[:, i + 1] = run.get_state()["leapstep"]
        fe[:, B + 1:] = fe[:, B + 1][:, None]           # frozen phase: leapStep = dualLeapStep (HMCDA.jl:140)
        run.execute_steps(last - B)
        out = run.fetch(); geps, gnl = run.fetch_diag()
    finally:
        run.close()
    refs = _oracle(O, om, [(O.sampler("HMCDA", start_step=s0, da_state=[eps0[c], eps0[c], dualH[c]], force_eps=fe[c], **skw),
                            (B + 1, 1, last), init[c], None, zn[c], un[c]) for c in range(C)])
    assert np.array_equal(geps, fe[:, B + 1:])
    return out, geps, gnl, refs


@pytest.mark.gpu
@pytest.mark.parametrize("label", CLOSED_SAMPLERS)
@pytest.mark.parametrize("d", CLOSED_D)
@pytest.mark.parametrize("fam", CLOSED_FAMS)
def test_closed_form_wave_transition_bit_exact(O, capi, ctx, fam, d, label):
    C = 70
    hy = CLOSED_HYPER[fam]
    kind, skw, rngt, sc = _closed_spec(label, fam, d)
    init = _closed_init(C, d, d)
    dm = capi.DeviceModel(ctx, fam, d, hyper=hy)
    om = O.Model(fam, d, hyper=hy)
    try:
        if kind == "HMCDA":
            out, geps, gnl, refs = _hmcda_teacher_forced(O, capi, dm, om, skw, C, d, init, d + 7)
            for c in range(C):
                r = refs[c]
                assert np.array_equal(r["accept"], out["accept"][c]) and np.array_equal(r["nleaps"], gnl[c]), (fam, d, c)
                assert np.allclose(r["eps"], geps[c], rtol=1e-9, atol=0), (fam, d, c)
            _assert_bit_exact(out, None, refs, range(C), (fam, d, label))
            assert len(np.unique(gnl)) >= 3                      # chains of different trajectory lengths in every wave
        else:
            zn, un = _draws(C, rngt[2], d, d + 1)
            run = capi.DeviceRun(dm, capi.sampler_cfg(kind, **skw), rngt, C, init, scale=sc, normals=zn, uniforms=un, engine="wave")
            try:
                run.execute(); out = run.fetch(); diag = run.fetch_diag() if run.has_diag else None
            finally:
                run.close()
            refs = _oracle(O, om, [(O.sampler(kind, **skw), rngt, init[c], sc, zn[c], un[c]) for c in range(C)])
            _assert_bit_exact(out, diag, refs, range(C), (fam, d, label))
        assert 0.1 < out["accept"].mean() < 1.0
    finally:
        dm.close()


def _fused_cases():
    return [("abs_normal", d, s) for d in FUSED_D for s in CLOSED_SAMPLERS] + [(f, 5, s) for f in ("normal_fn", "normal_dsl") for s in CLOSED_SAMPLERS]


@pytest.mark.gpu
@pytest.mark.parametrize("fam,d,label", _fused_cases(), ids=[f"{f}-d{d}-{s}" for f, d, s in _fused_cases()])
def test_closed_form_fused_bit_exact(O, capi, ctx, fam, d, label):
    """every instantiated D of the fused kernel; HMCDA without burn-in keeps its initial step size 1 (HMCDA.jl:140)"""
    C = 70
    hy = CLOSED_HYPER[fam]
    kind, skw, rngt, sc = _closed_spec(label, fam, d)
    if kind == "HMCDA":
        skw, rngt = dict(len=3.0 * CLOSED_SD[fam], max_leaps=64), (1, 1, 120)
    init = _closed_init(C, d, d + 50)
    zn, un = _draws(C, rngt[2], d, d + 51)
    dm = capi.DeviceModel(ctx, fam, d, hyper=hy)
    try:
        run = capi.DeviceRun(dm, capi.sampler_cfg(kind, **skw), rngt, C, init, scale=sc, normals=zn, uniforms=un, engine="fused")
        run.execute(); out = run.fetch(); diag = run.fetch_diag() if run.has_diag else None
        run.close()
    finally:
        dm.close()
    om = O.Model(fam, d, hyper=hy)
    refs = _oracle(O, om, [(O.sampler(kind, **skw), rngt, init[c], sc, zn[c], un[c]) for c in range(C)])
    _assert_bit_exact(out, diag, refs, range(C), (fam, d, label))
    assert 0.1 < out["accept"].mean() <= 1.0


@pytest.mark.gpu
@pytest.mark.parametrize("kind,skw", [("HMC", dict(scale=0.5, nleaps=6)), ("RWM", dict(scale=0.4)), ("MALA", dict(scale=0.2))])
@pytest.mark.parametrize("fam,d", [("abs_normal", 5), ("normal_fn", 8)])
def test_streamed_summaries_at_streaming_d(capi, ctx, fam, d, kind, skw):
    """the streaming fused variant above D = 4 (no 7-CTA launch bound) against a draw-storing run of the same chains and its
    stats pass, at the criteria of test_streamed_summaries_match_the_two_pass_stats"""
    C, rngt = 300, (101, 2, 1900)
    dm = capi.DeviceModel(ctx, fam, d, hyper=CLOSED_HYPER[fam])
    cfg = capi.sampler_cfg(kind, **skw)
    full = capi.DeviceRun(dm, cfg, rngt, C, np.ones(d), seed=21, chain_offset=5, engine="fused"); full.execute()
    ref = full.stats("bm", batchlen=50)
    st = capi.DeviceRun(dm, cfg, rngt, C, np.ones(d), seed=21, chain_offset=5, engine="fused", stream_stats=True, stream_batchlen=50); st.execute()
    out = st.stats("bm", batchlen=50)
    iid = st.stats("iid")
    full.close(); st.close(); dm.close()
    assert np.array_equal(out["mean"], ref["mean"]) and np.array_equal(out["accept_rate"], ref["accept_rate"])
    for k in ("var_iid", "var", "ess", "actime"):
        assert np.allclose(out[k], ref[k], rtol=1e-10, atol=0), k
    assert np.allclose(iid["var"], ref["var_iid"], rtol=1e-10, atol=0)
    assert 5 < ref["accept_rate"].mean() < 100


# ---- 4: storeLeaps through the wave engine's serial path ----------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("splits", (1, 6))
@pytest.mark.parametrize("d", (10, 49))
@pytest.mark.parametrize("fam", FAMS)
def test_store_leaps_regression(O, capi, ctx, fam, d, splits):
    """HMC storeLeaps on a regression model: every leap needs the log-target (need_ll), the Rao-Blackwell sums against the
    oracle's rb_out (mean.jl:17-31) within the draw-matched criteria"""
    C = 70
    chains = _checked(C, d)
    r = _run_regression(O, capi, ctx, fam, d, 1.0, "HMC", C, splits, chains, seed=3, store_rb=True)
    _assert_draw_matched(r, chains, (fam, d, splits))
    for c in chains:
        assert np.allclose(r["rb"][c], r["orb"][c], rtol=1e-9, atol=1e-12), (fam, d, splits, c)
    assert 0.1 < r["out"]["accept"].mean() < 1.0


@pytest.mark.gpu
@pytest.mark.parametrize("fam,engine", [("normal_fn", "fused"), ("normal_fn", "wave"), ("logistic", "wave")])
def test_store_leaps_hmcda(O, capi, ctx, fam, engine):
    """HMCDA storeLeaps: normal_fn from its initial step size 1 (no burn-in), logistic from restored per-chain step sizes"""
    C = 70
    if fam == "normal_fn":
        d, skw, hy, X, y = (8 if engine == "fused" else 9), dict(len=3.0, max_leaps=64), (), None, None
        init, da, rngt = _closed_init(C, d, 4), None, (1, 1, 100)
    else:
        d = 10
        X, y, hy, b0, H = _problem(fam, d, 1.0)
        eps = 1.6 * d ** -0.25 / math.sqrt(np.linalg.eigvalsh(H)[-1])
        skw, init, rngt = dict(len=5 * eps, max_leaps=64), _inits(b0, H, C, 4), (1, 1, 60)
        da = eps * np.random.default_rng(5).uniform(0.7, 1.3, C)
    zn, un = _draws(C, rngt[2], d, 6)
    dm = capi.DeviceModel(ctx, fam, d, X, y, hy)
    try:
        run = capi.DeviceRun(dm, capi.sampler_cfg("HMCDA", **skw), rngt, C, init, normals=zn, uniforms=un, engine=engine, store_rb=True)
        if da is not None:
            run.set_state(0, da, da, np.zeros(C))
        run.execute(); out = run.fetch(); rb = run.fetch_rb(); geps, gnl = run.fetch_diag()
        run.close()
    finally:
        dm.close()
    S = out["samples"].shape[1]
    orb = [np.full((S, d), np.nan) for _ in range(C)]
    refs = _oracle(O, O.Model(fam, d, X, y, hy), [(O.sampler("HMCDA", rb_out=orb[c], da_state=None if da is None else [da[c], da[c], 0.0], **skw),
                                                   rngt, init[c], None, zn[c], un[c]) for c in range(C)])
    for c in range(C):
        assert np.array_equal(refs[c]["accept"], out["accept"][c]) and np.array_equal(refs[c]["nleaps"], gnl[c]), c
        if fam == "normal_fn":
            assert np.array_equal(refs[c]["samples"], out["samples"][c]), c
            assert np.allclose(rb[c], orb[c], rtol=1e-13, atol=1e-15), c        # test_store_leaps_rao_blackwell's criterion
        else:
            assert np.allclose(refs[c]["samples"], out["samples"][c], rtol=1e-9, atol=1e-12), c
            assert np.allclose(rb[c], orb[c], rtol=1e-9, atol=1e-12), c
    assert 0.1 < out["accept"].mean() < 1.0 and len(np.unique(gnl)) >= (1 if fam == "normal_fn" else 3)


def test_oracle_hmcda_rb_out_is_the_hmc_formula(O):
    """the oracle's HMCDA storeLeaps (CPU): at a frozen step size HMCDA makes HMC's trajectories, so its rb_out must equal the
    HMC branch's, and both must equal mean.jl:17-31 applied to the leap states recomputed here (normal_fn: lt = -x'x)"""
    d, S, eps, L = 3, 40, 0.3, 5
    om = O.Model("normal_fn", d)
    zn, un = _draws(1, S, d, 9)
    init = np.array([0.7, -0.2, 1.1])
    rb_da, rb_hmc = np.full((S, d), np.nan), np.full((S, d), np.nan)
    da = O.run_chain(om, O.sampler("HMCDA", len=L * eps, rb_out=rb_da, da_state=[eps, eps, 0.0]), (1, 1, S), init, None, zn[0], un[0])
    hm = O.run_chain(om, O.sampler("HMC", scale=eps, nleaps=L, rb_out=rb_hmc), (1, 1, S), init, None, zn[0], un[0])
    assert np.all(da["nleaps"] == L) and np.array_equal(da["samples"], hm["samples"]) and np.array_equal(rb_da, rb_hmc)
    assert 0 < da["accept"].mean() < 1
    x, want = init.copy(), np.empty((S, d))
    for i in range(1, S + 1):
        m = zn[0, i].copy()
        H0 = x @ x + 0.5 * (m @ m)
        p, states, Hs = x.copy(), [], []
        for _ in range(L):
            m = m + 0.5 * (-2 * p) * eps
            p = p + eps * m
            m = m + 0.5 * (-2 * p) * eps
            states.append(p.copy()); Hs.append(p @ p + 0.5 * (m @ m))
        if un[0, i] < min(1.0, math.exp(H0 - Hs[-1])):
            x = p
        want[i - 1] = (x + sum(math.exp(H0 - h) * s for h, s in zip(Hs, states))) / (L + 1)
    assert np.allclose(rb_da, want, rtol=1e-13, atol=1e-15)


# ---- 5: wave-loop options, bit for bit ----------------------------------------------------------------------------------
PATH_CASES = [(f, d, s) for f, d in (("logistic", 17), ("probit", 49)) for s in ("HMC", "HMC-tuned", "HMCDA", "MALA")] + [("normal_fn", 21, "HMC")]
SEED, OFFSET = (1 << 40) + 3, (1 << 33) + 5          # 64-bit Philox seed and chain ids


def _path_setup(fam, d, label, C):
    if fam in FAMS:
        X, y, hy, b0, H = _problem(fam, d, 1.0)
        kind, skw, rngt, sc, eps = _spec(label, H, d)
        init = _inits(b0, H, C, 8)
    else:
        X, y, hy = None, None, CLOSED_HYPER[fam]
        kind, skw, rngt, sc = _closed_spec(label, fam, d)
        eps, init = None, _closed_init(C, d, 8)
    rngt = (1, 1, 80) if kind == "HMCDA" else (rngt[0], 1, 80)
    da = None if eps is None else eps * np.random.default_rng(9).uniform(0.7, 1.3, C)
    return X, y, hy, kind, skw, rngt, sc, init, da


def _path_run(capi, ctx, dm, setup, C, options=(), segments=None, inject=None):
    X, y, hy, kind, skw, rngt, sc, init, da = setup
    saved = []
    try:
        for k, v in options:
            ctx.set_option(k, v)
            saved.append(k)
        zn, un = inject if inject is not None else (None, None)
        run = capi.DeviceRun(dm, capi.sampler_cfg(kind, **skw), rngt, C, init, scale=sc, seed=SEED, chain_offset=OFFSET,
                             normals=zn, uniforms=un, engine="wave")
        try:
            if da is not None:
                run.set_state(0, da, da, np.zeros(C))
            if segments is None:
                nev = run.execute()["n_grad_evals"]
            else:
                nev = 0
                for n in segments:
                    nev += run.execute_steps(n)["n_grad_evals"]
            out = run.fetch()
            diag = run.fetch_diag() if run.has_diag else None
        finally:
            run.close()
    finally:
        for k in saved:                                  # the context is session-wide: restore every option
            ctx.set_option(k, dict(use_graphs=1, time_eval=0, poll_every=0, fuse_leap=1, force_splits=0)[k])
    return out, diag, nev


def _assert_identical(a, b, label):
    (oa, da, na), (ob, db, nb) = a, b
    for k in ("samples", "accept", "grads", "logtarget"):
        assert np.array_equal(oa[k], ob[k], equal_nan=True), (*label, k)
    if da is not None:
        assert np.array_equal(da[0], db[0]) and np.array_equal(da[1], db[1]), (*label, "diag")
    assert na == nb, (*label, "n_grad_evals", na, nb)


@pytest.mark.gpu
@pytest.mark.parametrize("fam,d,label", PATH_CASES, ids=[f"{f}-d{d}-{s}" for f, d, s in PATH_CASES])
def test_wave_loop_options_change_no_bit(capi, ctx, fam, d, label):
    C = 130
    setup = _path_setup(fam, d, label, C)
    X, y, hy = setup[:3]
    last = setup[5][2]
    dm = capi.DeviceModel(ctx, fam, d, X, y, hy)
    try:
        base = _path_run(capi, ctx, dm, setup, C)
        variants = {"use_graphs=0": dict(options=[("use_graphs", 0)]), "time_eval=1": dict(options=[("time_eval", 1)]),
                    "poll_every=1": dict(options=[("poll_every", 1)]), "poll_every=3": dict(options=[("poll_every", 3)]),
                    "segments": dict(segments=(7, 1, 30, last - 38)),
                    "injected": dict(inject=ctx.philox_draws(SEED, OFFSET, C, d, last))}
        for name, kw in variants.items():
            _assert_identical(base, _path_run(capi, ctx, dm, setup, C, **kw), (fam, d, label, name))
    finally:
        dm.close()
    assert 0.1 < base[0]["accept"].mean() < 1.0


@pytest.mark.gpu
@pytest.mark.parametrize("label", ("HMC-tuned", "HMCDA"))
@pytest.mark.parametrize("d", (17, 49, 200))
def test_fused_leapfrog_changes_no_bit(capi, ctx, d, label):
    """one row split: the likelihood kernel makes the interior leapfrogs (fuse_leap 1) or the cooperative transition kernel
    does (fuse_leap 0) -- chains of different trajectory lengths in every wave"""
    C, fam = 130, "logistic"
    setup = _path_setup(fam, d, label, C)
    dm = capi.DeviceModel(ctx, fam, d, *setup[:3])
    try:
        a = _path_run(capi, ctx, dm, setup, C, options=[("force_splits", 1)])
        b = _path_run(capi, ctx, dm, setup, C, options=[("force_splits", 1), ("fuse_leap", 0)])
    finally:
        dm.close()
    _assert_identical(a, b, (fam, d, label))
    assert 0.1 < a[0]["accept"].mean() < 1.0


@pytest.mark.gpu
@pytest.mark.parametrize("label", ("HMC", "MALA"))
def test_philox_mode_coop_run_replayed_through_oracle(O, capi, ctx, label):
    """the engine's own Philox draws at odd d > 16 (9 pairs: pair 8 in a second pass of the pair loop), dumped and replayed
    through the oracle at the draw-matched criteria"""
    fam, d, C = "logistic", 17, 70
    setup = _path_setup(fam, d, label, C)
    X, y, hy, kind, skw, rngt, sc, init, da = setup
    dm = capi.DeviceModel(ctx, fam, d, X, y, hy)
    try:
        out, _, _ = _path_run(capi, ctx, dm, setup, C)
    finally:
        dm.close()
    zn, un = ctx.philox_draws(SEED, OFFSET, C, d, rngt[2])
    refs = _oracle(O, O.Model(fam, d, X, y, hy), [(O.sampler(kind, **skw), rngt, init[c], sc, zn[c], un[c]) for c in range(C)])
    r = dict(out=out, diag=None, refs=dict(enumerate(refs)), X=X, kind=kind, tuned=False)
    _assert_draw_matched(r, range(C), (fam, d, label, "philox"))


# ---- 6: the case lists cover the kernels' boundaries (CPU) --------------------------------------------------------------
def _constants(path, names):
    src = open(os.path.join(CSRC, path)).read()
    return {n: int(re.search(r"\b%s\s*=\s*(\d+)" % n, src).group(1)) for n in names}


def test_case_lists_cover_the_kernel_boundaries():
    k = _constants("transition.cu", ("CO_GROUPS", "CO_UNROLL", "TR_GROUPS", "TR_UNROLL"))
    fused_max = _constants("fused_chain.h", ("FUSED_MAX_D",))["FUSED_MAX_D"]
    ladder = [int(m) for m in re.findall(r"if \(d <= (\d+)\) return launch_one<FAM, \1>", open(os.path.join(CSRC, "fused_chain.cu")).read())]
    coop_d = {c[1] for c in COOP_CASES}
    # the pair loop's second pass (and a half pair in it), the interior leapfrog's second pass with one element
    for b in (2 * k["CO_GROUPS"], 2 * k["CO_GROUPS"] + 1, k["CO_GROUPS"] * k["CO_UNROLL"] + 1):
        assert b in coop_d, b
    assert any(d > 2 * k["CO_GROUPS"] * k["CO_UNROLL"] for d in coop_d) and max(coop_d) == 200
    assert {c[1] for c in PATH_CASES if c[0] in FAMS} >= {2 * k["CO_GROUPS"] + 1}
    # transition_kernel's stage A: a second pass, above the fused engine's range (the automatic engine's choice there)
    assert k["TR_GROUPS"] * k["TR_UNROLL"] + 1 in CLOSED_D and min(CLOSED_D) > fused_max
    assert any(c[0] not in FAMS and c[1] == k["TR_GROUPS"] * k["TR_UNROLL"] + 1 for c in PATH_CASES)
    # every instantiated D of the fused kernel
    assert ladder == list(range(1, fused_max + 1)) and set(FUSED_D) == set(ladder)
    assert {c[1] for c in _fused_cases() if c[0] == "abs_normal"} == set(ladder)
    # the part-1 case list: every sampler x split class, d x split class and family x sampler
    assert {(c[2], c[3]) for c in COOP_CASES} == {(s, k_) for s in SAMPLERS for k_ in SPLITS}
    assert {(c[1], c[3]) for c in COOP_CASES} == {(d, k_) for d in COOP_D for k_ in SPLITS}
    assert {(c[0], c[2]) for c in COOP_CASES} == {(f, s) for f in FAMS for s in SAMPLERS}
    assert {c[4] for c in COOP_CASES} == set(PSD) and {c[5] for c in COOP_CASES} == {1, 70, 130}
    assert 4 < max(SPLITS) and 1 in SPLITS and any(1 < s <= 4 for s in SPLITS)     # engine.cu: nsplit > 4 takes the fold
