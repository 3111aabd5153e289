"""GPU suite: the CUDA path (through the C ABI) against the CPU oracle on the same seeded inputs, against the
committed golden fixtures, and -- at the full BASELINE sizes -- through size-independent properties.

Tolerances (north_star): log-target / gradient within 1e-12 relative (gradients relative to |X|'|r|, the
size of the summed terms); identical accept/reject decisions with injected draws.  Closed-form targets go
through identical IEEE operations on both sides and are compared bit for bit."""
import math

import numpy as np
import pytest

from conftest import load_golden, make_regression, ou_series

pytestmark = pytest.mark.gpu
TOL = 1e-12


def _lt_grad_check(O, capi, ctx, fam, N, d, C, seed, spread=0.3):
    X, y, hy, b0 = make_regression(fam, N, d, seed)
    om = O.Model(fam, d, X, y, hy)
    dm = capi.DeviceModel(ctx, fam, d, X, y, hy)
    rng = np.random.default_rng(seed + 100)
    B = b0 + spread * rng.standard_normal((C, d)) / math.sqrt(d)
    lt, g = dm.logtarget_grad(B)
    lt_only, none = dm.logtarget_grad(B, grad=False)
    # value-only waves read log Phi from the F table, value+gradient waves from the joint table: same function, last-bit differences
    assert none is None and np.allclose(lt, lt_only, rtol=1e-13, atol=0)
    gs = np.abs(X).sum(0)
    for c in range(C):
        olt, og = om.evalallg(B[c])
        assert abs(lt[c] - olt) <= TOL * abs(olt), (fam, N, d, c)
        assert np.all(np.abs(g[c] - og) <= TOL * gs), (fam, N, d, c)
    dm.close()


@pytest.mark.parametrize("fam", ["linear", "logistic", "probit"])
@pytest.mark.parametrize("N,d,C", [(1000, 10, 70), (39, 3, 1), (31, 1, 5), (33, 8, 64), (4097, 100, 130), (257, 104, 65), (2048, 20, 129),
                                   (300, 105, 66), (350, 113, 65), (513, 150, 64), (777, 200, 70)])
def test_regression_logtarget_gradient(O, capi, ctx, fam, N, d, C):
    # ragged everything: N not a multiple of the 32-row tile, C not a multiple of the 64-chain tile, d = 1 and d = 104
    _lt_grad_check(O, capi, ctx, fam, N, d, C, seed=N + d)


@pytest.mark.parametrize("name", ["normal_fn", "normal_dsl", "linear", "logistic", "logistic_plus", "probit", "ou", "probit_vaso"])
def test_models_against_mpmath_golden(capi, ctx, name):
    g = load_golden("golden_models.npz")[name]
    d = g["B"].shape[1]
    dm = capi.DeviceModel(ctx, g["family"], d, g["X"], g["y"], g["hyper"])
    lt, gr = dm.logtarget_grad(g["B"])
    for c in range(len(g["B"])):
        if np.isinf(g["lt"][c]):
            assert lt[c] == g["lt"][c] and np.all(gr[c] == 0)
            continue
        assert abs(lt[c] - g["lt"][c]) <= 1e-12 * max(1.0, abs(g["lt"][c]))
        scale = 1.0 if g["X"] is None else np.abs(g["X"]).sum(0)
        assert np.all(np.abs(gr[c] - g["grad"][c]) <= 1e-11 * np.maximum(scale, np.abs(g["grad"][c])))
    dm.close()


def test_out_of_support_semantics(O, capi, ctx):
    X, y, hy, _ = make_regression("logistic", 50, 3, 1)
    dm = capi.DeviceModel(ctx, "logistic", 3, X, y, hy)
    B = np.array([[0.0, 800.0, 0.0], [np.nan, 0.0, 0.0], [0.1, 0.2, 0.3]])
    lt, g = dm.logtarget_grad(B)
    assert lt[0] == -np.inf and np.all(g[0] == 0) and lt[1] == -np.inf and np.all(g[1] == 0) and np.isfinite(lt[2])
    dm.close()
    x = ou_series(50, 1)
    dm = capi.DeviceModel(ctx, "ou", 3, None, x, (100.0, 2.0, 20.0))
    lt, g = dm.logtarget_grad(np.array([[-1.0, 1, 1], [5, 2.5, 1], [5, 1, 21], [20, 0.1, 10]]))
    assert np.all(lt[:3] == -np.inf) and np.all(g[:3] == 0) and np.isfinite(lt[3])
    dm.close()
    # linear: the four-instruction link carries sum z^2 and a row count; a non-finite residual anywhere must still give (-Inf, zeros)
    Xl, yl, hyl, _ = make_regression("linear", 70, 3, 4)             # 70 rows: a ragged last tile
    om, dm = O.Model("linear", 3, Xl, yl, hyl), capi.DeviceModel(ctx, "linear", 3, Xl, yl, hyl)
    Bl = np.array([[np.nan, 0.0, 0.0], [1e200, 0.0, 0.0], [0.0, np.inf, 0.0], [0.3, -0.2, 0.1]])
    lt, g = dm.logtarget_grad(Bl)
    assert np.all(lt[:3] == -np.inf) and np.all(g[:3] == 0) and np.isfinite(lt[3]) and np.all(np.isfinite(g[3]))
    for c in range(4):
        olt, og = om.evalallg(Bl[c])
        assert (olt == lt[c] or abs(olt - lt[c]) <= 1e-12 * abs(olt)) and np.allclose(og, g[c], rtol=1e-12, atol=0), c
    dm.close()
    Xp, yp, hyp, _ = make_regression("probit", 30, 2, 2)
    dm = capi.DeviceModel(ctx, "probit", 2, Xp, yp, hyp)
    lt, _ = dm.logtarget_grad(np.array([[1e200, 1e200]]))
    assert np.isnan(lt[0])                                     # 0 * -Inf, probit_regression.jl:29
    dm.close()


def _run_both(O, capi, ctx, fam, d, X, y, hy, kind, skw, rngt, C, init, engine, scale=None, seed=1, force_eps=False, chains=None):
    """GPU run of C chains and oracle chains (all, or those listed in `chains`; None in refs for the others)"""
    om = O.Model(fam, d, X, y, hy)
    dm = capi.DeviceModel(ctx, fam, d, X, y, hy)
    rng = np.random.default_rng(seed)
    last = rngt[2]
    zn = rng.standard_normal((C, last + 1, d)); un = rng.random((C, last + 1))
    run = capi.DeviceRun(dm, capi.sampler_cfg(kind, **skw), rngt, C, init, scale=scale, normals=zn, uniforms=un, engine=engine)
    info = run.execute()
    out = run.fetch()
    diag = run.fetch_diag() if run.has_diag else None
    refs = [None] * C
    for c in (range(C) if chains is None else chains):
        kw = dict(skw)
        if force_eps:
            kw["force_eps"] = np.concatenate([[np.nan], diag[0][c]])       # needs rngt = (1, 1, last)
        ini = init[c] if np.ndim(init) == 2 else init
        refs[c] = O.run_chain(om, O.sampler(kind, **kw), rngt, ini, scale, zn[c], un[c])
    run.close(); dm.close()
    return out, diag, refs, info


CLOSED = [("normal_fn", 3, (), "RWM", dict(scale=0.1), (101, 1, 600)),
          ("normal_fn", 3, (), "HMC", dict(scale=0.75, nleaps=10), (51, 2, 400)),
          ("normal_dsl", 4, (0.0, 1.0), "MALA", dict(scale=0.5), (1, 1, 300)),
          ("normal_dsl", 7, (0.5, 2.0), "HMC", dict(scale=0.4, nleaps=3), (1, 3, 200)),
          ("normal_fn", 2, (), "HMC", dict(scale=0.3, nleaps=5, tuner=dict(target_rate=0.7, adapt_step=50)), (201, 1, 400)),
          ("normal_dsl", 2, (0.0, 1.0), "MALA", dict(scale=0.3, tuner=dict(target_rate=0.5, adapt_step=50)), (201, 1, 400)),
          ("normal_fn", 1, (), "RWM", dict(scale=0.5), (1, 1, 100)),
          ("normal_fn", 8, (), "MALA", dict(scale=0.2), (1, 1, 100))]


@pytest.mark.parametrize("engine", ["fused", "wave"])
@pytest.mark.parametrize("case", CLOSED, ids=lambda c: f"{c[0]}-d{c[1]}-{c[3]}")
def test_closed_form_runs_bit_exact(O, capi, ctx, engine, case):
    fam, d, hy, kind, skw, rngt = case
    C = 70
    out, diag, refs, _ = _run_both(O, capi, ctx, fam, d, None, None, hy, kind, skw, rngt, C, np.ones(d), engine)
    for c in range(C):
        assert np.array_equal(refs[c]["accept"], out["accept"][c])
        assert np.array_equal(refs[c]["samples"], out["samples"][c])
        assert np.array_equal(refs[c]["grads"], out["grads"][c], equal_nan=True)
        assert np.array_equal(refs[c]["logtarget"], out["logtarget"][c])
        if diag is not None:
            assert np.array_equal(diag[0][c], refs[c]["eps"]) and np.array_equal(diag[1][c], refs[c]["nleaps"])


@pytest.mark.parametrize("engine", ["fused", "wave"])
def test_ou_runs(O, capi, ctx, engine):
    x = ou_series(300, 4)
    init = np.array([20.0, 0.1, 10.0])
    for kind, skw, scale in [("RWM", dict(scale=0.01), np.array([1000.0, 1.0, 10.0])), ("HMC", dict(scale=0.002, nleaps=5), None),
                             ("MALA", dict(scale=1e-5), None)]:
        out, _, refs, _ = _run_both(O, capi, ctx, "ou", 3, None, x, (100.0, 2.0, 20.0), kind, skw, (1, 1, 150), 20, init, engine, scale=scale)
        for c in range(20):
            assert np.array_equal(refs[c]["accept"], out["accept"][c])
            assert np.allclose(refs[c]["samples"], out["samples"][c], rtol=1e-10, atol=0)


@pytest.mark.parametrize("fam", ["linear", "logistic", "probit"])
@pytest.mark.parametrize("kind,skw,rngt", [("RWM", dict(scale=0.02), (1, 1, 150)), ("MALA", dict(scale=0.001), (1, 1, 150)),
                                           ("HMC", dict(scale=0.02, nleaps=4), (51, 1, 150)),
                                           ("HMC", dict(scale=0.02, nleaps=3, tuner=dict(target_rate=0.8, adapt_step=20)), (61, 2, 140))])
def test_regression_runs_draw_matched(O, capi, ctx, fam, kind, skw, rngt):
    N, d, C = 1000, 10, 70
    X, y, hy, _ = make_regression(fam, N, d, 2)
    out, diag, refs, _ = _run_both(O, capi, ctx, fam, d, X, y, hy, kind, skw, rngt, C, np.zeros(d), "wave")
    gs = np.abs(X).sum(0)
    for c in range(C):
        assert np.array_equal(refs[c]["accept"], out["accept"][c]), (fam, kind, c)
        assert np.allclose(refs[c]["samples"], out["samples"][c], rtol=1e-9, atol=1e-12)
        assert np.allclose(refs[c]["logtarget"], out["logtarget"][c], rtol=1e-11, atol=0)
        if kind != "RWM":
            assert np.all(np.abs(refs[c]["grads"] - out["grads"][c]) <= 1e-9 * gs)
        else:
            assert np.all(np.isnan(out["grads"][c]))


@pytest.mark.parametrize("engine,fam", [("fused", "normal_fn"), ("wave", "normal_fn"), ("wave", "logistic")])
def test_hmcda_teacher_forced(O, capi, ctx, engine, fam):
    """HMCDA's dual averaging is a chaotic map once eps crosses the leapfrog stability limit (it starts at 1 and
    jumps to ~19), so last-bit libm differences (exp/log/pow, CUDA vs glibc) grow without bound over a burn-in.
    The check is therefore one step ahead: the oracle replays every trajectory with the GPU's step size and must
    reproduce (i) the accept decision, (ii) the state, (iii) the NEXT adapted step size and leap count."""
    if fam == "normal_fn":
        d, X, y, hy, init, skw, C = 3, None, None, (), np.ones(3), dict(len=2.0), 40
    else:
        d = 10
        X, y, hy, _ = make_regression(fam, 1000, d, 2)
        init, skw, C = np.zeros(d), dict(len=0.2, max_leaps=256), 24
    rngt = (1, 1, 120)
    # burn-in must cover the run for adaptation to be active: kept range starts after burn-in, so run with
    # first = 1 on both sides but tell the sampler about a long burn-in through a second, shifted pass below
    out, diag, refs, _ = _run_both(O, capi, ctx, fam, d, X, y, hy, "HMCDA", skw, rngt, C, init, engine, force_eps=True)
    for c in range(C):
        assert np.all(diag[0][c] == 1.0)        # burnin = 0: frozen initial dual step (HMCDA.jl:140)
        assert np.array_equal(refs[c]["accept"], out["accept"][c])
    # adaptation active: burnin = 60, everything after is kept; the teacher-forced oracle needs eps for all steps,
    # which the diagnostics only hold for kept steps -> compare kept-step eps / nleaps / decisions statistically
    # close and exactly over the first kept step (its eps is the adapted dual step, a pure function of the burn-in)
    rng = np.random.default_rng(3)
    last = 90
    zn = rng.standard_normal((C, last + 1, d)); un = rng.random((C, last + 1))
    dm = capi.DeviceModel(ctx, fam, d, X, y, hy)
    om = O.Model(fam, d, X, y, hy)
    # short burn-ins stay below the chaotic horizon: exact agreement of the adapted step after b steps
    for b in (2, 3, 5):
        run = capi.DeviceRun(dm, capi.sampler_cfg("HMCDA", **skw), (b + 1, 1, b + 6), C, init, normals=zn[:, :b + 7], uniforms=un[:, :b + 7], engine=engine)
        run.execute(); eps, nl = run.fetch_diag(); o = run.fetch()
        for c in range(C):
            ref = O.run_chain(om, O.sampler("HMCDA", **skw), (b + 1, 1, b + 6), init, None, zn[c, :b + 7], un[c, :b + 7])
            assert np.allclose(eps[c], ref["eps"], rtol=1e-9), (b, c)
            assert np.array_equal(nl[c], ref["nleaps"]) and np.array_equal(o["accept"][c], ref["accept"])
        run.close()
    dm.close()


def test_golden_chains(capi, ctx):
    for name, g in load_golden("golden_chains.npz").items():
        r = np.random.default_rng(g["draw_seed"])
        last = g["range"][2]
        z = r.standard_normal((last + 1, 3)); u = r.random(last + 1)
        dm = capi.DeviceModel(ctx, "normal_fn", 3)
        for engine in ("fused", "wave"):
            run = capi.DeviceRun(dm, capi.sampler_cfg(g["kind"], **g["kw"]), g["range"], 1, np.ones(3), normals=z[None], uniforms=u[None], engine=engine)
            run.execute(); out = run.fetch()
            assert np.array_equal(out["accept"][0], g["accept"]), (name, engine)
            assert np.array_equal(out["samples"][0], g["samples"]), (name, engine)
            assert np.array_equal(out["logtarget"][0], g["logtarget"]), (name, engine)
            run.close()
        dm.close()


def test_philox_streams(O, capi, ctx):
    z, u = ctx.philox_draws(12345, 7, 5, 5, 9)
    for c in range(5):
        for i in range(10):
            assert u[c, i] == O.draw_uniform(12345, 7 + c, i)                      # integer path + exact conversion
            assert np.allclose(z[c, i], O.draw_normals(12345, 7 + c, i, 5), rtol=0, atol=4e-15)
    z2, u2 = ctx.philox_draws((1 << 40) + 3, (1 << 33), 2, 4, 3)                   # 64-bit seed and chain ids
    assert u2[1, 2] == O.draw_uniform((1 << 40) + 3, (1 << 33) + 1, 2)
    zz, _ = ctx.philox_draws(9, 0, 4096, 2, 24)
    assert abs(zz.mean()) < 0.01 and abs(zz.var() - 1) < 0.01


@pytest.mark.parametrize("engine", ["fused", "wave"])
def test_philox_mode_replayed_through_oracle(O, capi, ctx, engine):
    """non-injected mode: the engine's own Philox draws, dumped and replayed through the oracle"""
    d, C, rngt, seed, off = 3, 50, (11, 1, 200), 77, 1000
    dm = capi.DeviceModel(ctx, "normal_fn", d)
    run = capi.DeviceRun(dm, capi.sampler_cfg("HMC", scale=0.75, nleaps=10), rngt, C, np.ones(d), seed=seed, chain_offset=off, engine=engine)
    run.execute(); out = run.fetch()
    zn, un = ctx.philox_draws(seed, off, C, d, rngt[2])
    om = O.Model("normal_fn", d)
    for c in range(C):
        ref = O.run_chain(om, O.sampler("HMC", scale=0.75, nleaps=10), rngt, np.ones(d), None, zn[c], un[c])
        assert np.array_equal(ref["accept"], out["accept"][c]) and np.array_equal(ref["samples"], out["samples"][c])
    run.close(); dm.close()


def test_chain_sharding_is_invariant(capi, ctx):
    """chains keyed by GLOBAL id: running [0, C) at once or as two shards gives identical draws (SURVEY 8e.1)"""
    d, C, rngt = 3, 256, (1, 1, 60)
    dm = capi.DeviceModel(ctx, "normal_fn", d)
    cfg = capi.sampler_cfg("HMC", scale=0.75, nleaps=10)
    full = capi.DeviceRun(dm, cfg, rngt, C, np.ones(d), seed=5); full.execute(); a = full.fetch()
    lo = capi.DeviceRun(dm, cfg, rngt, 100, np.ones(d), seed=5, chain_offset=0); lo.execute(); b = lo.fetch()
    hi = capi.DeviceRun(dm, cfg, rngt, 156, np.ones(d), seed=5, chain_offset=100, engine="wave"); hi.execute(); c = hi.fetch()
    assert np.array_equal(a["samples"][:100], b["samples"]) and np.array_equal(a["samples"][100:], c["samples"])
    assert np.array_equal(a["accept"][100:], c["accept"])
    for r in (full, lo, hi):
        r.close()
    dm.close()


def test_stepwise_execution_and_resume(O, capi, ctx):
    X, y, hy, _ = make_regression("logistic", 500, 6, 3)
    dm = capi.DeviceModel(ctx, "logistic", 6, X, y, hy)
    cfg = capi.sampler_cfg("HMCDA", len=0.3, max_leaps=64)
    C, rngt = 40, (11, 1, 60)
    one = capi.DeviceRun(dm, cfg, rngt, C, np.zeros(6), seed=9, engine="wave"); one.execute(); a = one.fetch()
    seg = capi.DeviceRun(dm, cfg, rngt, C, np.zeros(6), seed=9, engine="wave")
    for n in (7, 1, 30, 100):
        seg.execute_steps(n)
    b = seg.fetch()
    assert np.array_equal(a["samples"], b["samples"]) and np.array_equal(a["accept"], b["accept"])
    # true resume: stop at step 30, save, continue in a fresh run from the saved state
    first = capi.DeviceRun(dm, cfg, (11, 1, 30), C, np.zeros(6), seed=9, engine="wave"); first.execute()
    st = first.get_state()
    cont = capi.DeviceRun(dm, capi.sampler_cfg("HMCDA", len=0.3, max_leaps=64), (31, 1, 60), C, st["pars"], seed=9, engine="wave")
    cont.set_state(30, st["leapstep"], st["dual_leapstep"], st["dualH"])
    cont.execute(); c2 = cont.fetch()
    assert np.allclose(a["samples"][:, 20:], c2["samples"], rtol=1e-9, atol=1e-12)
    assert np.array_equal(a["accept"][:, 20:], c2["accept"])
    for r in (one, seg, first, cont):
        r.close()
    dm.close()


@pytest.mark.parametrize("vtype", ["iid", "bm", "imse", "ipse"])
def test_stats_parity(O, capi, ctx, vtype):
    rng = np.random.default_rng(8)
    C, S, d = 70, 500, 3
    x = np.empty((C, S, d))
    rho = rng.uniform(-0.7, 0.95, size=(C, d))
    x[:, 0] = rng.standard_normal((C, d))
    for t in range(1, S):
        x[:, t] = rho * x[:, t - 1] + rng.standard_normal((C, d))
    for kw in (dict(), dict(maxlag=25), dict(batchlen=20)):
        st = ctx.stats(x, vtype, kw.get("maxlag", -1), kw.get("batchlen", 100))
        for c in range(0, C, 7):
            for j in range(d):
                s = x[c, :, j]
                assert st["mean"][c, j] == O.mean(s)
                assert st["var_iid"][c, j] == O.mcvar(s, "iid")
                okw = {k: v for k, v in kw.items() if (k == "maxlag" and vtype in ("imse", "ipse")) or (k == "batchlen" and vtype == "bm")}
                ref = O.mcvar(s, vtype, **okw)
                assert abs(st["var"][c, j] - ref) <= 1e-13 * abs(ref)
                if vtype != "iid":
                    assert abs(st["ess"][c, j] - O.ess(s, vtype, **okw)) <= 1e-12 * abs(O.ess(s, vtype, **okw))
                    assert abs(st["actime"][c, j] - O.actime(s, vtype, **okw)) <= 1e-12 * O.actime(s, vtype, **okw)


def test_stats_golden(capi, ctx):
    for name, g in load_golden("golden_stats.npz").items():
        x = g["x"][None, :, None]
        assert abs(ctx.stats(x, "iid")["var"][0, 0] - g["iid"]) <= 1e-11 * g["iid"]
        assert abs(ctx.stats(x, "bm", batchlen=g["bm_len"])["var"][0, 0] - g["bm"]) <= 1e-11 * g["bm"]
        assert abs(ctx.stats(x, "imse")["var"][0, 0] - g["imse"]) <= 1e-11 * g["imse"]
        assert abs(ctx.stats(x, "ipse")["var"][0, 0] - g["ipse"]) <= 1e-11 * g["ipse"]
        assert abs(ctx.stats(x, "imse", maxlag=21)["var"][0, 0] - g["imse_lag21"]) <= 1e-11 * g["imse_lag21"]


def test_error_paths(capi, ctx):
    dm = capi.DeviceModel(ctx, "ou", 3, None, ou_series(30, 1), (100.0, 2.0, 20.0))
    run = capi.DeviceRun(dm, capi.sampler_cfg("RWM", scale=0.1), (1, 1, 10), 4, np.array([-1.0, 1.0, 1.0]))
    with pytest.raises(capi.MCMCGPUError) as e:
        run.execute()
    assert e.value.code == capi.E_SUPPORT and "Initial values out of model support" in str(e.value)   # RWM.jl:55
    run.close()
    for bad_rng in [(0, 1, 10), (11, 1, 10), (1, 0, 10)]:                                              # SerialMC.jl:25-27
        with pytest.raises(capi.MCMCGPUError) as e:
            capi.DeviceRun(dm, capi.sampler_cfg("RWM", scale=0.1), bad_rng, 4, np.array([20.0, 0.1, 10.0]))
        assert e.value.code == capi.E_ARG
    for bad in [capi.sampler_cfg("RWM", scale=-1.0), capi.sampler_cfg("HMC", scale=0.1, nleaps=0), capi.sampler_cfg("HMCDA", rate=1.5)]:
        with pytest.raises(capi.MCMCGPUError):
            capi.DeviceRun(dm, bad, (1, 1, 10), 4, np.array([20.0, 0.1, 10.0]))
    dm.close()
    with pytest.raises(capi.MCMCGPUError):
        capi.DeviceModel(ctx, "logistic", 201, np.zeros((10, 201)), np.zeros(10), (1.0, -1.0))        # d > 200 in this build
    with pytest.raises(capi.MCMCGPUError):
        ctx.stats(np.zeros((2, 50, 1)), "bm", batchlen=40)                                             # var.jl:22


def test_host_api_end_to_end(O):
    """the reference's README session through the Python mirror (test/test_syntax.jl:40-82)"""
    import mcmc_jl_b200 as mj
    m1 = mj.model("normal", init=np.ones(3), gradient=False)
    m2 = mj.model("normal", init=np.ones(3))
    chain = mj.run(m1, mj.RWM(0.1), mj.SerialMC(steps=1000, burnin=100))
    assert chain.samples.shape == (900, 3) and list(chain.samples.columns) == ["pars.1", "pars.2", "pars.3"]
    assert chain.gradients.shape == (900, 3) and chain.gradients.isna().all().all()                   # SerialMC.jl:42
    assert list(chain.diagnostics["step"][:3]) == [101, 102, 103] and chain.diagnostics["accept"].dtype == bool
    assert mj.run(m1 * mj.RWM(0.1) * mj.SerialMC(range(101, 1001, 5))).samples.shape == (180, 3)
    c2 = mj.run(m2, mj.HMC(0.75), mj.SerialMC(steps=10000, burnin=1000))
    assert 77 < mj.acceptance(c2) < 83                                                                 # README.md:121
    e = mj.ess(c2); a = mj.actime(c2)
    assert e.shape == (3,) and np.all((0.48 * 9000 < e) & (e < 0.70 * 9000)) and np.all((1.4 < a) & (a < 2.1))
    s = c2.samples.values
    assert np.allclose(mj.var(c2, vtype="iid"), [O.mcvar(s[:, j], "iid") for j in range(3)], rtol=1e-13)
    assert np.allclose(mj.var(c2), [O.mcvar(s[:, j], "imse") for j in range(3)], rtol=1e-12)
    assert np.allclose(mj.var(c2, vtype="bm"), [O.mcvar(s[:, j], "bm") for j in range(3)], rtol=1e-12)
    assert np.allclose(mj.std(c2, vtype="ipse"), np.sqrt([O.mcvar(s[:, j], "ipse") for j in range(3)]), rtol=1e-12)
    assert np.allclose(mj.mean(c2), s.mean(0), rtol=0, atol=1e-14)
    assert np.allclose(c2.gradients.values, -2 * s)
    with pytest.raises(AssertionError):
        mj.run(m1 * mj.MALA(0.1) * mj.SerialMC(1, 1000))                                               # test_syntax.jl:75
    chains = mj.run(m2 * [mj.RWM(0.1), mj.MALA(0.1), mj.HMC(3, 0.1)] * mj.SerialMC(steps=1000))        # test_syntax.jl:79
    assert len(chains) == 3 and chains[1].samples.shape == (1000, 3)
    again = mj.resume(chain, steps=500)
    assert again.samples.shape == (500, 3)
    batch = mj.run(m2 * mj.HMC(0.75) * mj.GPUMC(steps=2000, burnin=200, nchains=512, seed=3))
    assert len(batch) == 512 and batch[5].samples.shape == (1800, 3)
    acc = mj.acceptance(batch)
    assert acc.shape == (512,) and 78 < acc.mean() < 82
    assert mj.ess(batch).shape == (512, 3)
    batch.close()
    import io
    buf = io.StringIO(); mj.describe(c2, buf)
    assert "MC Error" in buf.getvalue() and "pars.3" in buf.getvalue()
    with pytest.raises(AssertionError):
        mj.model("ou", x=ou_series(30, 1), tau=-0.05, sigma=1.0, mu=1.0)                               # likmodel.jl:54


def test_full_size_properties_config2(capi, ctx):
    """BASELINE config 2 shape (65 536 chains, HMC(0.75), 3-D target N(0, I/2)): moments within Monte Carlo error,
    acceptance in the README band, KS distance to the exact cdf (the reference's test_dists.jl method with a real threshold)."""
    from scipy.stats import norm, kstest
    C, d = 65536, 3
    dm = capi.DeviceModel(ctx, "normal_fn", d)
    run = capi.DeviceRun(dm, capi.sampler_cfg("HMC", scale=0.75, nleaps=10), (101, 1, 400), C, np.ones(d), seed=1, store_grad=False, store_logtarget=False)
    info = run.execute()
    assert info["n_grad_evals"] == C * (1 + 400 * 10)
    st = run.stats("imse")
    assert 79.0 < st["accept_rate"].mean() < 81.0
    gm = st["mean"].mean(0)
    assert np.all(np.abs(gm) < 5 * math.sqrt(0.5 / (C * 300 * 0.55)))
    out = run.fetch(grads=False, logtarget=False)
    last = out["samples"][:, -1, :]                            # one draw per chain: independent across chains
    assert np.all(np.abs(last.var(0) - 0.5) < 5 * 0.5 * math.sqrt(2 / C))
    for j in range(d):
        assert kstest(last[::8, j], norm(0, math.sqrt(0.5)).cdf).statistic < 1.63 / math.sqrt(C / 8)   # alpha = 0.01
    ess = st["ess"]
    assert 0.45 < np.median(ess) / 300 < 0.75
    run.close(); dm.close()


def test_linear_regression_posterior_moments(capi, ctx):
    """linear model: Gaussian posterior in closed form; many-chain HMC means must match within MC error"""
    N, d, C = 500, 5, 2048
    X, y, hy, _ = make_regression("linear", N, d, 11)
    P = X.T @ X + np.eye(d)                                   # prior N(0, I), noise sd 1
    mu = np.linalg.solve(P, X.T @ y); cov = np.linalg.inv(P)
    dm = capi.DeviceModel(ctx, "linear", d, X, y, hy)
    run = capi.DeviceRun(dm, capi.sampler_cfg("HMC", scale=0.04, nleaps=12), (201, 1, 500), C, mu, seed=2, store_grad=False)
    run.execute()
    out = run.fetch(grads=False, logtarget=False)
    assert 0.6 < out["accept"].mean() < 1.0
    last = out["samples"][:, -1, :]
    assert np.all(np.abs(last.mean(0) - mu) < 5 * np.sqrt(np.diag(cov) / C))
    assert np.all(np.abs(last.var(0) / np.diag(cov) - 1) < 5 * math.sqrt(2 / C))
    run.close(); dm.close()


def test_dsl_models_end_to_end(O):
    """model(expression, ...) for the reference's example models (SURVEY 8f.3), as test/test_syntax.jl:9-34 uses them"""
    import mcmc_jl_b200 as mj
    rng = np.random.default_rng(1)
    n, nbeta = 1000, 10
    X = np.concatenate([np.ones((n, 1)), rng.standard_normal((n, nbeta - 1))], axis=1)
    beta0 = rng.standard_normal(nbeta)
    Y = (rng.random(n) < 1 / (1 + np.exp(-X @ beta0))).astype(float)
    ex = """
        vars ~ Normal(0, 1.0)  # Normal prior, std 1.0 for predictors
        prob = 1 / (1. + exp(- X * vars))
        Y ~ Bernoulli(prob)
    """
    m = mj.model(ex, vars=np.zeros(nbeta), gradient=True, X=X, Y=Y)
    om = O.Model("logistic", nbeta, X, Y, (1.0, -1.0))
    lt, g = m.evalallg(m.init)
    olt, og = om.evalallg(np.zeros(nbeta))
    assert abs(lt - olt) <= 1e-12 * abs(olt) and np.allclose(g, og, rtol=1e-11, atol=1e-9)
    for smp in (mj.RWM(0.05), mj.HMC(2, 0.1), mj.MALA(0.001)):                       # test/test_syntax.jl:25-28
        res = mj.run(m * smp * mj.SerialMC(100, 1000))
        assert res.samples.shape == (901, nbeta) and list(res.samples.columns)[:2] == ["vars.1", "vars.2"]
        assert np.isfinite(res.samples.values).all()
    res = mj.run(m, mj.HMC(2, 0.1), mj.SerialMC(thinning=10, burnin=0))              # test_syntax.jl:33
    assert res.samples.shape == (10, nbeta)
    m0 = mj.model(ex, vars=np.zeros(nbeta), gradient=False, X=X, Y=Y)
    with pytest.raises(AssertionError):
        mj.run(m0 * mj.HMC(2, 0.1) * mj.SerialMC(1, 10))                             # HMC.jl:111
    ou = mj.model("""tau ~ Uniform(0, 100)
                     sigma ~ Uniform(0, 2)
                     mu ~ Uniform(0, 20)
                     fac = exp(- 1. / tau)
                     resid = x[2:end] - x[1:end-1] * fac - mu * (1. - fac)
                     resid ~ Normal(0, sigma)""", tau=0.05, sigma=1.0, mu=1.0, gradient=True, x=ou_series(1000, 1),
                  scale=np.array([1000.0, 1.0, 10.0]))
    res = mj.run(ou * mj.HMC(5, 0.002) * mj.SerialMC(1000, 2000))                    # examples/ornstein.jl:38
    assert list(res.samples.columns) == ["tau", "sigma", "mu"] and res.samples.shape == (1001, 3)


def test_run_chains_single_call(O, capi, ctx):
    """mcmcgpu_run_chains: the one-call form the Julia glue uses (create + execute + fetch + destroy)"""
    import ctypes as C
    d, Cn, rngt = 3, 17, (11, 3, 100)
    S = len(range(rngt[0], rngt[2] + 1, rngt[1]))
    dm = capi.DeviceModel(ctx, "normal_fn", d)
    scfg = capi.sampler_cfg("HMC", scale=0.75, nleaps=10)
    r = capi.RunnerCfg()
    r.first, r.step, r.last, r.nchains, r.chain_offset, r.seed = rngt[0], rngt[1], rngt[2], Cn, 0, 0
    rng = np.random.default_rng(4)
    zn = rng.standard_normal((Cn, rngt[2] + 1, d)); un = rng.random((Cn, rngt[2] + 1))
    samples = np.empty((Cn, S, d)); grads = np.empty((Cn, S, d)); acc = np.empty((Cn, S), dtype=np.uint8); lt = np.empty((Cn, S))
    info = capi.RunInfo()
    init = np.ones(d)
    capi.check(capi.lib().mcmcgpu_run_chains(dm.h, C.byref(scfg), C.byref(r), capi.dptr(init), None, capi.dptr(zn), capi.dptr(un),
                                            capi.dptr(samples), capi.dptr(grads), acc.ctypes.data_as(C.POINTER(C.c_uint8)),
                                            capi.dptr(lt), C.byref(info)))
    om = O.Model("normal_fn", d)
    for c in range(Cn):
        ref = O.run_chain(om, O.sampler("HMC", scale=0.75, nleaps=10), rngt, init, None, zn[c], un[c])
        assert np.array_equal(ref["samples"], samples[c]) and np.array_equal(ref["accept"], acc[c])
        assert np.array_equal(ref["grads"], grads[c]) and np.array_equal(ref["logtarget"], lt[c])
    assert info.n_launches == 1 and info.n_grad_evals == Cn * (1 + rngt[2] * 10)
    dm.close()


@pytest.mark.parametrize("engine", ["fused", "wave"])
@pytest.mark.parametrize("fam,d,hy", [("normal_fn", 3, ()), ("normal_dsl", 6, (0.5, 2.0)), ("normal_fn", 1, ())])
def test_ram_closed_form(O, capi, ctx, engine, fam, d, hy):
    """RAM.jl:41-80 (SURVEY 8f.4): the factor update S = chol(S (I + eta (alpha - rate) r r'/|r|^2) S')' in the reference's
    operation order; pow() differs in the last bit between CUDA and glibc, hence a tolerance instead of bit equality"""
    C, rngt = 40, (51, 1, 400)
    out, diag, refs, _ = _run_both(O, capi, ctx, fam, d, None, None, hy, "RAM", dict(scale=1.0, rate=0.234), rngt, C, np.ones(d), engine)
    for c in range(C):
        assert np.array_equal(refs[c]["accept"], out["accept"][c])
        assert np.allclose(refs[c]["samples"], out["samples"][c], rtol=1e-9, atol=1e-12)
        assert np.allclose(diag[0][c], refs[c]["eps"], rtol=1e-9)           # "scale" diagnostic = trace(S)
        assert np.all(np.isnan(out["grads"][c]))
    acc = out["accept"][:, 200:].mean()
    assert 0.15 < acc < 0.40                                                 # coerced towards the target rate 0.234


def test_ram_examples(O, capi, ctx):
    """examples/linear_regression.jl:26 `RAM(1., 0.3)` (d = 10, wave engine) and examples/ornstein.jl:33 `RAM()` with m.scale"""
    X, y, hy, _ = make_regression("linear", 1000, 10, 3)
    out, diag, refs, _ = _run_both(O, capi, ctx, "linear", 10, X, y, hy, "RAM", dict(scale=1.0, rate=0.3), (101, 1, 400), 24, np.zeros(10), "wave")
    for c in range(24):
        assert np.array_equal(refs[c]["accept"], out["accept"][c])
        assert np.allclose(refs[c]["samples"], out["samples"][c], rtol=1e-8, atol=1e-11)
        assert np.allclose(diag[0][c], refs[c]["eps"], rtol=1e-8)
    x = ou_series(300, 4)
    sc = np.array([1000.0, 1.0, 10.0])
    for engine in ("fused", "wave"):
        out, diag, refs, _ = _run_both(O, capi, ctx, "ou", 3, None, x, (100.0, 2.0, 20.0), "RAM", dict(scale=1.0, rate=0.234), (1, 1, 200), 16,
                                       np.array([20.0, 0.1, 10.0]), engine, scale=sc)
        for c in range(16):
            assert np.array_equal(refs[c]["accept"], out["accept"][c])
            assert np.allclose(refs[c]["samples"], out["samples"][c], rtol=1e-8, atol=0)
    import mcmc_jl_b200 as mj
    m = mj.model("linear", X=X, Y=y, vars=np.zeros(10))
    ch = mj.run(m * mj.RAM(1.0, 0.3) * mj.SerialMC(1000, 5000))
    assert 20 < mj.acceptance(ch) < 40                                       # linear_regression.jl:27 "~ 29.7%"


@pytest.mark.parametrize("order", [1, 2])
def test_zv_control_variates(O, capi, ctx, order):
    """linearZv / quadraticZv (src/stats/zv.jl:8-66, SURVEY 8f.4) on the device against the oracle (same elimination,
    bit for bit) and against a numpy restatement that calls inv() like the reference"""
    X, y, hy, _ = make_regression("logistic", 300, 4, 6)
    dm = capi.DeviceModel(ctx, "logistic", 4, X, y, hy)
    run = capi.DeviceRun(dm, capi.sampler_cfg("HMC", scale=0.05, nleaps=5), (201, 1, 1200), 70, np.zeros(4), seed=3, engine="wave")
    run.execute()
    out = run.fetch()
    zv, a = run.zv(order)
    zv2, a2 = ctx.zv(out["samples"], out["grads"], order)                      # host-array entry point
    assert np.array_equal(zv, zv2) and np.array_equal(a, a2)
    d = 4
    k = d if order == 1 else d * (d + 3) // 2
    assert a.shape == (70, k, d)
    for c in range(0, 70, 9):
        x, g = out["samples"][c], out["grads"][c]
        ozv, oa = O.zv(x, g, order)
        assert np.array_equal(a[c], oa) and np.allclose(zv[c], ozv, rtol=0, atol=1e-13)
        z = -g / 2
        feats = [z] if order == 1 else [z, 2 * z * x - 1] + [np.column_stack([x[:, i] * z[:, j] + x[:, j] * z[:, i] for i in range(d - 1) for j in range(i + 1, d)])]
        F = np.column_stack(feats)
        ar = np.empty((k, d))
        for i in range(d):
            cv = np.cov(np.column_stack([F, x[:, i]]), rowvar=False)
            ar[:, i] = -np.linalg.inv(cv[:k, :k]) @ cv[:k, k]
        assert np.allclose(a[c], ar, rtol=1e-7, atol=1e-9)
        assert np.all(zv[c].var(0) < 0.35 * x.var(0))                          # the control variates do reduce variance
        assert np.allclose(zv[c].mean(0), x.mean(0), atol=5 * x.std(0) / np.sqrt(30))
    run.close(); dm.close()
    import mcmc_jl_b200 as mj
    ch = mj.run(mj.model("normal", init=np.ones(3)) * mj.HMC(0.75) * mj.SerialMC(steps=3000, burnin=300))
    zvc, aa = (mj.linearZv if order == 1 else mj.quadraticZv)(ch)
    assert zvc.shape == (2700, 3) and np.all(np.abs(zvc) < 1e-9)               # Gaussian target: z = x, the estimator is exact


@pytest.mark.parametrize("engine", ["fused", "wave"])
def test_store_leaps_rao_blackwell(O, capi, ctx, engine):
    """HMC storeLeaps + mean_rb (HMC.jl:145-150, src/stats/mean.jl:11-41, SURVEY 8f.2): the Rao-Blackwell sums are
    accumulated over the leap states on the device; the oracle keeps the leap states and applies mean.jl literally"""
    d, C, rngt = 3, 50, (21, 1, 300)
    rng = np.random.default_rng(12)
    zn = rng.standard_normal((C, rngt[2] + 1, d)); un = rng.random((C, rngt[2] + 1))
    dm = capi.DeviceModel(ctx, "normal_fn", d)
    run = capi.DeviceRun(dm, capi.sampler_cfg("HMC", scale=0.4, nleaps=6), rngt, C, np.ones(d), normals=zn, uniforms=un, engine=engine, store_rb=True)
    run.execute(); out = run.fetch(); rb = run.fetch_rb()
    om = O.Model("normal_fn", d)
    S = out["samples"].shape[1]
    for c in range(C):
        orb = np.full((S, d), np.nan)
        ref = O.run_chain(om, O.sampler("HMC", scale=0.4, nleaps=6, rb_out=orb), rngt, np.ones(d), None, zn[c], un[c])
        assert np.array_equal(ref["samples"], out["samples"][c]) and np.array_equal(ref["accept"], out["accept"][c])
        assert np.allclose(rb[c], orb, rtol=1e-13, atol=1e-15)
    run.close(); dm.close()
    import mcmc_jl_b200 as mj
    ch = mj.run(mj.model("normal", init=np.ones(3)) * mj.HMC(0.3, storeLeaps=True) * mj.SerialMC(steps=4000, burnin=500))
    m_rb, m = mj.mean_rb(ch), mj.mean(ch)
    assert m_rb.shape == (3,) and np.all(np.abs(m_rb) < 0.1) and np.all(np.abs(m) < 0.1)


def test_edge_shapes(O, capi, ctx):
    """smallest and most ragged shapes: one observation, one parameter, one chain, one kept step, thinning past the end,
    a single leapfrog, the HMCDA leap cap"""
    rng = np.random.default_rng(21)
    # N = 1, d = 1, C = 1 regression
    X = np.array([[1.0]]); y = np.array([1.0])
    for fam, hy in (("linear", (1.0, 1.0)), ("logistic", (1.0, -1.0)), ("probit", (10.0,))):
        dm = capi.DeviceModel(ctx, fam, 1, X, y, hy)
        om = O.Model(fam, 1, X, y, hy)
        lt, g = dm.logtarget_grad(np.array([[0.3]]))
        olt, og = om.evalallg(np.array([0.3]))
        assert abs(lt[0] - olt) <= 1e-13 * abs(olt) and abs(g[0, 0] - og[0]) <= 1e-13
        zn = rng.standard_normal((1, 6, 1)); un = rng.random((1, 6))
        for rngt in ((5, 1, 5), (2, 7, 5), (1, 1, 1)):                       # one kept step; thinning past the end; one step in all
            zz, uu = zn[:, :rngt[2] + 1], un[:, :rngt[2] + 1]
            run = capi.DeviceRun(dm, capi.sampler_cfg("HMC", scale=0.3, nleaps=1), rngt, 1, np.zeros(1), normals=zz, uniforms=uu, engine="wave")
            run.execute(); out = run.fetch()
            ref = O.run_chain(om, O.sampler("HMC", scale=0.3, nleaps=1), rngt, np.zeros(1), None, zz[0], uu[0])
            assert out["samples"].shape == (1, 1, 1) and np.array_equal(out["accept"][0], ref["accept"])
            assert np.allclose(out["samples"][0], ref["samples"], rtol=1e-12, atol=1e-15)
            run.close()
        dm.close()
    # HMCDA with a tiny leap cap: nLeaps = min(round(len/eps), max_leaps)
    dm = capi.DeviceModel(ctx, "normal_fn", 2)
    zn = rng.standard_normal((3, 41, 2)); un = rng.random((3, 41))
    for engine in ("fused", "wave"):
        run = capi.DeviceRun(dm, capi.sampler_cfg("HMCDA", len=50.0, max_leaps=7), (1, 1, 40), 3, np.ones(2), normals=zn, uniforms=un, engine=engine)
        run.execute(); out = run.fetch(); eps, nl = run.fetch_diag()
        assert np.all(nl == 7) and np.all(eps == 1.0)                         # burn-in 0: eps stays 1, round(50/1) = 50 capped at 7
        for c in range(3):
            ref = O.run_chain(O.Model("normal_fn", 2), O.sampler("HMCDA", len=50.0, max_leaps=7), (1, 1, 40), np.ones(2), None, zn[c], un[c])
            assert np.array_equal(out["samples"][c], ref["samples"]) and np.array_equal(out["accept"][c], ref["accept"])
        run.close()
    dm.close()
    # per-chain initial values (d x nchains init), RWM with model.scale
    dm = capi.DeviceModel(ctx, "normal_dsl", 3, hyper=(1.0, 0.5))
    init = rng.standard_normal((5, 3)); sc = np.array([0.5, 1.0, 2.0])
    zn = rng.standard_normal((5, 31, 3)); un = rng.random((5, 31))
    for engine in ("fused", "wave"):
        run = capi.DeviceRun(dm, capi.sampler_cfg("RWM", scale=0.3), (1, 1, 30), 5, init, scale=sc, normals=zn, uniforms=un, engine=engine)
        run.execute(); out = run.fetch()
        for c in range(5):
            ref = O.run_chain(O.Model("normal_dsl", 3, hyper=(1.0, 0.5)), O.sampler("RWM", scale=0.3), (1, 1, 30), init[c], sc, zn[c], un[c])
            assert np.array_equal(out["samples"][c], ref["samples"])
        run.close()
    dm.close()


@pytest.mark.parametrize("fam", ["logistic", "probit"])
def test_link_functions_over_wide_range(O, capi, ctx, fam):
    """the kernel's own exp / reciprocal / log / table-driven log Phi and phi/Phi over the whole range of eta, incl. the
    libm fall-back paths (|eta| >= 36.9 probit, >= 700 logistic).  For the logistic model the reference forms 1 - p by
    subtraction, so its log-likelihood is ill-conditioned where p -> 1: the tolerance carries that conditioning."""
    from scipy.special import log_ndtr, expit
    rng = np.random.default_rng(5)
    N, d = 4000, 2
    X = np.column_stack([np.ones(N), np.linspace(-1, 1, N)])
    y = (rng.random(N) < 0.5).astype(float)
    hy = (1.0, -1.0) if fam == "logistic" else (10.0,)
    om, dm = O.Model(fam, d, X, y, hy), capi.DeviceModel(ctx, fam, d, X, y, hy)
    scales = [0.5, 3.0, 10.0, 25.0, 34.0] + ([36.0, 40.0, 300.0] if fam == "probit" else [])
    B = np.array([[rng.normal(0, 0.3), s] for s in scales])            # eta spans [-s, s]
    lt, g = dm.logtarget_grad(B)
    for c, b in enumerate(B):
        olt, og = om.evalallg(b)
        eta = X @ b
        if fam == "logistic":
            p = expit(eta)
            cond = np.sum(np.finfo(float).eps / np.minimum(np.where(y == 1, p, 1 - p), 1.0))   # |d log(1-p)| for a last-bit change of p
            assert abs(lt[c] - olt) <= 1e-12 * abs(olt) + 4 * cond, (c, lt[c], olt)
            assert np.all(np.abs(g[c] - og) <= 1e-11 * np.abs(X).sum(0) + 4 * cond), c
        else:
            truth = np.sum(np.where(y == 1, log_ndtr(eta), log_ndtr(-eta))) - 0.5 * (d * np.log(2 * np.pi) + d * np.log(100.0)) - 0.5 * (b @ b) / 100.0
            assert abs(lt[c] - olt) <= 1e-12 * abs(olt) and abs(lt[c] - truth) <= 1e-11 * abs(truth), (c, lt[c], olt, truth)
            assert np.all(np.abs(g[c] - og) <= 1e-11 * (np.abs(X) * np.maximum(1.0, np.abs(eta))[:, None]).sum(0)), c
    # far beyond every fast path: logistic saturates to the support boundary, the sampler must see (-Inf, zeros)
    if fam == "logistic":
        lt2, g2 = dm.logtarget_grad(np.array([[0.0, 800.0], [0.0, 40.0]]))
        o0, o1 = om.evalallg(np.array([0.0, 800.0])), om.evalallg(np.array([0.0, 40.0]))
        assert lt2[0] == o0[0] == -np.inf and np.all(g2[0] == 0)
        assert (lt2[1] == -np.inf) == (o1[0] == -np.inf)
    dm.close()


@pytest.mark.parametrize("sign", [-1.0, 1.0])
def test_logistic_link_elementwise(capi, ctx, sign):
    """r = d loglik / d eta of the logistic link, element by element (N = 1, X = [1], one chain per eta), against mpmath:
    the table-driven exp (tools/gen_exp_table.py), the cubic reciprocal step and the sign handling on bit patterns of
    K1's fast path must keep ~1e-15 relative accuracy over the whole fast range, for both sign conventions
    (examples/logistic_regression.jl:18, test/test_syntax.jl:18) and both responses."""
    import mpmath as mp
    mp.mp.dps = 40
    rng = np.random.default_rng(11)
    eta = np.concatenate([np.linspace(-36.5, 36.5, 1500), rng.uniform(-5, 5, 1500), rng.uniform(-690, 690, 200), [0.0, 1e-300, -1e-17]])
    sd = 1e6
    for yval in (1.0, 0.0):
        dm = capi.DeviceModel(ctx, "logistic", 1, np.ones((1, 1)), np.array([yval]), (sd, sign))
        lt, g = dm.logtarget_grad(eta.reshape(-1, 1))
        for c, b in enumerate(eta):
            x = mp.mpf(sign) * mp.mpf(float(b))
            pr = 1 / (1 + mp.exp(x))                                   # prob = 1/(1 + exp(sign * eta))
            r = (-mp.mpf(sign) * (1 - pr)) if yval == 1.0 else mp.mpf(sign) * pr
            truth = r - mp.mpf(float(b)) / (sd * sd)
            if yval == 0.0 and sign * b <= -36.736800569677101:        # 1 - p == 0 in binary64: out of support, (-Inf, zeros)
                assert lt[c] == -np.inf and g[c, 0] == 0.0
                continue
            assert abs(mp.mpf(float(g[c, 0])) - truth) <= mp.mpf(1e-15) * (abs(r) + abs(mp.mpf(float(b))) / (sd * sd)), (sign, yval, b, g[c, 0], truth)
            assert np.isfinite(lt[c])
        dm.close()
    with pytest.raises(capi.MCMCGPUError):
        capi.DeviceModel(ctx, "logistic", 1, np.ones((1, 1)), np.array([1.0]), (1.0, -2.0))     # sign must be +-1


def test_probit_link_elementwise(capi, ctx):
    """log Phi(+-eta) and r = +-phi/Phi of the probit link, element by element (N = 1, X = [1], one chain per eta), against
    mpmath: the two-doubles-and-a-float-pair table of K1's fast path (tools/gen_probit_table.py: W', W'' from
    W' = -W (z + W) in double, the cubic / quartic tail in float, the grid index in float) must keep the accuracy the
    generator's emulation states -- relative for z < 0, absolute for z >= 0 -- over the whole fast range incl. grid points,
    interval edges and the shared-memory / global-memory table boundary at |z| = 8; the libm path takes over at 36.9
    (examples/probit_regression.jl:29,39-40)."""
    import mpmath as mp
    mp.mp.dps = 40
    rng = np.random.default_rng(12)
    grid = np.arange(-1100, 1100) / 128.0
    eta = np.concatenate([np.linspace(-36.8, 36.8, 1200), rng.uniform(-6, 6, 1500), grid[::7], grid[::11] + 0.99 / 256, grid[::13] - 0.99 / 256,
                          [0.0, 1e-300, -1e-17, 7.999, 8.001, -7.999, -8.001, 36.89, -36.89, 36.95, -36.95, 39.0, -39.0]])
    sd = 1e6
    prior = lambda b: -0.5 * (mp.log(2 * mp.pi) + 2 * mp.log(sd)) - mp.mpf(float(b)) ** 2 / (2 * mp.mpf(sd) ** 2)
    for yval in (1.0, 0.0):
        dm = capi.DeviceModel(ctx, "probit", 1, np.ones((1, 1)), np.array([yval]), (sd,))
        lt, g = dm.logtarget_grad(eta.reshape(-1, 1))
        for c, b in enumerate(eta):
            z = mp.mpf(float(b)) if yval == 1.0 else -mp.mpf(float(b))
            F = mp.log(mp.ncdf(z))
            W = mp.npdf(z) / mp.ncdf(z)
            r = W if yval == 1.0 else -W
            tol_f = 1e-15 * abs(F) + 4e-16 + 3e-16 * abs(prior(b))
            tol_w = (5e-15 * abs(W) if z < 0 else 6e-15) + 1e-16 * abs(float(b)) / (sd * sd)
            assert abs(mp.mpf(float(lt[c])) - (F + prior(b))) <= tol_f, (yval, b, lt[c], F + prior(b))
            assert abs(mp.mpf(float(g[c, 0])) - (r - mp.mpf(float(b)) / (sd * sd))) <= tol_w, (yval, b, g[c, 0], r)
        dm.close()
    # a response that is neither 0 nor 1 sends the whole model down the general path (the table path tests y once, at pack time)
    dm = capi.DeviceModel(ctx, "probit", 1, np.ones((2, 1)), np.array([1.0, 0.5]), (sd,))
    lt, g = dm.logtarget_grad(np.array([[0.3]]))
    truth = mp.log(mp.ncdf(0.3)) + 0.5 * mp.log(mp.ncdf(0.3)) + 0.5 * mp.log(mp.ncdf(-0.3)) + prior(0.3)
    assert abs(mp.mpf(float(lt[0])) - truth) <= 1e-14 * abs(truth)
    dm.close()


def test_readme_snippet():
    """the usage example of README.md runs as written"""
    import mcmc_jl_b200 as mj
    rng = np.random.default_rng(2)
    X = np.concatenate([np.ones((1000, 1)), rng.standard_normal((1000, 9))], axis=1)
    Y = (rng.random(1000) < 1 / (1 + np.exp(-X @ rng.standard_normal(10)))).astype(float)
    m = mj.model("""vars ~ Normal(0, 1.0)
                   prob = 1 / (1. + exp(- X * vars))
                   Y ~ Bernoulli(prob)""", vars=np.zeros(10), gradient=True, X=X, Y=Y)
    chain = mj.run(m * mj.HMC(2, 0.1) * mj.SerialMC(1000, 10000))
    batch = mj.run(m * mj.HMCDA(len=0.2) * mj.GPUMC(steps=2000, burnin=1000, nchains=4096, seed=1))
    acc, ess_min, vbm, (zv, a) = mj.acceptance(chain), mj.ess(batch).min(axis=1), mj.var(chain, vtype="bm"), mj.linearZv(chain)
    assert 20 < acc <= 100 and ess_min.shape == (4096,) and vbm.shape == (10,) and zv.shape == (9001, 10) and a.shape == (10, 10)
    assert np.median(mj.acceptance(batch)) > 40 and np.isfinite(batch[7].samples.values).all()
    assert np.all(zv.var(0) < chain.samples.values.var(0))
    batch.close()


# ---- the headline regime (BASELINE configs[3]: HMCDA on the logistic regression through K1 + leapfrog waves) ---------------
def _oracle_chains(O, om, jobs):
    """oracle chains on a thread pool (ctypes releases the GIL): jobs = [(sampler, range, init, normals, uniforms)]"""
    from concurrent.futures import ThreadPoolExecutor
    import os
    with ThreadPoolExecutor(max_workers=min(32, os.cpu_count() or 1)) as ex:
        return list(ex.map(lambda j: O.run_chain(om, j[0], j[1], j[2], None, j[3], j[4]), jobs))


def _headline_problem(seed=11):
    N, d, C = 4097, 100, 130
    X, y, hy, b0 = make_regression("logistic", N, d, seed)
    sc = math.sqrt(1e6 / N)                         # posterior scale relative to cfg4's N = 1e6
    rng = np.random.default_rng(seed + 1)
    eps = rng.uniform(1.2e-3, 2.2e-3, size=C) * sc  # per-chain step sizes around the adapted value of cfg4 (1.97e-3)
    init = b0[None, :] + 0.02 * rng.standard_normal((C, d))
    return N, d, C, X, y, hy, eps, 0.02 * sc, init, rng


def test_hmcda_headline_regime_frozen_phase(O, capi, ctx):
    """HMCDA on logistic, d = 100, per-chain step sizes restored with set_state (the state bench.py's cfg4 runs in):
    ~8-17 leapfrogs per step, different per chain, so every wave mixes chains that finish a trajectory with chains in
    the middle of one.  Draw-matched against the oracle: identical accept flags and leap counts, samples to 1e-9."""
    N, d, C, X, y, hy, eps, L, init, rng = _headline_problem()
    K = 32
    zn = rng.standard_normal((C, K + 1, d)); un = rng.random((C, K + 1))
    dm = capi.DeviceModel(ctx, "logistic", d, X, y, hy)
    om = O.Model("logistic", d, X, y, hy)
    run = capi.DeviceRun(dm, capi.sampler_cfg("HMCDA", len=L, max_leaps=64), (1, 1, K), C, init, normals=zn, uniforms=un, engine="wave")
    run.set_state(0, eps, eps, np.zeros(C))
    info = run.execute(); out = run.fetch(); geps, gnl = run.fetch_diag()
    run.close(); dm.close()
    refs = _oracle_chains(O, om, [(O.sampler("HMCDA", len=L, max_leaps=64, da_state=[eps[c], eps[c], 0.0]), (1, 1, K), init[c], zn[c], un[c])
                                  for c in range(C)])
    acc = out["accept"].mean()
    assert 0.3 < acc < 1.0                                                      # a real mix of accepts and rejects
    assert len(np.unique(gnl)) >= 5 and gnl.min() >= 6 and gnl.max() <= 20      # mixed trajectory lengths in every wave
    assert info["n_grad_evals"] == C + gnl.sum()
    gs = np.abs(X).sum(0)
    for c in range(C):
        r = refs[c]
        assert r["rc"] == 0
        assert np.array_equal(r["accept"], out["accept"][c]), c
        assert np.array_equal(r["nleaps"], gnl[c]) and np.array_equal(r["eps"], geps[c]), c
        assert np.allclose(r["samples"], out["samples"][c], rtol=1e-9, atol=1e-12), c
        assert np.allclose(r["logtarget"], out["logtarget"][c], rtol=1e-11, atol=0), c
        assert np.all(np.abs(r["grads"] - out["grads"][c]) <= 1e-9 * gs), c
    assert sum(int(r["accept"].sum()) for r in refs) == int(out["accept"].sum()) > 0.3 * C * K


def test_hmcda_headline_regime_adapting(O, capi, ctx):
    """the same regime with the dual averaging ON (i < burnin, HMCDA.jl:133-138), continued from a restored state at step
    100 whose dualH is consistent with the step size (eps = exp(mu - sqrt(i) dualH / shrinkage)): 25 adapting steps, then
    15 kept ones.  The adaptation multiplies a difference in the acceptance probability by sqrt(i)/shrinkage = 200, so the
    oracle is teacher-forced (it replays every trajectory with the GPU's step size, read back after every burn-in step
    through the stepwise API, and reports its OWN adapted step sizes): decisions and leap counts identical, samples to
    1e-9, step sizes to 1e-7.  The stepwise run must also equal the asynchronous one-call run bit for bit."""
    N, d, C, X, y, hy, eps, L, init, rng = _headline_problem(seed=12)
    s0, B, last = 100, 125, 140
    dualH = (math.log(10.0) - np.log(eps)) * 0.05 / math.sqrt(s0)
    zn = rng.standard_normal((C, last + 1, d)); un = rng.random((C, last + 1))
    dm = capi.DeviceModel(ctx, "logistic", d, X, y, hy)
    om = O.Model("logistic", d, X, y, hy)
    mk = lambda: capi.DeviceRun(dm, capi.sampler_cfg("HMCDA", len=L, max_leaps=64), (B + 1, 1, last), C, init, normals=zn, uniforms=un, engine="wave")
    one = mk(); one.set_state(s0, eps, eps, dualH); one.execute(); out1 = one.fetch(); one.close()     # asynchronous leapfrog waves
    run = mk(); run.set_state(s0, eps, eps, dualH)
    fe = np.full((C, last + 1), np.nan)
    fe[:, s0 + 1] = eps
    for i in range(s0 + 1, B + 1):                       # after step i the state holds the step size of step i + 1
        run.execute_steps(1)
        fe[:, i + 1] = run.get_state()["leapstep"]
    fe[:, B + 1:] = fe[:, B + 1][:, None]                # frozen phase: leapStep = dualLeapStep (HMCDA.jl:140)
    run.execute_steps(last - B)
    out = run.fetch(); geps, gnl = run.fetch_diag(); st = run.get_state()
    run.close(); dm.close()
    assert np.array_equal(out["samples"], out1["samples"]) and np.array_equal(out["accept"], out1["accept"])
    assert np.array_equal(geps, fe[:, B + 1:])
    refs = _oracle_chains(O, om, [(O.sampler("HMCDA", len=L, max_leaps=64, start_step=s0, da_state=[eps[c], eps[c], dualH[c]], force_eps=fe[c]),
                                   (B + 1, 1, last), init[c], zn[c], un[c]) for c in range(C)])
    assert 0.3 < out["accept"].mean() < 1.0
    assert np.abs(geps[:, 0] / eps - 1).max() > 0.02                              # the adaptation moved the step sizes
    assert len(np.unique(np.round(L / fe[:, s0 + 1:B + 1]))) >= 5                 # and the leap counts differed during it
    for c in range(C):
        r = refs[c]
        assert np.array_equal(r["accept"], out["accept"][c]), c
        assert np.array_equal(r["nleaps"], gnl[c]), c
        assert np.allclose(r["eps"], geps[c], rtol=1e-7, atol=0), c              # the oracle's own adaptation == the GPU's
        assert np.allclose(r["samples"], out["samples"][c], rtol=1e-9, atol=1e-12), c
        assert np.allclose(st["leapstep"][c], r["eps"][-1], rtol=1e-7)            # frozen phase: leapStep = dualLeapStep


@pytest.mark.parametrize("name,fam,N,d,C,splits", [("cfg4", "logistic", 1000000, 100, 10000, 13), ("cfg4-auto", "logistic", 1000000, 100, 8, 0),
                                                   ("cfg3", "probit", 100000, 20, 16384, 0), ("cfg5-shard", "logistic", 200000, 200, 512, 0)])
def test_full_geometry_logtarget_gradient(O, capi, ctx, name, fam, N, d, C, splits):
    """one likelihood launch at the launch geometry of each BASELINE config (cfg4: 157 chain tiles x 13 row splits over
    31 250 row tiles; cfg3: 256 chain tiles, 3 CTAs per SM; cfg5: d = 200, one CTA per SM), 8 chains spread over the
    chain tiles checked against the oracle at 1e-12."""
    import bench
    X, y, b0 = (bench.synth_logistic if fam == "logistic" else bench.synth_probit)(N, d, 4 if fam == "logistic" else 3)
    hy = (1.0, -1.0) if fam == "logistic" else (10.0,)
    dm = capi.DeviceModel(ctx, fam, d, X, y, hy)
    om = O.Model(fam, d, X, y, hy)
    rng = np.random.default_rng(N + d)
    B = b0[None, :] + (2.0 / math.sqrt(N)) * rng.standard_normal((C, d))
    ctx.set_option("force_splits", splits)
    try:
        lt, g = dm.logtarget_grad(B)
    finally:
        ctx.set_option("force_splits", 0)
    dm.close()
    pick = sorted(set(min(max(c, 0), C - 1) for c in (0, 1, 63, 64, C // 2, C - 65, C - 2, C - 1)))
    from concurrent.futures import ThreadPoolExecutor
    with ThreadPoolExecutor(max_workers=8) as ex:
        refs = list(ex.map(lambda c: om.evalallg(B[c]), pick))
    gs = np.abs(X).sum(0)
    for c, (olt, og) in zip(pick, refs):
        assert abs(lt[c] - olt) <= TOL * abs(olt), (name, c, lt[c], olt)
        assert np.all(np.abs(g[c] - og) <= TOL * gs), (name, c)
    assert np.all(np.isfinite(lt)) and np.all(np.isfinite(g))


def test_regression_chain_sharding_invariance(capi, ctx):
    """regression families: chain sharding reproduces the unsharded draws bit for bit when the row-split count is pinned
    (`force_splits`; the automatic choice depends on the shard's chain count and changes the summation order by ~1e-16)."""
    X, y, hy, b0 = make_regression("logistic", 3000, 12, 5)
    dm = capi.DeviceModel(ctx, "logistic", 12, X, y, hy)
    cfg = capi.sampler_cfg("HMC", scale=0.02, nleaps=5)
    ctx.set_option("force_splits", 4)
    try:
        outs = []
        for off, n in ((0, 200), (0, 72), (72, 128)):
            r = capi.DeviceRun(dm, cfg, (1, 1, 40), n, b0, seed=7, chain_offset=off, engine="wave"); r.execute(); outs.append(r.fetch()); r.close()
    finally:
        ctx.set_option("force_splits", 0)
    assert np.array_equal(outs[0]["samples"][:72], outs[1]["samples"]) and np.array_equal(outs[0]["samples"][72:], outs[2]["samples"])
    assert np.array_equal(outs[0]["accept"][72:], outs[2]["accept"])
    dm.close()


@pytest.mark.parametrize("kind,skw", [("HMC", dict(scale=0.75, nleaps=10)), ("RWM", dict(scale=0.5)), ("MALA", dict(scale=0.4))])
def test_streamed_summaries_match_the_two_pass_stats(capi, ctx, kind, skw):
    """stream_stats: the fused kernel keeps no draws and accumulates the summaries while sampling; same chains (same Philox
    keys) as a draw-storing run, whose src/stats pass is the reference: the mean bit for bit (same serial sum), the one-pass
    variances, batch-means variance, ESS and IAT to 1e-10, the acceptance rate exactly."""
    d, C, rngt = 3, 300, (101, 2, 1900)
    dm = capi.DeviceModel(ctx, "normal_fn", d)
    cfg = capi.sampler_cfg(kind, **skw)
    full = capi.DeviceRun(dm, cfg, rngt, C, np.ones(d), seed=21, chain_offset=5, engine="fused"); full.execute()
    ref = full.stats("bm", batchlen=50)
    st = capi.DeviceRun(dm, cfg, rngt, C, np.ones(d), seed=21, chain_offset=5, engine="fused", stream_stats=True, stream_batchlen=50); st.execute()
    out = st.stats("bm", batchlen=50)
    assert np.array_equal(out["mean"], ref["mean"]) and np.array_equal(out["accept_rate"], ref["accept_rate"])
    for k in ("var_iid", "var", "ess", "actime"):
        assert np.allclose(out[k], ref[k], rtol=1e-10, atol=0), k
    iid = st.stats("iid")
    assert np.allclose(iid["var"], ref["var_iid"], rtol=1e-10, atol=0)
    with pytest.raises(capi.MCMCGPUError):
        st.fetch()                                    # no draws were stored
    with pytest.raises(capi.MCMCGPUError):
        st.stats("imse")                              # the Geyer estimators need the draws
    with pytest.raises(capi.MCMCGPUError):
        capi.DeviceRun(dm, cfg, rngt, C, np.ones(d), engine="wave", stream_stats=True)
    full.close(); st.close(); dm.close()


@pytest.mark.parametrize("fam,d,N", [("normal_dsl", 20, 0), ("logistic", 40, 600), ("linear", 128, 500)])
def test_ram_large_d(O, capi, ctx, fam, d, N):
    """RAM beyond 16 parameters (RAM.jl:41-80 has no size limit): one CTA per chain, every matrix element summed by one
    thread in the reference's order -- same arithmetic as the one-thread kernel, so the same tolerance (pow's last bit)."""
    C, rngt = 12, (1, 1, 60)
    if N:
        X, y, hy, b0 = make_regression(fam, N, d, 9)
        init = b0
    else:
        X, y, hy, init = None, None, (0.5, 2.0), np.ones(d)
    out, diag, refs, _ = _run_both(O, capi, ctx, fam, d, X, y, hy, "RAM", dict(scale=0.02 if N else 1.0, rate=0.234), rngt, C, init, "wave")
    for c in range(C):
        assert np.array_equal(refs[c]["accept"], out["accept"][c]), c
        assert np.allclose(refs[c]["samples"], out["samples"][c], rtol=1e-8, atol=1e-11), c
        assert np.allclose(diag[0][c], refs[c]["eps"], rtol=1e-8), c
    assert 0 < out["accept"].mean() < 1
    with pytest.raises(capi.MCMCGPUError):
        capi.DeviceRun(capi.DeviceModel(ctx, "normal_dsl", 129, hyper=(0.0, 1.0)), capi.sampler_cfg("RAM", scale=1.0, rate=0.234), (1, 1, 5), 2, np.ones(129), engine="wave")


_FUSED = [("HMC", dict(scale=0.02, nleaps=5), (11, 1, 60)),
          ("HMC", dict(scale=0.02, nleaps=1), (1, 1, 40)),
          ("HMC", dict(scale=0.02, nleaps=3, tuner=dict(target_rate=0.8, adapt_step=10)), (31, 2, 70)),
          ("HMCDA", dict(len=0.1, max_leaps=64), (1, 1, 40)),
          ("MALA", dict(scale=0.001), (1, 1, 40))]


@pytest.mark.parametrize("fam", ["logistic", "probit", "linear"])
@pytest.mark.parametrize("kind,skw,rngt,d", [pytest.param(*c, 10, id=f"{c[0]}-skw{i}-rngt{i}") for i, c in enumerate(_FUSED)] +
                         # fixed-length HMC at one d per resident-CTA class and probit table copy (DK 4, 8, 9, 13, 14, 25)
                         [pytest.param(*_FUSED[0], d, id=f"HMC-skw0-rngt0-d{d}") for d in (29, 64, 71, 104, 112, 197)])
def test_unsplit_likelihood_fuses_the_leapfrog(O, capi, ctx, fam, kind, skw, rngt, d):
    """one row split (the launch-bound small-N regime; forced here): the likelihood kernel makes the interior leapfrog
    updates and advances the chains' counters itself, the transition kernel is skipped on those waves (fixed-length HMC)
    or ignores those chains (HMCDA, tuned HMC).  Draw-matched against the oracle, stepwise == one call, evaluation counts."""
    N, C = 700, 70
    X, y, hy, _ = make_regression(fam, N, d, 6)
    checked = range(C) if d == 10 else range(0, C, 5)   # oracle chains (CPU time grows with d)
    ctx.set_option("force_splits", 1)
    try:
        kw = dict(skw)
        if "scale" in kw and d != 10:            # HMC's energy error grows with d and with X'X's condition number
            kw["scale"] = kw["scale"] * math.sqrt(10 / d)
        if kind == "HMCDA":                      # realistic restored step sizes (the adaptation from eps = 1 is chaotic)
            rng = np.random.default_rng(1)
            eps = rng.uniform(0.01, 0.03, size=C)
            om = O.Model(fam, d, X, y, hy); dm = capi.DeviceModel(ctx, fam, d, X, y, hy)
            last = rngt[2]
            zn = rng.standard_normal((C, last + 1, d)); un = rng.random((C, last + 1))
            run = capi.DeviceRun(dm, capi.sampler_cfg(kind, **kw), rngt, C, np.zeros(d), normals=zn, uniforms=un, engine="wave")
            run.set_state(0, eps, eps, np.zeros(C))
            info = run.execute(); out = run.fetch(); geps, gnl = run.fetch_diag(); run.close(); dm.close()
            refs = [O.run_chain(om, O.sampler(kind, da_state=[eps[c], eps[c], 0.0], **kw), rngt, np.zeros(d), None, zn[c], un[c]) for c in range(C)]
            assert info["n_grad_evals"] == C + gnl.sum() and len(np.unique(gnl)) >= 3
        else:
            out, diag, refs, info = _run_both(O, capi, ctx, fam, d, X, y, hy, kind, kw, rngt, C, np.zeros(d), "wave", chains=checked)
            if kind == "HMC" and "tuner" not in kw:
                assert info["n_grad_evals"] == C * (1 + rngt[2] * kw["nleaps"])
                assert info["n_launches"] < 2 * info["n_waves"] or kw["nleaps"] == 1      # no transition launch on interior waves
        gs = np.abs(X).sum(0)
        for c in checked:
            assert np.array_equal(refs[c]["accept"], out["accept"][c]), (fam, kind, d, c)
            assert np.allclose(refs[c]["samples"], out["samples"][c], rtol=1e-9, atol=1e-12)
            assert np.allclose(refs[c]["logtarget"], out["logtarget"][c], rtol=1e-11, atol=0)
            assert np.all(np.abs(refs[c]["grads"] - out["grads"][c]) <= 1e-9 * gs)
        assert 0.2 < out["accept"].mean() <= 1.0
        if kind == "HMC" and "tuner" not in kw:   # stepwise execution (pauses between steps) gives the same chains
            dm = capi.DeviceModel(ctx, fam, d, X, y, hy)
            a = capi.DeviceRun(dm, capi.sampler_cfg(kind, **kw), rngt, C, np.zeros(d), seed=3, engine="wave"); a.execute(); fa = a.fetch()
            b = capi.DeviceRun(dm, capi.sampler_cfg(kind, **kw), rngt, C, np.zeros(d), seed=3, engine="wave")
            for n in (3, 1, 20, 100):
                b.execute_steps(n)
            fb = b.fetch()
            assert np.array_equal(fa["samples"], fb["samples"]) and np.array_equal(fa["accept"], fb["accept"])
            ctx.set_option("fuse_leap", 0)     # and the unfused path (transition kernel does the update) gives the same bits
            try:
                u = capi.DeviceRun(dm, capi.sampler_cfg(kind, **kw), rngt, C, np.zeros(d), seed=3, engine="wave"); u.execute(); fu = u.fetch(); u.close()
            finally:
                ctx.set_option("fuse_leap", 1)
            assert np.array_equal(fa["samples"], fu["samples"]) and np.array_equal(fa["accept"], fu["accept"])
            a.close(); b.close(); dm.close()
    finally:
        ctx.set_option("force_splits", 0)
