"""NUTS with a diagonal metric against NUTS with a dense metric, both adapted in Stan's windows, in one process: the card,
its power limit and two workloads.

  1. logistic regression, N = 1e5, d = 50 and d = 100, features from a seeded equicorrelated (rho = 0.9) Gaussian design,
     4096 chains, W = 1000 warm-up steps (burn-in W + 1) and 200 kept steps, from eps = 1.  Per metric: leapfrogs per kept
     step, min-ESS per gradient evaluation and per second (tools/nuts_perf.py's measure over the whole run, warm-up
     included), the time per wave outside the likelihood kernel (time_eval: nuts_kernel, which makes the dense metric's two
     d^2 passes per leaf, plus launch gaps), and the adapted metric against the empirical covariance of the kept draws.
  2. the small-N shape (N = 256, d = 100, 94 720 chains) with time_eval on and a frozen step size: the time per wave
     outside the likelihood kernel with the diagonal metric, a dense metric shared by every chain and a dense metric per
     chain (the same identity matrix, so the trees are the same; the per-chain layout comes from the adaptation call,
     which has no window to adapt in here).

usage: python tools/nuts_dense_perf.py [--out FILE] [--N 100000] [--chains 4096] [--warmup 1000] [--kept 200]
       [--dims 50,100] [--small-chains 94720]
(prints one JSON object; --dims "" or --small-chains 0 leaves a workload out; smaller sizes are for quick looks and are
reported as run)"""
import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

import mcmc_jl_b200 as mj  # noqa: E402
from mcmc_jl_b200 import _capi as capi  # noqa: E402
from nuts_perf import card, min_ess  # noqa: E402


def equicorrelated_logistic(N, d, rho, seed):
    """intercept plus d - 1 features with unit variance and pairwise correlation rho"""
    r = np.random.default_rng(seed)
    Z = r.standard_normal((N, d - 1))
    F = np.sqrt(1.0 - rho) * Z + np.sqrt(rho) * r.standard_normal((N, 1))
    X = np.concatenate([np.ones((N, 1)), F], axis=1)
    b0 = r.standard_normal(d) / np.sqrt(d)
    y = (r.random(N) < 1 / (1 + np.exp(-X @ b0))).astype(float)
    return X, y, b0


def timed(ctx, run):
    ctx.set_option("time_eval", 1)
    try:
        info = run.execute()
    finally:
        ctx.set_option("time_eval", 0)
    info["outside_likelihood_ms_per_wave"] = (info["gpu_ms"] - info["eval_ms"] - info["comm_ms"]) / info["n_waves"]
    return info


def workload1(ctx, N, d, C, W, K):
    X, y, b0 = equicorrelated_logistic(N, d, 0.9, 11 + d)
    dm = capi.DeviceModel(ctx, "logistic", d, X, y, (1.0, -1.0))
    cfg = mj.NUTS()._cfg()
    warm = capi.DeviceRun(dm, cfg, (2, 1, 3), C, b0, seed=1, engine="wave", store_grad=False, store_logtarget=False)
    warm.execute(); warm.close()
    res = {}
    for name in ("diag", "dense"):
        run = capi.DeviceRun(dm, cfg, (W + 2, 1, W + 1 + K), C, b0, seed=2, engine="wave", store_grad=False, store_logtarget=False)
        if name == "dense":
            run.set_dense_metric(None)
        run.set_metric_adaptation(75, 50, 25)
        info = timed(ctx, run)
        s = info["gpu_ms"] / 1e3
        _, leaps = run.fetch_diag()
        ess, frac_bad = min_ess(ctx, run, K)
        x = run.fetch(grads=False, logtarget=False)["samples"]               # (C, K, d)
        emp = np.cov((x - x.mean(axis=1, keepdims=True)).reshape(-1, d).T)   # within-chain posterior covariance
        if name == "dense":
            A = np.median(run.get_dense_metric(), axis=0)
            met = dict(rel_frobenius_error_median_A=float(np.linalg.norm(A - emp) / np.linalg.norm(emp)))
        else:
            minv = np.median(run.get_metric(), axis=0)
            met = dict(rel_frobenius_error_median_A=float(np.linalg.norm(np.diag(minv) - emp) / np.linalg.norm(emp)))
        met["median_diag_ratio_A_over_empirical"] = float(np.median((np.diag(A) if name == "dense" else minv) / np.diag(emp)))
        res[name] = dict(seconds=s, grad_evals=info["n_grad_evals"], leapfrogs_per_kept_step=float(leaps.mean()),
                         min_ess=ess, min_ess_per_grad_eval=ess / info["n_grad_evals"], min_ess_per_s=ess / s,
                         frac_series_without_ess=frac_bad, n_waves=info["n_waves"], eval_ms=info["eval_ms"],
                         outside_likelihood_ms_per_wave=info["outside_likelihood_ms_per_wave"], **met)
        run.close()
    dm.close()
    return dict(N=N, d=d, rho=0.9, chains=C, warmup_W=W, kept=K,
                leapfrog_ratio_diag_over_dense=res["diag"]["leapfrogs_per_kept_step"] / res["dense"]["leapfrogs_per_kept_step"],
                **res)


def workload2(ctx, C):
    N, d = 256, 100
    X, y, b0 = equicorrelated_logistic(N, d, 0.0, 12)
    dm = capi.DeviceModel(ctx, "logistic", d, X, y, (1.0, -1.0))
    cfg = mj.NUTS()._cfg()
    warm = capi.DeviceRun(dm, cfg, (2, 1, 3), C, b0, seed=1, engine="wave", store_grad=False, store_logtarget=False)
    warm.execute(); warm.close()
    res = {}
    for rep in range(2):                                                    # alternate the three, twice
        for name in ("diag", "dense_shared", "dense_per_chain"):
            run = capi.DeviceRun(dm, cfg, (21, 1, 40), C, b0, seed=3, engine="wave", store_grad=False, store_logtarget=False)
            run.set_state(20, np.full(C, 0.02), np.full(C, 0.02), np.zeros(C))
            if name == "diag":
                run.set_metric(np.ones(d))
            else:
                run.set_dense_metric(None)
                if name == "dense_per_chain":
                    run.set_metric_adaptation()                             # W = 19 < 20: no window, per-chain matrices
            info = timed(ctx, run)
            run.close()
            res.setdefault(name, []).append(dict(ms_per_wave=info["gpu_ms"] / info["n_waves"],
                                                 outside_likelihood_ms_per_wave=info["outside_likelihood_ms_per_wave"],
                                                 n_waves=info["n_waves"]))
    dm.close()
    return dict(N=N, d=d, chains=C, steps=20, **res)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--N", type=int, default=100_000)
    ap.add_argument("--chains", type=int, default=4096)
    ap.add_argument("--warmup", type=int, default=1000)
    ap.add_argument("--kept", type=int, default=200)
    ap.add_argument("--dims", default="50,100")
    ap.add_argument("--small-chains", type=int, default=94_720)
    a = ap.parse_args()
    ctx = capi.Context(0)
    res = dict(card=card())
    if a.small_chains:
        res["workload2"] = workload2(ctx, a.small_chains)
    res["workload1"] = [workload1(ctx, a.N, int(d), a.chains, a.warmup, a.kept) for d in a.dims.split(",") if d]
    ctx.close()
    s = json.dumps(res, indent=1)
    print(s)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(s)


if __name__ == "__main__":
    main()
