"""NUTS with the identity metric against NUTS with a diagonal metric adapted in Stan's windows, in one process: the card,
its power limit and two workloads.

  1. logistic regression, N = 1e5, d = 100, columns scaled by 10**linspace(0, 1.5, d), 4096 chains, W = 1000 warm-up
     steps (burn-in W + 1) and 200 kept steps, from eps = 1.  Per metric: gradient evaluations per post-warm-up step
     (mean leapfrogs per kept step), min-ESS per gradient evaluation and per second (tools/nuts_perf.py's measure: min
     over parameters of ESS(x) and ESS((x - mean)^2), Geyer IMSE, summed over chains; the evaluations and seconds are
     those of the whole run, warm-up included), and the adapted metric against the identity's posterior variance scale.
  2. the small-N shape (N = 256, d = 100, 94 720 chains) with time_eval on and a frozen step size: the time per wave
     outside the likelihood kernel and its split fold -- nuts_kernel plus launch gaps -- without a metric and with an
     all-ones metric, which makes the same trees, so the difference is the metric's cost in nuts_kernel.

usage: python tools/nuts_metric_perf.py [--out FILE] [--N 100000] [--chains 4096] [--warmup 1000] [--kept 200]
(prints one JSON object; smaller sizes are for quick looks and are reported as run)"""
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
from nuts_perf import card, logistic, min_ess  # noqa: E402


def workload1(ctx, N, C, W, K):
    d = 100
    X, y, b0 = logistic(N, d, 11)
    sc = 10.0 ** np.linspace(0, 1.5, d)
    X, b0 = X * sc, b0 / sc                                                 # the same linear predictor, badly scaled coordinates
    dm = capi.DeviceModel(ctx, "logistic", d, X, y, (1.0, -1.0))
    cfg = mj.NUTS()._cfg()
    warm = capi.DeviceRun(dm, cfg, (2, 1, 3), C, b0, seed=1, engine="wave", store_grad=False, store_logtarget=False)
    warm.execute(); warm.close()
    res = {}
    for name in ("identity", "adapted"):
        run = capi.DeviceRun(dm, cfg, (W + 2, 1, W + 1 + K), C, b0, seed=2, engine="wave", store_grad=False, store_logtarget=False)
        if name == "adapted":
            run.set_metric_adaptation(75, 50, 25)
        info = run.execute()
        s = info["gpu_ms"] / 1e3
        _, leaps = run.fetch_diag()
        ess, frac_bad = min_ess(ctx, run, K)
        minv = run.get_metric()
        res[name] = dict(seconds=s, grad_evals=info["n_grad_evals"], grad_evals_per_kept_step=float(leaps.mean()),
                         min_ess=ess, min_ess_per_grad_eval=ess / info["n_grad_evals"], min_ess_per_s=ess / s,
                         accept_rate=float(run.fetch(samples=False, grads=False)["accept"].mean()),
                         frac_series_without_ess=frac_bad, n_waves=info["n_waves"],
                         inv_metric_median_first_last=[float(np.median(minv[:, 0])), float(np.median(minv[:, -1]))])
        run.close()
    dm.close()
    ratio = res["identity"]["grad_evals_per_kept_step"] / res["adapted"]["grad_evals_per_kept_step"]
    return dict(N=N, d=d, column_scale="10**linspace(0, 1.5, d)", chains=C, warmup_W=W, kept=K,
                leapfrog_ratio_identity_over_adapted=ratio, **res)


def workload2(ctx):
    N, d, C = 256, 100, 94_720
    X, y, b0 = logistic(N, d, 12)
    dm = capi.DeviceModel(ctx, "logistic", d, X, y, (1.0, -1.0))
    cfg = mj.NUTS()._cfg()
    warm = capi.DeviceRun(dm, cfg, (2, 1, 3), C, b0, seed=1, engine="wave", store_grad=False, store_logtarget=False)
    warm.execute(); warm.close()
    res = {}
    for rep in range(2):                                                    # alternate the two, twice
        for name in ("no_metric", "ones_metric"):
            run = capi.DeviceRun(dm, cfg, (21, 1, 40), C, b0, seed=3, engine="wave", store_grad=False, store_logtarget=False)
            run.set_state(20, np.full(C, 0.02), np.full(C, 0.02), np.zeros(C))
            if name == "ones_metric":
                run.set_metric(np.ones(d))
            ctx.set_option("time_eval", 1)
            try:
                info = run.execute()
            finally:
                ctx.set_option("time_eval", 0)
            run.close()
            outside = (info["gpu_ms"] - info["eval_ms"] - info["comm_ms"]) / info["n_waves"]
            res.setdefault(name, []).append(dict(ms_per_wave=info["gpu_ms"] / info["n_waves"], outside_likelihood_ms_per_wave=outside,
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
    a = ap.parse_args()
    ctx = capi.Context(0)
    res = dict(card=card(), workload1=workload1(ctx, a.N, a.chains, a.warmup, a.kept), workload2=workload2(ctx))
    ctx.close()
    s = json.dumps(res, indent=1)
    print(s)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(s)


if __name__ == "__main__":
    main()
