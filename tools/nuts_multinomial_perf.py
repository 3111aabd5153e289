"""Slice NUTS against multinomial NUTS (Stan's transition) in one process, alternating them: the card, its power limit and
two workloads.

  1. the small-N shape (N = 256, d = 100, 94 720 chains) with time_eval on and a frozen step size: the time per wave
     outside the likelihood kernel (nuts_kernel plus launch gaps) with the identity metric, a diagonal metric and a dense
     metric shared by every chain, for each transition.
  2. logistic regression, N = 1e4, d = 50, features from a seeded equicorrelated (rho = 0.9) Gaussian design, 1024 chains,
     W = 1000 warm-up steps (burn-in W + 1) with a diagonal metric adapted in Stan's windows, and 200 kept steps, from
     eps = 1.  Per transition: leapfrogs per kept step, min-ESS per gradient evaluation and per second (tools/nuts_perf.py's
     measure over the whole run, warm-up included), and the number of divergent kept steps (multinomial only: slice NUTS
     does not report them).

usage: python tools/nuts_multinomial_perf.py [--out FILE] [--N 10000] [--d 50] [--chains 1024] [--warmup 1000] [--kept 200]
       [--small-chains 94720]
(prints one JSON object; --d 0 or --small-chains 0 leaves a workload out; smaller sizes are for quick looks and are
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
from nuts_dense_perf import equicorrelated_logistic, timed  # noqa: E402
from nuts_perf import card, min_ess  # noqa: E402

TRANSITIONS = (("slice", capi.NUTS_SLICE), ("multinomial", capi.NUTS_MULTINOMIAL))


def workload1(ctx, C):
    N, d = 256, 100
    X, y, b0 = equicorrelated_logistic(N, d, 0.0, 12)
    dm = capi.DeviceModel(ctx, "logistic", d, X, y, (1.0, -1.0))
    cfg = mj.NUTS()._cfg()
    warm = capi.DeviceRun(dm, cfg, (2, 1, 3), C, b0, seed=1, engine="wave", store_grad=False, store_logtarget=False)
    warm.execute(); warm.close()
    res = {}
    for rep in range(2):                                                    # alternate the transitions, twice
        for metric in ("unit", "diag", "dense_shared"):
            for tname, t in TRANSITIONS:
                run = capi.DeviceRun(dm, cfg, (21, 1, 40), C, b0, seed=3, engine="wave", store_grad=False, store_logtarget=False)
                run.set_nuts_transition(t)
                run.set_state(20, np.full(C, 0.02), np.full(C, 0.02), np.zeros(C))
                if metric == "diag":
                    run.set_metric(np.ones(d))
                elif metric == "dense_shared":
                    run.set_dense_metric(None)
                info = timed(ctx, run)
                _, leaps = run.fetch_diag()
                run.close()
                res.setdefault(f"{metric}_{tname}", []).append(dict(
                    ms_per_wave=info["gpu_ms"] / info["n_waves"], outside_likelihood_ms_per_wave=info["outside_likelihood_ms_per_wave"],
                    n_waves=info["n_waves"], leapfrogs_per_kept_step=float(leaps.mean())))
    dm.close()
    return dict(N=N, d=d, chains=C, steps=20, eps=0.02, **res)


def workload2(ctx, N, d, C, W, K):
    X, y, b0 = equicorrelated_logistic(N, d, 0.9, 11 + d)
    dm = capi.DeviceModel(ctx, "logistic", d, X, y, (1.0, -1.0))
    cfg = mj.NUTS()._cfg()
    warm = capi.DeviceRun(dm, cfg, (2, 1, 3), C, b0, seed=1, engine="wave", store_grad=False, store_logtarget=False)
    warm.execute(); warm.close()
    res = {}
    for tname, t in TRANSITIONS:
        run = capi.DeviceRun(dm, cfg, (W + 2, 1, W + 1 + K), C, b0, seed=2, engine="wave", store_grad=False, store_logtarget=False)
        run.set_nuts_transition(t)
        run.set_metric_adaptation(75, 50, 25)
        info = run.execute()
        s = info["gpu_ms"] / 1e3
        _, leaps = run.fetch_diag()
        ess, frac_bad = min_ess(ctx, run, K)
        r = dict(seconds=s, grad_evals=info["n_grad_evals"], leapfrogs_per_kept_step=float(leaps.mean()), min_ess=ess,
                 min_ess_per_grad_eval=ess / info["n_grad_evals"], min_ess_per_s=ess / s, frac_series_without_ess=frac_bad,
                 n_waves=info["n_waves"])
        if t == capi.NUTS_MULTINOMIAL:
            st = run.fetch_nuts_stats()
            r.update(divergent_kept_steps=int(st["divergent"].sum()), mean_accept_stat=float(st["accept_stat"].mean()))
        res[tname] = r
        run.close()
    dm.close()
    return dict(N=N, d=d, rho=0.9, chains=C, warmup_W=W, kept=K, metric="diag, adapted", **res)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--N", type=int, default=10_000)
    ap.add_argument("--d", type=int, default=50)
    ap.add_argument("--chains", type=int, default=1024)
    ap.add_argument("--warmup", type=int, default=1000)
    ap.add_argument("--kept", type=int, default=200)
    ap.add_argument("--small-chains", type=int, default=94_720)
    a = ap.parse_args()
    ctx = capi.Context(0)
    res = dict(card=card())
    if a.small_chains:
        res["workload1"] = workload1(ctx, a.small_chains)
    if a.d:
        res["workload2"] = workload2(ctx, a.N, a.d, a.chains, a.warmup, a.kept)
    ctx.close()
    s = json.dumps(res, indent=1)
    print(s)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(s)


if __name__ == "__main__":
    main()
