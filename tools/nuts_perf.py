"""NUTS against HMCDA on the wave engine, in one process: the card, its power limit and two workloads.

  1. logistic regression, N = 1e5, d = 100, 4096 chains, 600 steps of which 300 burn-in: HMCDA as bench.py runs it
     (len = CFG4_LEN, max_leaps = 64) and NUTS with its defaults, each from eps = 1 with its own dual averaging.  Per
     sampler: gradient evaluations/s, chain-steps/s, mean leapfrogs per kept step, min-ESS/s and min-ESS per gradient
     evaluation (min over parameters of ESS(x) and ESS((x - mean)^2), Geyer IMSE, summed over chains; bench.py's measure).
  2. the small-N shape (N = 256, d = 100, 94 720 chains) with time_eval on: the share of the wave time outside the
     likelihood kernel and its split fold, i.e. the NUTS kernel plus launch gaps.

usage: python tools/nuts_perf.py [--out FILE]   (prints one JSON object)"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from bench import CFG4_LEN  # noqa: E402
import mcmc_jl_b200 as mj  # noqa: E402
from mcmc_jl_b200 import _capi as capi  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True, check=True).stdout.strip().splitlines()[0]
    name, plimit, clk = [s.strip() for s in q.split(",")]
    return dict(name=name, power_limit=plimit, max_sm_clock=clk)


def logistic(N, d, seed):
    r = np.random.default_rng(seed)
    X = np.concatenate([np.ones((N, 1)), r.standard_normal((N, d - 1))], axis=1)
    b0 = r.standard_normal(d) / np.sqrt(d)
    y = (r.random(N) < 1 / (1 + np.exp(-X @ b0))).astype(float)
    return X, y, b0


def min_ess(ctx, run, keep):
    ex = run.stats("imse")["ess"]
    x = run.fetch(grads=False, logtarget=False)["samples"]
    e2 = ctx.stats((x - x.mean(axis=1, keepdims=True)) ** 2, "imse", want=("ess",))["ess"]
    comb = np.fmin(np.where(ex > 0, ex, np.nan), np.where(e2 > 0, e2, np.nan))
    return float(np.nansum(np.nanmin(comb, axis=1))), float(np.mean(np.isnan(comb)))


def workload1(ctx):
    N, d, C, B, L = 100_000, 100, 4096, 300, 600
    X, y, b0 = logistic(N, d, 11)
    dm = capi.DeviceModel(ctx, "logistic", d, X, y, (1.0, -1.0))
    res = {}
    for name, cfg in (("HMCDA", capi.sampler_cfg("HMCDA", len=CFG4_LEN, max_leaps=64)), ("NUTS", mj.NUTS()._cfg())):
        warm = capi.DeviceRun(dm, cfg, (2, 1, 3), C, b0, seed=1, engine="wave", store_grad=False, store_logtarget=False)
        warm.execute(); warm.close()
        run = capi.DeviceRun(dm, cfg, (B + 1, 1, L), C, b0, seed=2, engine="wave", store_grad=False, store_logtarget=False)
        info = run.execute()
        s = info["gpu_ms"] / 1e3
        eps, leaps = run.fetch_diag()
        ess, frac_bad = min_ess(ctx, run, L - B)
        res[name] = dict(seconds=s, grad_evals_per_s=info["n_grad_evals"] / s, chain_steps_per_s=C * L / s,
                         mean_leaps_per_kept_step=float(leaps.mean()), accept_rate=float(run.fetch(samples=False, grads=False)["accept"].mean()),
                         final_eps_median=float(np.median(eps[:, -1])), min_ess_per_s=ess / s,
                         min_ess_per_grad_eval=ess / info["n_grad_evals"], frac_series_without_ess=frac_bad, n_waves=info["n_waves"])
        run.close()
    dm.close()
    return dict(N=N, d=d, chains=C, steps=L, burnin=B, **res)


def workload2(ctx):
    N, d, C = 256, 100, 94_720
    X, y, b0 = logistic(N, d, 12)
    dm = capi.DeviceModel(ctx, "logistic", d, X, y, (1.0, -1.0))
    cfg = mj.NUTS()._cfg()
    warm = capi.DeviceRun(dm, cfg, (2, 1, 3), C, b0, seed=1, engine="wave", store_grad=False, store_logtarget=False)
    warm.execute(); warm.close()
    # a realistic step size for this posterior (sd ~ 1 / sqrt(N)), frozen: every wave is a leaf of a real tree
    run = capi.DeviceRun(dm, cfg, (21, 1, 40), C, b0, seed=3, engine="wave", store_grad=False, store_logtarget=False)
    run.set_state(20, np.full(C, 0.02), np.full(C, 0.02), np.zeros(C))
    ctx.set_option("time_eval", 1)
    try:
        info = run.execute()
    finally:
        ctx.set_option("time_eval", 0)
    _, leaps = run.fetch_diag()
    run.close(); dm.close()
    share = 1.0 - (info["eval_ms"] + info["comm_ms"]) / info["gpu_ms"]
    return dict(N=N, d=d, chains=C, steps=20, gpu_ms=info["gpu_ms"], eval_ms=info["eval_ms"], fold_ms=info["comm_ms"],
                n_waves=info["n_waves"], ms_per_wave=info["gpu_ms"] / info["n_waves"], mean_leaps_per_step=float(leaps.mean()),
                share_outside_likelihood=share, nuts_state_bytes_per_chain_per_wave_est=12 * d * 8)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    ctx = capi.Context(0)
    res = dict(card=card(), workload1=workload1(ctx), workload2=workload2(ctx))
    ctx.close()
    s = json.dumps(res, indent=1)
    print(s)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(s)


if __name__ == "__main__":
    main()
