#!/usr/bin/env python
"""bench.py -- the measurement contract of this repo.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload cfg4|cfg2|cfg3|cfg5|smallN] [--impl reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N --steps K --warmup W

One JSON line on rank 0.  A "step" is one MCMC step of every chain (one pass of the hot path over the batch); the headline
leg times exactly --steps of them, and `observed.grad_evals_per_chain_step` is the device's count of gradient evaluations
in that timed run over chains x steps.
--dump-outputs DIR writes what the timed run of the headline leg computed in its last step (rank 0's chains) as float64
.npy files, so that two builds can be compared output for output: the inputs depend only on the arguments.

Headline workload (BASELINE.json `metric` "chain-steps/s ..., HMC logistic regression", configs[3]):
  cfg4  HMCDA logistic regression, synthetic N = 1e6, d = 100 (X = [1, N(0,1)], beta0 ~ N(0,1)/sqrt(d), seed 4),
        10 000 chains per GPU (chain-sharded: no collective; weak scaling), sampling phase of HMCDA: the
        dual-averaged step size found by the pilot adaptation (tools/pilot_adapt.py, profiles/pilot_cfg4_r01.json)
        is restored with mcmcgpu_run_set_state, len = 0.02 => nLeaps = round(len/eps) = 10 leapfrogs per step.

Keys of the line (headline leg):
`value`      device-timed (CUDA events on the launching stream, barrier + synchronize on both sides, max over
             ranks), inputs resident in HBM.
`e2e`        the same K steps through the C-ABI run call with HOST buffers: H2D of the chain state, execute,
             D2H of the kept draws / gradients / accept flags / log-targets into pinned host memory.
`roofline`   the likelihood kernel K1 against the FP64 tensor (DMMA) roofline: algorithmic 4*N*d flop per chain
             per evaluation, peak = cuBLAS FP64 GEMM measured live (MEASURED_PEAKS.json has no FP64 entry).
`cpu_baseline` the oracle (CPU restatement of the reference, the reference itself being Julia 0.2 source that
             cannot run here) timed on the host cores on a bounded sample of the same workload: all cores (one chain
             per thread, the `prun` analogue) and `one_core` (SerialMC itself is single-threaded).  N = 1 only.
`min_ess_per_s`  min-ESS/s (the second half of BASELINE's metric): Geyer-IMSE ESS (src/stats/ess.jl) of x AND of
             (x - mean)^2 per (chain, parameter) series from a pilot of the same chains; raw fractions of degenerate
             estimates; a sweep over the trajectory length `len` with the best one timed as well.
Sub-blocks of the default (cfg4) run, each a driver-timed number for another BASELINE config:
`configs`    cfg3 (MALA probit N=1e5 d=20, 16 384 chains/GPU), cfg2 (HMC(0.75) 3-D Normal, 65 536 chains/GPU, fused
             per-chain kernel), smallN (HMC logistic N=256 d=100, 94 720 chains/GPU: the launch-bound regime in which
             the north star's 1e9 gradient evaluations/s is arithmetically reachable).
`row_sharded` cfg5: tall data (6.25e6 rows x d=200 per GPU; 5e7 rows at 8 GPUs), chains replicated, one NCCL all-reduce
             of the (d+2) x C partials per leapfrog; K1 ms/launch and fold+all-reduce ms/leapfrog from CUDA events; at
             N > 1 a sharded-vs-unsharded parity check runs first (`parity`).
`strong`     (N > 1) cfg4 with 10 000 chains in TOTAL, chain-sharded: strong scaling of the headline.
`population` (N > 1) SeqMC over regression models sharded over the GPUs (ncclAllGather per target) and SerialTempMC replicas sharded by
             replica id, each checked against the single-GPU run of the same population (`*_sharded_parity`).
"""
import argparse
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

# dual-averaged HMCDA step size after burn-in on cfg4 (median over 512 pilot chains; profiles/pilot_cfg4_r01.json)
CFG4_EPS = 1.97e-3
CFG4_LEN = 0.02
ESS_SWEEP_LENS = (0.02, 0.008, 0.004)      # HMCDA trajectory lengths tried for min-ESS per gradient (10 / 4 / 2 leapfrogs)
DUMP_BYTES = 64 * 10 ** 6 - 4096            # --dump-outputs writes at most 64 MB, .npy headers included


def synth_logistic(N, d, seed):
    """SURVEY.md 8d: X = [1, N(0,1)^(d-1)], beta0 ~ N(0,1)/sqrt(d), y ~ Bernoulli(sigmoid(X beta0)). Column-major X."""
    r = np.random.default_rng(seed)
    Xt = np.empty((d, N))
    Xt[0] = 1.0
    for j in range(1, d):
        Xt[j] = r.standard_normal(N)
    b0 = r.standard_normal(d) / np.sqrt(d)
    eta = b0 @ Xt
    y = (r.random(N) < 1.0 / (1.0 + np.exp(-eta))).astype(np.float64)
    return Xt.T, y, b0          # Xt.T is an F-ordered N x d view


def synth_probit(N, d, seed):
    from scipy.special import ndtr
    r = np.random.default_rng(seed)
    Xt = np.empty((d, N))
    Xt[0] = 1.0
    for j in range(1, d):
        Xt[j] = r.standard_normal(N)
    b0 = 0.5 * r.standard_normal(d)
    y = (r.random(N) < ndtr(b0 @ Xt)).astype(np.float64)
    return Xt.T, y, b0


WORKLOADS = {
    "cfg4": dict(desc="HMCDA logistic regression N=1e6 d=100, 10000 chains/GPU (BASELINE configs[3])", family="logistic",
                 N=1000000, d=100, chains=10000, sampler="HMCDA", seed=4),
    "cfg3": dict(desc="MALA probit regression N=1e5 d=20, 16384 chains/GPU (BASELINE configs[2])", family="probit",
                 N=100000, d=20, chains=16384, sampler="MALA", seed=3),
    "cfg5": dict(desc="HMC logistic regression, tall data d=200, rows sharded over the GPUs (6.25e6 rows per GPU; 5e7 at 8 GPUs), "
                      "256 replicated chains, NCCL all-reduce of (d+2) x C partials per leapfrog (BASELINE configs[4])",
                 family="logistic", N=6250000, d=200, chains=256, sampler="HMC", seed=5),
    "cfg2": dict(desc="HMC(0.75) 3-D Normal -dot(v,v), 65536 chains/GPU (BASELINE configs[1])", family="normal_fn",
                 N=0, d=3, chains=65536, sampler="HMC", seed=1, steps=1000),
    "smallN": dict(desc="HMC (8 leapfrogs) logistic regression N=256 d=100, 94720 chains/GPU (5 full waves of 296 resident 64-chain CTAs): launch-bound small-N regime "
                        "(SURVEY 8d: 1e9 gradient evaluations/s is reachable only for N <~ 740)", family="logistic",
                   N=256, d=100, chains=94720, sampler="HMC", seed=6, nleaps=8, eps=0.1, steps=20),
}
# default --steps where a workload has none above: one MCMC step of cfg2 is ~2 us of device work and one of smallN ~3.4 ms, so
# they time more steps by default to make the timed window long enough
DEFAULT_STEPS = 5


def config_block(name, wl, world):
    """the `config` object: the same keys and values in the native and the reference arm (the driver compares them)"""
    d, row = wl["d"], name == "cfg5"
    return dict(workload=name, description=wl["desc"], N=wl["N"], d=d, chains_per_gpu=wl["chains"], sampler=wl["sampler"],
                parallelism=(f"rows sharded over {world} GPU(s) ({wl['N']} rows each), chains replicated, ncclAllReduce per leapfrog"
                             if row else f"chains sharded over {world} GPU(s), no collective"),
                l2=("inputs larger than L2 (packed X = %.0f MB)" % (wl["N"] * (8 * ((d + 7) // 8) + 4) * 8 / 1e6)) if wl["N"] * d * 8 > 126e6
                else ("no input data; kept draws written once" if not wl["N"] else "X is L2-resident (%.1f MB); chain state streams through HBM" % (wl["N"] * d * 8 / 1e6)),
                seed=wl["seed"], eps=CFG4_EPS if wl["sampler"] == "HMCDA" else None, len=CFG4_LEN if wl["sampler"] == "HMCDA" else None)


class ClockSampler:
    """samples SM clock and throttle reasons during the timed region (NVML)"""

    def __init__(self, index):
        self.samples, self.reasons, self.max_mhz, self._stop = [], set(), None, threading.Event()
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None
        self.t = threading.Thread(target=self._loop, daemon=True)

    def _loop(self):
        nv = self.nv
        names = {"hw_slowdown": 0x8, "sw_power_cap": 0x4, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20,
                 "hw_power_brake_slowdown": 0x80}
        while not self._stop.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h) if hasattr(nv, "nvmlDeviceGetCurrentClocksEventReasons") \
                    else nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for k, bit in names.items():
                    if r & bit:
                        self.reasons.add(k)
            except Exception:
                pass
            self._stop.wait(0.1)

    def __enter__(self):
        if self.nv:
            self.t.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        if self.nv:
            self.t.join(timeout=2)

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons)}
        return {"sm_mhz": float(np.median(self.samples)), "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons)}


def dgemm_peak_tflops(torch, n=8192, reps=5):
    a = torch.randn(n, n, device="cuda", dtype=torch.float64)
    b = torch.randn(n, n, device="cuda", dtype=torch.float64)
    c = torch.empty_like(a)
    for _ in range(2):
        torch.matmul(a, b, out=c)
    torch.cuda.synchronize()
    best = 1e30
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); torch.matmul(a, b, out=c); e1.record(); torch.cuda.synchronize()
        best = min(best, e0.elapsed_time(e1))
    del a, b, c
    torch.cuda.empty_cache()
    return 2.0 * n ** 3 / best / 1e9


def dump_last_step(out_dir, res):
    """--dump-outputs: the arrays fetch() returns for a run, at its last step (samples / grads (C, d), logtarget / accept (C,)).
    When they exceed DUMP_BYTES, a fixed, seeded sample of chains is written; chain_index.npy lists the chains written."""
    last = {k: np.asarray(v[:, -1], dtype=np.float64) for k, v in res.items()}
    C = len(last["accept"])
    per_chain = 8 * (1 + sum(v[0].size for v in last.values()))
    idx = np.arange(C)
    if C * per_chain > DUMP_BYTES:
        idx = np.sort(np.random.default_rng(0).choice(C, DUMP_BYTES // per_chain, replace=False))
    out = {k: v[idx] for k, v in last.items()}
    out["chain_index"] = idx.astype(np.float64)
    os.makedirs(out_dir, exist_ok=True)
    for k, v in out.items():
        np.save(os.path.join(out_dir, k + ".npy"), v)


def make_problem(wl):
    if wl["family"] == "logistic":
        X, y, b0 = synth_logistic(wl["N"], wl["d"], wl["seed"])
        return X, y, (1.0, -1.0), b0
    if wl["family"] == "probit":
        X, y, b0 = synth_probit(wl["N"], wl["d"], wl["seed"])
        return X, y, (10.0,), b0
    return None, None, (), np.ones(wl["d"])


def sampler_for(wl, capi_or_oracle, is_oracle=False, force_eps=None, len_=None):
    mk = capi_or_oracle.sampler if is_oracle else capi_or_oracle.sampler_cfg
    if wl["sampler"] == "HMCDA":
        kw = dict(len=CFG4_LEN if len_ is None else len_, max_leaps=64)
        if is_oracle:
            kw["force_eps"] = force_eps
        return mk("HMCDA", **kw)
    if wl["sampler"] == "MALA":
        return mk("MALA", scale=wl.get("drift", 2.4 ** 2 * wl["d"] ** (-1.0 / 3.0) / wl["N"]))
    if "nleaps" in wl:                      # smallN
        return mk("HMC", scale=wl["eps"], nleaps=wl["nleaps"])
    if wl["family"] == "logistic":          # cfg5: step size scaled from the cfg4 pilot by sqrt(N) and d^(1/4)
        ntot = wl["N"] * int(os.environ.get("WORLD_SIZE", "1"))
        return mk("HMC", scale=0.8 * CFG4_EPS * (1e6 / ntot) ** 0.5 * (100.0 / wl["d"]) ** 0.25, nleaps=10)
    return mk("HMC", scale=0.75, nleaps=10)


# ----------------------------------------------------------------------------------------------------------------
def cpu_baseline(wl, steps, warmup, cores, problem=None):
    """oracle ("port") on `cores` host threads, one independent chain per thread (the prun analogue,
    runners.jl:35-42); ctypes releases the GIL so the threads run in parallel."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import oracle as O
    X, y, hy, b0 = problem if problem is not None else make_problem(wl)
    d = wl["d"]
    # the CPU legs time the stronger shape of the restatement: row-blocked (X read from DRAM once per evaluation), 4 partial sums
    # per dot product, AVX2 / AVX-512 clones -- what an optimised dgemv does; the parity oracle itself keeps the serial sums
    O.set_fast_baseline(True)
    om = O.Model(wl["family"], d, X, y, hy)
    init = b0 if wl["family"] != "normal_fn" else np.ones(d)
    states = [init.copy() for _ in range(cores)]

    def chain_steps(k, nsteps, state):
        rng = np.random.default_rng(1000 + k)
        zn = rng.standard_normal((nsteps + 1, d)); un = rng.random(nsteps + 1)
        fe = np.full(nsteps + 1, CFG4_EPS) if wl["sampler"] == "HMCDA" else None
        res = O.run_chain(om, sampler_for(wl, O, True, fe), (1, 1, nsteps), state, None, zn, un)
        return res["samples"][-1], res["n_grad_evals"]

    def work(k, nsteps, out):
        out[k] = chain_steps(k, nsteps, states[k])

    def run_all(nsteps):
        out = [None] * cores
        ts = [threading.Thread(target=work, args=(k, nsteps, out)) for k in range(cores)]
        t0 = time.perf_counter()
        for t in ts:
            t.start()
        for t in ts:
            t.join()
        dt = time.perf_counter() - t0
        for k in range(cores):
            states[k] = out[k][0]
        return dt, sum(o[1] for o in out)

    if warmup > 0:
        run_all(warmup)
    dt, nev = run_all(steps)
    O.set_fast_baseline(False)
    return dict(value=cores * steps / dt, unit="chain-steps/s", cores=cores, kind="port",
                sample=f"{cores} chain(s) x {steps} steps (1 chain per host thread) of the {wl['chains']}-chain workload, full N",
                grad_evals_per_s=nev / dt, seconds=dt)


def run_reference_arm(args, wl, wl_name):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    world = int(os.environ.get("WORLD_SIZE", "1"))
    cores = os.cpu_count() or 1
    cb = cpu_baseline(wl, args.steps, args.warmup, cores)
    cfg = config_block(wl_name, wl, world)
    line = dict(metric="chain-steps/s", value=cb["value"], unit="chain-steps/s", n_gpus=args.gpus, steps=args.steps,
                warmup=args.warmup, ms_per_step=1e3 * cb["seconds"] / args.steps, higher_is_better=True, scaling="weak",
                vs_baseline=None, dtype="f64", data="synthetic", impl="reference", config=cfg,
                note="reference = CPU oracle (C restatement of MCMC.jl; the Julia 0.2 reference cannot run here), all host threads, "
                     "one chain per thread (the prun analogue); each step is one MCMC step of `cores` chains of the configured workload",
                cpu_baseline=dict(value=cb["value"], unit="chain-steps/s", cores=cores, kind="port", sample=cb["sample"]),
                e2e=dict(value=cb["value"], unit="chain-steps/s", h2d_bytes_per_step=0, d2h_bytes_per_step=0),
                grad_evals_per_s=cb["grad_evals_per_s"], gpu_launches=0)
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------------------------------------------
class Bench:
    """state shared by the legs of the native arm"""

    def __init__(self, args):
        import torch
        import torch.distributed as dist
        import mcmc_jl_b200
        from mcmc_jl_b200 import _capi as capi
        self.torch, self.dist, self.capi, self.mj, self.args = torch, dist, capi, mcmc_jl_b200, args
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        torch.cuda.set_device(self.local)
        if self.world > 1:
            dist.init_process_group("nccl", device_id=torch.device("cuda", self.local))
        self.ctx = capi.Context(self.local)
        self.stream = torch.cuda.current_stream()
        self.ctx.set_stream(self.stream.cuda_stream)      # library launches on torch's stream so torch events bracket them
        self.ctx.set_option("time_eval", 1)
        self.peak = None
        self.comm_ready = False

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max_over_ranks(self, *vals):
        t = self.torch.tensor(list(vals), dtype=self.torch.float64, device="cuda")
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return t.tolist()

    def sum_over_ranks(self, *vals):
        t = self.torch.tensor(list(vals), dtype=self.torch.float64, device="cuda")
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.SUM)
        return t.tolist()

    def pin(self, shape, dt=np.float64):
        torch = self.torch
        return torch.empty(shape, dtype={np.float64: torch.float64, np.uint8: torch.uint8}[dt]).pin_memory().numpy()

    def fp64_peak(self):
        if self.peak is None:
            self.peak = dgemm_peak_tflops(self.torch)
        return self.peak

    def dump_run(self, r):
        """--dump-outputs (rank 0): the last step of a timed run that has finished.  The C ABI returns a run's outputs only whole,
        so every kept step of the samples and gradients crosses to the host here, once, after the timed region: 1.2 GB for
        the smallN headline and 3.7 GB for cfg2 at their default --steps (as much as the e2e leg's pinned buffers)."""
        if self.args.dump_outputs and self.rank == 0:
            dump_last_step(self.args.dump_outputs, r.fetch(samples=True, grads=True, logtarget=True))

    # ---- one wave-engine leg: W warm-up steps, K timed steps of the same chains; returns device ms (this rank) ----
    def wave_leg(self, dm, scfg, C, d, init_state, K, W, seed, offset, set_state=None, clock=False, time_eval=True, dump=False):
        """time_eval: CUDA events around every likelihood launch (run_info.eval_ms / comm_ms); the engine then launches every
        wave on the stream.  Without it the wave loop of the launch-bound workloads is replayed from a CUDA graph.
        dump: this is the headline leg, whose last step goes to --dump-outputs (after the timed region, see dump_run)."""
        capi, torch = self.capi, self.torch
        self.ctx.set_option("time_eval", 1 if time_eval else 0)
        step0 = set_state[0] if set_state else 0
        r = capi.DeviceRun(dm, scfg, (step0 + 1, 1, step0 + W + K), C, init_state, seed=seed, chain_offset=offset, engine="wave")
        if set_state:
            r.set_state(*set_state)
        r.execute_steps(W)
        self.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        clk = ClockSampler(self.local) if clock else None
        if clk:
            clk.__enter__()
        e0.record(self.stream); info = r.execute_steps(K); e1.record(self.stream)
        self.barrier()
        if clk:
            clk.__exit__()
        ms = e0.elapsed_time(e1)
        acc = float(r.fetch(samples=False, grads=False, logtarget=False)["accept"][:, W:].mean())
        if dump:
            self.dump_run(r)
        r.close()
        return ms, info, acc, (clk.summary() if clk else None)

    def e2e_leg(self, dm, scfg, C, d, init_state, K, seed, offset, set_state=None, engine="wave"):
        """the same K steps through the C-ABI run with HOST buffers (pinned): H2D + execute + D2H inside the timed region"""
        capi, torch = self.capi, self.torch
        step0 = set_state[0] if set_state else 0
        bufs = dict(samples=self.pin((C, K, d)), grads=self.pin((C, K, d)), accept=self.pin((C, K), np.uint8), logtarget=self.pin((C, K)))
        self.barrier()
        t0 = time.perf_counter()
        r = capi.DeviceRun(dm, scfg, (step0 + 1, 1, step0 + K), C, init_state, seed=seed, chain_offset=offset, engine=engine)
        if set_state:
            r.set_state(*set_state)
        r.execute()
        r.fetch(out=bufs)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        r.close()
        h2d = (C * d * 8 if np.ndim(init_state) == 2 else d * 8) + (3 * C * 8 if set_state and len(set_state) > 1 else 0)
        d2h = C * K * d * 8 * 2 + C * K + C * K * 8
        return dt, h2d, d2h

    def k1_roofline(self, wl, C, info, ms, traffic=None):
        per = info["eval_ms"] / max(info["n_waves"], 1)
        flop = 4.0 * wl["N"] * wl["d"] * C
        ach = flop / per / 1e9
        peak = self.fp64_peak()
        return dict(bound="tensor", achieved=ach, peak=peak, unit="TFLOP/s", frac=ach / peak, traffic=traffic,
                    kernel="k1_kernel (FP64 DMMA m8n8k4)", ms_per_launch=per, share_of_step=info["eval_ms"] / ms,
                    peak_source="cuBLAS FP64 GEMM 8192^3 measured live in this run (MEASURED_PEAKS.json has no FP64 entry)")


def headline_state(wl, C, b0, rank):
    """synthetic start of the timed chains: around the generating beta0; HMCDA in its sampling phase (step size restored)"""
    rng = np.random.default_rng(100 + rank)
    d = wl["d"]
    if wl["sampler"] == "HMCDA":
        init = b0[None, :] + 2e-3 * rng.standard_normal((C, d))
        return init, (1000, np.full(C, CFG4_EPS), np.full(C, CFG4_EPS), np.zeros(C))
    if wl["family"] == "normal_fn":
        return np.ones(d), None
    scale = 1e-3 if wl["N"] >= 10000 else 0.05
    return b0[None, :] + scale * np.random.default_rng(100).standard_normal((C, d)), None      # same on every rank


def ess_pilot(B, dm, wl, init_state, set_state, offset, lens, ce=256, keep=400, skip=30):
    """ESS per chain-step from a pilot of the same chains: Geyer IMSE (ess.jl:6-10) of x on the device-resident draws and
    of (x - mean)^2 (an antithetic chain scores ESS_x >= n while its squares mix slowly).  No clipping: degenerate
    estimates are counted, not replaced."""
    capi = B.capi
    d, out = wl["d"], []
    step0 = set_state[0] if set_state else 0
    for L in lens:
        scfg = sampler_for(wl, capi, len_=L)
        r0 = capi.DeviceRun(dm, scfg, (step0 + 1, 1, step0 + skip), ce, init_state[:ce] if np.ndim(init_state) == 2 else init_state,
                            seed=wl["seed"] + 7, chain_offset=offset, engine="wave", store_grad=False, store_logtarget=False)
        if set_state:
            r0.set_state(set_state[0], *(a[:ce] for a in set_state[1:]))
        r0.execute()
        st0 = r0.get_state()
        r0.close()
        # the kept range starts right after the hand-over step, so HMCDA's burn-in adaptation (i < first - 1) stays off
        rr = capi.DeviceRun(dm, scfg, (step0 + skip + 1, 1, step0 + skip + keep), ce, st0["pars"], seed=wl["seed"] + 7, chain_offset=offset,
                            engine="wave", store_grad=False, store_logtarget=False)
        if set_state:
            rr.set_state(step0 + skip, st0["leapstep"], st0["dual_leapstep"], st0["dualH"])
        else:
            rr.set_state(step0 + skip)
        info = rr.execute()
        st = rr.stats("imse")
        x = rr.fetch(grads=False, logtarget=False)
        rr.close()
        ex = st["ess"]                                          # (ce, d), raw
        sq = (x["samples"] - x["samples"].mean(axis=1, keepdims=True)) ** 2
        e2 = B.ctx.stats(sq, "imse", want=("ess",))["ess"]
        ok_x = np.isfinite(ex) & (ex > 0)
        ok_2 = np.isfinite(e2) & (e2 > 0)
        comb = np.where(ok_x & ok_2, np.minimum(ex, e2), np.where(ok_2, e2, np.where(ok_x, ex, np.nan)))
        per_chain = np.nanmin(comb, axis=1) / keep
        out.append(dict(len=L, nleaps=float(info["n_grad_evals"]) / (ce * keep), accept=float(x["accept"].mean()),
                        ess_per_chain_step=float(np.nanmedian(per_chain)),
                        median_min_ess_x_per_step=float(np.median(np.min(np.where(np.isnan(ex), -np.inf, ex), axis=1)) / keep),
                        median_min_ess_x2_per_step=float(np.median(np.min(np.where(np.isnan(e2), -np.inf, e2), axis=1)) / keep),
                        frac_x_nonpositive=float(np.mean(ex <= 0)), frac_x_ge_n=float(np.mean(ex >= keep)), frac_x_nan=float(np.mean(np.isnan(ex))),
                        frac_x2_nonpositive=float(np.mean(e2 <= 0)), frac_x2_ge_n=float(np.mean(e2 >= keep)), frac_x2_nan=float(np.mean(np.isnan(e2)))))
        out[-1]["min_ess_per_grad"] = out[-1]["ess_per_chain_step"] / out[-1]["nleaps"]
    return out, f"{ce} chains x {keep} kept steps after {skip} discarded, Geyer IMSE on the device; per chain: min over parameters of min(ESS(x), ESS((x-mean)^2)); median over chains; no clipping"


# ----------------------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None, help="timed MCMC steps (default: 1000 for cfg2, 20 for smallN, else 5)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--workload", default="cfg4", choices=sorted(WORKLOADS))
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--chains", type=int, default=0, help="override chains per GPU")
    ap.add_argument("--N", type=int, default=0, help="override observation count")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-ess", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="headline leg only (no configs / row_sharded / strong sub-blocks)")
    ap.add_argument("--cpu-steps", type=int, default=2)
    ap.add_argument("--shrink", type=int, default=1, help="divide the sizes of the sub-block workloads (tests)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's outputs to DIR/<name>.npy (float64, <= 64 MB)")
    args = ap.parse_args()
    wl = dict(WORKLOADS[args.workload])
    if args.steps is None:
        args.steps = wl.get("steps", DEFAULT_STEPS)
    if args.steps < (2 if args.workload == "cfg2" and args.impl == "native" else 1):
        ap.error("--steps must be at least 1 (2 for cfg2: its summaries leg takes batch means)")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the native arm's timed run")
    if args.chains:
        wl["chains"] = args.chains
    if args.N:
        wl["N"] = args.N
    if args.warmup < 3 and args.impl == "native":
        args.warmup = 3                      # timing rule: W >= 3
    if args.impl == "reference":
        return run_reference_arm(args, wl, args.workload)

    # keep stdout clean for the one JSON line: libraries (NCCL prints its version banner to stdout) write to stderr instead
    sys.stdout.flush()
    saved_stdout = os.dup(1)
    os.dup2(2, 1)
    B = Bench(args)
    capi, torch, dist, world, rank = B.capi, B.torch, B.dist, B.world, B.rank
    t_start = time.perf_counter()
    K, W, C, d = args.steps, args.warmup, wl["chains"], wl["d"]
    name = args.workload
    line = dict(metric="chain-steps/s", unit="chain-steps/s", n_gpus=world, steps=args.steps, warmup=args.warmup, higher_is_better=True,
                scaling="weak", vs_baseline=None, dtype="f64", data="synthetic", config=config_block(name, wl, world))

    if name == "cfg5":
        blk = row_sharded_block(B, wl, K, W, parity=False, dump=True)
        line.update(value=blk["value"], ms_per_step=blk["ms_per_step"], gpu_launches=blk["gpu_launches"], e2e=blk["e2e"], clocks=blk.pop("clocks"),
                    roofline=blk["roofline"], row_sharded=blk)
    elif name == "cfg2":
        blk = cfg2_block(B, wl, K, W, clock=True, dump=True)
        line.update(value=blk["value"], ms_per_step=blk["ms"] / args.steps, gpu_launches=blk["gpu_launches"], e2e=blk["e2e"], clocks=blk["clocks"],
                    roofline=blk["roofline"], observed=dict(grad_evals_per_chain_step=blk["grad_evals"] / (C * K)))
    elif name in ("cfg3", "smallN"):
        blk = wave_block(B, name, wl, K, W, clock=True, dump=True)
        line.update(value=blk["value"], ms_per_step=blk["ms_per_step"], gpu_launches=blk["gpu_launches"], e2e=blk["e2e"], clocks=blk.pop("clocks"),
                    roofline=blk["roofline"], grad_evals_per_s=blk["grad_evals_per_s"],
                    observed=dict(accept_rate=blk["accept_rate"], grad_evals_per_chain_step=blk["grad_evals"] / (C * K)))
    else:
        problem = make_problem(wl)
        X, y, hy, b0 = problem
        dm = capi.DeviceModel(B.ctx, wl["family"], d, X, y, hy)
        offset = rank * C                     # global chain ids: Philox streams differ across ranks
        scfg = sampler_for(wl, capi)
        init_state, set_state = headline_state(wl, C, b0, rank)
        B.fp64_peak()
        ms, info, acc_rate, clocks = B.wave_leg(dm, scfg, C, d, init_state, K, W, wl["seed"], offset, set_state, clock=True, dump=True)
        e2e_s, h2d, d2h = B.e2e_leg(dm, scfg, C, d, init_state, K, wl["seed"] + 1, offset, set_state)
        ms_max, e2e_ms_max = B.max_over_ranks(ms, e2e_s * 1e3)
        (evals,) = B.sum_over_ranks(float(info["n_grad_evals"]))
        value = C * world * K / (ms_max / 1e3)
        traffic = None
        prof = os.path.join(ROOT, "profiles", "k1_full_r02_summary.json")
        if not os.path.exists(prof):
            prof = os.path.join(ROOT, "profiles", "k1_full_r01_summary.json")
        if name == "cfg4" and wl["N"] == 1000000 and C == 10000 and os.path.exists(prof):
            m = json.load(open(prof))["metrics"]     # one ncu --set full capture of this kernel on this workload
            traffic = float(m["dram__bytes_read.sum"]["values"][0]) * 1e9 + float(m["dram__bytes_write.sum"]["values"][0]) * 1e6
        line.update(value=value, ms_per_step=ms_max / args.steps, grad_evals_per_s=evals / (ms_max / 1e3), gpu_launches=int(info["n_launches"]),
                    e2e=dict(value=C * world * K / (e2e_ms_max / 1e3), unit="chain-steps/s", h2d_bytes_per_step=h2d / K, d2h_bytes_per_step=d2h / K),
                    clocks=clocks, roofline=B.k1_roofline(wl, C, info, ms, traffic),
                    observed=dict(accept_rate=acc_rate, grad_evals_per_chain_step=info["n_grad_evals"] / (C * K)))

        extras = (name == "cfg4") and not args.no_extras
        if extras and world > 1:
            line["strong"] = strong_block(B, dm, wl, scfg, b0, K, W)
        if not args.no_ess:
            # every rank takes part (the best-len leg is timed with a barrier); the pilot itself runs on rank 0's chains only
            line["min_ess_per_s"] = min_ess_block(B, dm, wl, init_state, set_state, offset, value, K, W)
        if not args.no_cpu_baseline and world == 1:
            cores = os.cpu_count() or 1
            cs = args.cpu_steps if wl["N"] * d > 1e6 else 2000
            cw = 1 if wl["N"] * d > 1e6 else 200
            cb = cpu_baseline(wl, cs, cw, cores, problem)
            c1 = cpu_baseline(wl, cs, cw, 1, problem)
            line["cpu_baseline"] = dict(value=cb["value"], unit="chain-steps/s", cores=cores, kind="port", sample=cb["sample"],
                                        grad_evals_per_s=cb["grad_evals_per_s"],
                                        one_core=dict(value=c1["value"], unit="chain-steps/s", cores=1, sample=c1["sample"],
                                                      grad_evals_per_s=c1["grad_evals_per_s"],
                                                      note="SerialMC is single-threaded (SerialMC.jl:37-85): this is the reference's own shape"),
                                        flags="gcc -O3 -ffp-contract=off (no fast-math); logistic evaluation row-blocked with 4-way partial sums, "
                                              "AVX2/AVX-512 function clones")
        dm.close()
        del problem, X, y
        if extras:
            sh = max(1, args.shrink)
            line["row_sharded"] = row_sharded_block(B, dict(WORKLOADS["cfg5"], N=WORKLOADS["cfg5"]["N"] // sh), 3, 3, parity=world > 1)
            line["row_sharded"].pop("clocks", None)
            if world > 1:
                line["population"] = population_block(B)
            cfgs = {}
            w3 = dict(WORKLOADS["cfg3"]); w3["N"] //= sh; w3["chains"] //= sh
            cfgs["cfg3"] = wave_block(B, "cfg3", w3, 5, 3); cfgs["cfg3"].pop("clocks")
            w2 = dict(WORKLOADS["cfg2"]); w2["chains"] //= sh
            cfgs["cfg2"] = cfg2_block(B, w2, 1000, 600)
            ws = dict(WORKLOADS["smallN"]); ws["chains"] //= sh
            cfgs["smallN"] = wave_block(B, "smallN", ws, 20, 3); cfgs["smallN"].pop("clocks")
            line["configs"] = cfgs
    line["bench_seconds"] = time.perf_counter() - t_start
    if rank == 0:
        sys.stdout.flush()
        os.dup2(saved_stdout, 1)
        print(json.dumps(line), flush=True)
        os.dup2(2, 1)
    B.ctx.close()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def wave_block(B, name, wl, K, W, clock=False, dump=False):
    """compact sub-block: one regression workload through the wave engine (device-timed value, roofline, e2e)"""
    capi, world, rank = B.capi, B.world, B.rank
    C, d = wl["chains"], wl["d"]
    problem = make_problem(wl)
    X, y, hy, b0 = problem
    dm = capi.DeviceModel(B.ctx, wl["family"], d, X, y, hy)
    scfg = sampler_for(wl, capi)
    init_state, set_state = headline_state(wl, C, b0, rank)
    # the value without per-launch events (graph replay of the wave loop), then the same steps with them for the kernel time
    ms, info, acc, clocks = B.wave_leg(dm, scfg, C, d, init_state, K, W, wl["seed"], rank * C, set_state, clock=clock, time_eval=False, dump=dump)
    ms_t, info_t, _, _ = B.wave_leg(dm, scfg, C, d, init_state, K, W, wl["seed"], rank * C, set_state, time_eval=True)
    B.ctx.set_option("time_eval", 0)
    e2e_s, h2d, d2h = B.e2e_leg(dm, scfg, C, d, init_state, K, wl["seed"] + 1, rank * C, set_state)
    B.ctx.set_option("time_eval", 1)
    ms_max, e2e_ms = B.max_over_ranks(ms, e2e_s * 1e3)
    (evals,) = B.sum_over_ranks(float(info["n_grad_evals"]))
    ess = None
    if rank == 0 and not B.args.no_ess:      # min-ESS per chain-step of this sampler on this target (pilot of the same chains)
        sweep, sample = ess_pilot(B, dm, wl, init_state, set_state, rank * C, (None,), ce=min(256, C))
        ess = dict(value=sweep[0]["ess_per_chain_step"] * C * world * K / (ms_max / 1e3), unit="min-ESS/s (min over parameters, summed over chains)",
                   **{k: v for k, v in sweep[0].items() if k not in ("len", "nleaps", "min_ess_per_grad")}, sample=sample)
    dm.close()
    rf = B.k1_roofline(wl, C, info_t, ms_t)
    rf["share_of_step"] = info_t["eval_ms"] / ms                   # share of the (graph-replayed) step
    return dict(description=wl["desc"], N=wl["N"], d=d, chains_per_gpu=C, sampler=wl["sampler"], steps=K, warmup=W,
                value=C * world * K / (ms_max / 1e3), unit="chain-steps/s", ms_per_step=ms_max / K,
                grad_evals_per_s=evals / (ms_max / 1e3), grad_evals=int(info["n_grad_evals"]), accept_rate=acc, gpu_launches=int(info["n_launches"]),
                clocks=clocks, min_ess_per_s=ess,
                e2e=dict(value=C * world * K / (e2e_ms / 1e3), unit="chain-steps/s", h2d_bytes_per_step=h2d / K, d2h_bytes_per_step=d2h / K),
                roofline=dict(bound="tensor", achieved=rf["achieved"], peak=rf["peak"], unit="TFLOP/s", frac=rf["frac"],
                              ms_per_launch=rf["ms_per_launch"], share_of_step=rf["share_of_step"]))


def cfg2_block(B, wl, K, W, clock=False, dump=False):
    """fused per-chain kernel: the whole chain is one launch, so warm-up and timed region are separate runs"""
    capi, torch, world, rank = B.capi, B.torch, B.world, B.rank
    C, d = wl["chains"], wl["d"]
    dm = capi.DeviceModel(B.ctx, "normal_fn", d)
    scfg = sampler_for(wl, capi)

    def fresh(nsteps):
        return capi.DeviceRun(dm, scfg, (1, 1, nsteps), C, np.ones(d), seed=wl["seed"], chain_offset=rank * C, engine="fused")
    r = fresh(W); r.execute(); r.close()
    r = fresh(K)
    B.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    clk = ClockSampler(B.local) if clock else None
    if clk:
        clk.__enter__()
    e0.record(B.stream); info = r.execute(); e1.record(B.stream)
    B.barrier()
    if clk:
        clk.__exit__()
    ms = e0.elapsed_time(e1)
    if dump:
        B.dump_run(r)
    r.close()
    e2e_s, h2d, d2h = B.e2e_leg(dm, scfg, C, d, np.ones(d), K, wl["seed"], rank * C, None, engine="fused")
    # summaries instead of draws: the same run, then src/stats on the device-resident draws (mean, MC variance, ESS, acceptance:
    # what ess(batch) / mean(batch) / acceptance(batch) of the host API do); only the d x C summaries cross PCIe
    bl = min(100, K // 2)                # ess(vtype=:bm) needs at least two batches
    B.barrier()
    t0 = time.perf_counter()
    r = capi.DeviceRun(dm, scfg, (1, 1, K), C, np.ones(d), seed=wl["seed"], chain_offset=rank * C, engine="fused", stream_stats=True,
                       stream_batchlen=bl)
    r.execute()
    st = r.stats("bm", batchlen=bl)
    torch.cuda.synchronize()
    sum_s = time.perf_counter() - t0
    r.close()
    ms_max, e2e_ms, sum_ms = B.max_over_ranks(ms, e2e_s * 1e3, sum_s * 1e3)
    dm.close()
    bytes_per = 8 * d * 2 + 8 + 1       # sample + gradient + log-target + accept flag per kept chain-step
    pk = os.path.join(ROOT, "MEASURED_PEAKS.json")
    hbm = json.load(open(pk))["hbm_gbs"] if os.path.exists(pk) else 6650.0
    ach = bytes_per * C * K / (ms / 1e3) / 1e9
    return dict(description=wl["desc"], chains_per_gpu=C, steps=K, warmup=W, ms=ms_max, grad_evals=int(info["n_grad_evals"]), value=C * world * K / (ms_max / 1e3),
                unit="chain-steps/s", gpu_launches=int(info["n_launches"]), clocks=clk.summary() if clk else None,
                e2e=dict(value=C * world * K / (e2e_ms / 1e3), unit="chain-steps/s", h2d_bytes_per_step=h2d / K, d2h_bytes_per_step=d2h / K),
                e2e_summaries=dict(value=C * world * K / (sum_ms / 1e3), unit="chain-steps/s", h2d_bytes_per_step=d * 8 / K,
                                   d2h_bytes_per_step=(5 * d + 1) * C * 8 / K, median_ess_per_step=float(np.median(st["ess"])) / K,
                                   min_ess_per_s=float(np.median(st["ess"].min(axis=1))) / K * C * world * K / (ms_max / 1e3),
                                   min_ess_note=f"median over chains of min over parameters of ess(vtype=:bm, batch length {bl}) per step x the device-timed chain-steps/s",
                                   note="stream_stats run: mean / var_iid / var_bm / ess(bm) / actime / acceptance accumulated in registers while "
                                        "sampling (mcmcgpu_runner_cfg.stream_stats), no draw is stored; only the d x C summaries cross PCIe"),
                roofline=dict(bound="hbm", achieved=ach, peak=hbm, unit="GB/s", frac=ach / hbm, traffic=None, kernel="fused_chain_kernel",
                              note="store bandwidth of kept draws; the kernel is FP64-ALU/latency bound, see DESIGN.md"))


def strong_block(B, dm, wl, scfg, b0, K, W, total=10000):
    """cfg4 with `total` chains over all GPUs (BASELINE configs[3] as written: '10k chains, chain-sharded at 1/2/4/8')"""
    world, rank = B.world, B.rank
    lo, hi = rank * total // world, (rank + 1) * total // world
    C, d = hi - lo, wl["d"]
    rng = np.random.default_rng(300 + rank)
    init = b0[None, :] + 2e-3 * rng.standard_normal((C, d))
    ss = (1000, np.full(C, CFG4_EPS), np.full(C, CFG4_EPS), np.zeros(C))
    ms, info, acc, _ = B.wave_leg(dm, scfg, C, d, init, K, W, wl["seed"], lo, ss)
    (ms_max,) = B.max_over_ranks(ms)
    rf = B.k1_roofline(wl, C, info, ms)
    return dict(total_chains=total, chains_per_gpu=C, steps=K, value=total * K / (ms_max / 1e3), unit="chain-steps/s", scaling="strong",
                ms_per_step=ms_max / K, k1_ms_per_launch=rf["ms_per_launch"], k1_tflops=rf["achieved"], frac=rf["frac"],
                share_of_step=rf["share_of_step"], accept_rate=acc)


def min_ess_block(B, dm, wl, init_state, set_state, offset, value, K, W):
    lens = ESS_SWEEP_LENS if wl["sampler"] == "HMCDA" else (None,)
    if B.rank == 0:
        sweep, sample = ess_pilot(B, dm, wl, init_state, set_state, offset, lens)
        best = max(range(len(sweep)), key=lambda i: sweep[i]["min_ess_per_grad"] if np.isfinite(sweep[i]["min_ess_per_grad"]) else -1.0)
    else:
        sweep, sample, best = None, None, 0
    head = sweep[0] if sweep else None
    blk = None
    if B.world > 1:
        t = B.torch.tensor([best], device="cuda")
        B.dist.broadcast(t, src=0)
        best = int(t.item())
    best_leg = None
    if wl["sampler"] == "HMCDA" and best != 0:
        # time the same chains at the trajectory length that maximises min-ESS per gradient (a measured number, not a projection)
        C, d = wl["chains"], wl["d"]
        ms, info, acc, _ = B.wave_leg(dm, sampler_for(wl, B.capi, len_=lens[best]), C, d, init_state, K, W, wl["seed"] + 3, offset, set_state)
        (ms_max,) = B.max_over_ranks(ms)
        best_leg = dict(len=lens[best], chain_steps_per_s=C * B.world * K / (ms_max / 1e3), accept_rate=acc,
                        grad_evals_per_chain_step=info["n_grad_evals"] / (C * K))
    if B.rank == 0:
        blk = dict(value=head["ess_per_chain_step"] * value, unit="min-ESS/s (min over parameters, summed over chains)", len=head["len"],
                   ess_per_chain_step=head["ess_per_chain_step"], sweep=sweep, sample=sample)
        if best_leg:
            best_leg.update(ess_per_chain_step=sweep[best]["ess_per_chain_step"], value=sweep[best]["ess_per_chain_step"] * best_leg["chain_steps_per_s"])
            blk["best"] = best_leg
    return blk


def _small_regression(N, d, seed):
    r = np.random.default_rng(seed)
    X = np.concatenate([np.ones((N, 1)), r.standard_normal((N, d - 1))], axis=1)
    b0 = r.standard_normal(d) / np.sqrt(d)
    y = (r.random(N) < 1 / (1 + np.exp(-X @ b0))).astype(float)
    return X, y, b0


def row_shard_parity(B):
    """sharded == unsharded (the body of tests/multigpu_rowshard.py): log-target / gradient to 1e-12, identical accept flags
    with injected draws, every rank identical"""
    capi, torch, dist, rank, world = B.capi, B.torch, B.dist, B.rank, B.world
    N, d, C = 5003, 24, 96
    X, y, b0 = _small_regression(N, d, 5)
    lo, hi = rank * N // world, (rank + 1) * N // world
    full = capi.DeviceModel(B.ctx, "logistic", d, X, y, (1.0, -1.0))
    shard = capi.DeviceModel(B.ctx, "logistic", d, X[lo:hi], y[lo:hi], (1.0, -1.0), row_sharded=True)
    rng = np.random.default_rng(1)
    Bm = b0 + 0.2 * rng.standard_normal((C, d))
    lt0, g0 = full.logtarget_grad(Bm)
    lt1, g1 = shard.logtarget_grad(Bm)
    err_lt = float(np.max(np.abs(lt1 - lt0) / np.abs(lt0)))
    err_g = float(np.max(np.abs(g1 - g0) / np.abs(X).sum(0)))
    zn = rng.standard_normal((C, 31, d)); un = rng.random((C, 31))
    outs = []
    for m in (full, shard):
        run = capi.DeviceRun(m, capi.sampler_cfg("HMC", scale=0.01, nleaps=5), (1, 1, 30), C, np.zeros(d), normals=zn, uniforms=un, engine="wave")
        run.execute(); outs.append(run.fetch()); run.close()
    same_acc = bool(np.array_equal(outs[0]["accept"], outs[1]["accept"]))
    close = bool(np.allclose(outs[0]["samples"], outs[1]["samples"], rtol=1e-9, atol=1e-12))
    t = torch.from_numpy(outs[1]["samples"]).cuda()
    ref = t.clone()
    dist.broadcast(ref, src=0)
    ok = torch.tensor([int(err_lt <= 1e-12 and err_g <= 1e-12 and same_acc and close and bool(torch.equal(t, ref)))], device="cuda")
    dist.all_reduce(ok, op=dist.ReduceOp.MIN)
    full.close(); shard.close()
    return ("ok" if int(ok.item()) == 1 else "FAILED"), dict(max_rel_err_logtarget=err_lt, max_rel_err_gradient=err_g,
                                                              accept_rate=float(outs[1]["accept"].mean()))


def population_block(B):
    """population runners over GPUs (N > 1): a SeqMC population of regression models sharded over the ranks (one ncclAllGather of
    particle states and weights per target, every rank resampling its slots from the global weights) and SerialTempMC replicas
    sharded by global replica id (no communication) must reproduce the single-GPU run of the same population."""
    capi, torch, dist, rank, world = B.capi, B.torch, B.dist, B.rank, B.world
    N, d, npl, nrl = 600, 8, 128, 64
    X, y, b0 = _small_regression(N, d, 7)
    hys = [(4.0, -1.0), (2.0, -1.0), (1.0, -1.0)]
    smp = [capi.sampler_cfg("RWM", scale=0.03), capi.sampler_cfg("MALA", scale=0.002), capi.sampler_cfg("HMC", scale=0.04, nleaps=3)]
    solo = capi.Context(B.local)                      # no communicator: the whole population on this GPU
    out = {}
    try:
        shard_m = [capi.DeviceModel(B.ctx, "logistic", d, X, y, h) for h in hys]
        solo_m = [capi.DeviceModel(solo, "logistic", d, X, y, h) for h in hys]
        rng = np.random.default_rng(13)
        gp = npl * world
        parts = b0 + 0.1 * rng.standard_normal((gp, d))
        steps, burnin = 4, 1
        trig = 1e300                                   # resample after every target: the all-gathered weights decide every slot
        t0 = time.perf_counter()
        sh = B.ctx.run_seqmc_models(shard_m, smp, steps, burnin, trig, parts[rank * npl:(rank + 1) * npl], seed=5)
        t_sh = time.perf_counter() - t0
        ref = solo.run_seqmc_models(solo_m, smp, steps, burnin, trig, parts, seed=5)
        rs = ref["samples"].reshape(steps - burnin, gp, d)[:, rank * npl:(rank + 1) * npl].reshape(-1, d)
        rw = ref["weights"].reshape(steps - burnin, gp)[:, rank * npl:(rank + 1) * npl].reshape(-1)
        ok_seq = sh["n_resamples"] == ref["n_resamples"] and np.allclose(sh["samples"], rs, rtol=1e-9, atol=1e-12) and np.allclose(sh["weights"], rw, rtol=1e-7)
        inits = b0 + 0.05 * rng.standard_normal((3, d))
        tsteps, tburn, swap = 30, 5, 3
        a = B.ctx.run_serialtemp_models(shard_m, smp, tsteps, tburn, swap, nrl, inits, seed=6, rep_offset=rank * nrl)
        b = solo.run_serialtemp_models(solo_m, smp, tsteps, tburn, swap, nrl * world, inits, seed=6)
        ok_tmp = np.array_equal(a["at"], b["at"][rank * nrl:(rank + 1) * nrl]) and np.allclose(a["samples"], b["samples"][rank * nrl:(rank + 1) * nrl], rtol=1e-9, atol=1e-12)
        flags = torch.tensor([int(ok_seq), int(ok_tmp)], device="cuda")
        dist.all_reduce(flags, op=dist.ReduceOp.MIN)
        out = dict(seqmc_sharded_parity="ok" if int(flags[0]) else "FAILED", serialtemp_sharded_parity="ok" if int(flags[1]) else "FAILED",
                   models="3 logistic regressions N=600 d=8 (prior sd 4, 2, 1), tasks RWM / MALA / HMC(3 leapfrogs)",
                   seqmc=dict(particles_total=gp, targets=3, iterations=steps, n_resamples=int(sh["n_resamples"]), seconds=t_sh,
                              allgather_bytes_per_target=(d + 2) * ((npl + 63) // 64 * 64) * 8 * world),
                   serialtemp=dict(replicas_total=nrl * world, steps=tsteps, swap_period=swap, tasks_visited=sorted(set(int(v) for v in np.unique(a["at"])))))
        for m in shard_m + solo_m:
            m.close()
    finally:
        solo.close()
    return out


def row_sharded_block(B, wl, K, W, parity, dump=False):
    """cfg5: every rank generates ITS rows on the device (seeded per rank); chains replicated with identical Philox keys"""
    capi, torch, dist, world, rank = B.capi, B.torch, B.dist, B.world, B.rank
    d, C, N = wl["d"], wl["chains"], wl["N"]
    if world > 1 and not B.comm_ready:
        uid = B.mj.broadcast_unique_id(dist, capi.Context.comm_unique_id, rank)
        B.ctx.comm_init(rank, world, uid)
        B.comm_ready = True
    par, par_detail = ("skipped (1 GPU: no shards)", None)
    if parity and world > 1:
        par, par_detail = row_shard_parity(B)
    g = torch.Generator(device="cuda"); g.manual_seed(wl["seed"] * 1000 + rank)
    g0 = torch.Generator(device="cuda"); g0.manual_seed(wl["seed"])
    b0_t = torch.randn(d, generator=g0, device="cuda", dtype=torch.float64) / d ** 0.5
    Xt = torch.randn(d, N, generator=g, device="cuda", dtype=torch.float64)   # (d, N) row-major == N x d column-major
    Xt[0] = 1.0
    y_t = (torch.rand(N, generator=g, device="cuda", dtype=torch.float64) < torch.sigmoid(b0_t @ Xt)).double()
    torch.cuda.synchronize()
    dm = capi.DeviceModel.from_device(B.ctx, "logistic", N, d, Xt.data_ptr(), y_t.data_ptr(), (1.0, -1.0), row_sharded=world > 1)
    b0 = b0_t.cpu().numpy()
    del Xt, y_t
    torch.cuda.empty_cache()
    scfg = sampler_for(wl, capi)
    init = b0[None, :] + 1e-3 * np.random.default_rng(100).standard_normal((C, d))   # same on every rank
    ms, info, acc, clocks = B.wave_leg(dm, scfg, C, d, init, K, W, wl["seed"], 0, None, clock=True, dump=dump)
    e2e_s, h2d, d2h = B.e2e_leg(dm, scfg, C, d, init, K, wl["seed"] + 1, 0, None)
    ms_max, e2e_ms, k1_ms, comm_ms = B.max_over_ranks(ms, e2e_s * 1e3, info["eval_ms"] / max(info["n_waves"], 1), info["comm_ms"] / max(info["n_waves"], 1))
    dm.close()
    torch.cuda.empty_cache()
    Cp = (C + 63) // 64 * 64
    rf = B.k1_roofline(wl, C, info, ms)
    blk = dict(workload="cfg5", description=wl["desc"], rows_per_gpu=N, rows_total=N * world, d=d, chains=C, steps=K, warmup=W,
               value=C * K / (ms_max / 1e3), unit="chain-steps/s", ms_per_step=ms_max / K, gpu_launches=int(info["n_launches"]),
               k1_ms_per_launch=k1_ms, fold_allreduce_ms_per_leapfrog=comm_ms, allreduce_payload_bytes=(d + 2) * Cp * 8,
               leapfrogs_per_step=info["n_waves"] / K, accept_rate=acc, parity=par, parity_detail=par_detail,
               e2e=dict(value=C * K / (e2e_ms / 1e3), unit="chain-steps/s", h2d_bytes_per_step=h2d / K, d2h_bytes_per_step=d2h / K),
               roofline=dict(bound="tensor", achieved=rf["achieved"], peak=rf["peak"], unit="TFLOP/s", frac=rf["frac"],
                             ms_per_launch=rf["ms_per_launch"], share_of_step=rf["share_of_step"], traffic=None,
                             kernel="k1_kernel (FP64 DMMA m8n8k4)", peak_source=rf["peak_source"]),
               limiter="K1 (likelihood kernel); the fold + all-reduce is fold_allreduce_ms_per_leapfrog of every k1_ms_per_launch",
               clocks=clocks)
    return blk


if __name__ == "__main__":
    main()
