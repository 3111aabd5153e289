import os
import subprocess
import sys

import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_row_sharded_matches_unsharded():
    import torch
    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip("needs >= 2 GPUs")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
           "--master-port", "29611", os.path.join(ROOT, "tests", "multigpu_rowshard.py")]
    p = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert p.returncode == 0 and "ROWSHARD_OK" in p.stdout, p.stdout[-2000:] + p.stderr[-4000:]


def test_seqmc_population_sharded_over_two_gpus():
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs >= 2 GPUs")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
           "--master-port", "29613", os.path.join(ROOT, "tests", "multigpu_seqmc.py")]
    p = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert p.returncode == 0 and "SEQMC_SHARDED_OK" in p.stdout, p.stdout[-2000:] + p.stderr[-4000:]


def test_bench_native_arm_small(tmp_path):
    """bench.py end to end on a reduced cfg4 with every sub-block (the JSON contract keys of the native arm)"""
    import json
    import numpy as np
    small = ["--N", "40000", "--chains", "512", "--steps", "2", "--warmup", "3"]
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *small, "--cpu-steps", "1", "--shrink", "64",
                        "--dump-outputs", str(tmp_path / "a")], capture_output=True, text=True, timeout=900)
    assert p.returncode == 0, p.stderr[-3000:]
    lines = [l for l in p.stdout.strip().splitlines() if l.startswith("{")]
    assert len(lines) == 1 and p.stdout.strip() == lines[0], "stdout must carry exactly the JSON line"
    line = json.loads(lines[0])
    for key in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype",
                "data", "config", "e2e", "gpu_launches", "clocks", "roofline", "cpu_baseline", "min_ess_per_s", "configs", "row_sharded", "observed"):
        assert key in line, key
    assert line["value"] > 0 and line["e2e"]["value"] > 0 and line["e2e"]["d2h_bytes_per_step"] > 0 and line["gpu_launches"] > 0
    rf = line["roofline"]
    assert rf["bound"] == "tensor" and 0 < rf["frac"] < 1.2 and abs(rf["frac"] - rf["achieved"] / rf["peak"]) < 1e-9
    cb = line["cpu_baseline"]
    assert cb["kind"] == "port" and cb["value"] > 0 and cb["one_core"]["value"] > 0 and cb["one_core"]["cores"] == 1
    me = line["min_ess_per_s"]
    assert len(me["sweep"]) == 3 and all(0 <= s["frac_x_nonpositive"] <= 1 and s["nleaps"] >= 1 for s in me["sweep"])
    assert me["value"] > 0 and abs(me["value"] - me["ess_per_chain_step"] * line["value"]) < 1e-6 * me["value"]
    for name in ("cfg3", "cfg2", "smallN"):
        blk = line["configs"][name]
        assert blk["value"] > 0 and blk["e2e"]["value"] > 0 and 0 < blk["roofline"]["frac"] < 1.2, name
    rs = line["row_sharded"]
    assert rs["value"] > 0 and rs["k1_ms_per_launch"] > 0 and rs["fold_allreduce_ms_per_leapfrog"] >= 0 and rs["allreduce_payload_bytes"] == 202 * 256 * 8
    # the reference arm echoes the same config object (the driver compares them)
    q = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--N", "40000", "--chains", "512", "--steps", "1",
                        "--warmup", "1"], capture_output=True, text=True, timeout=900)
    assert q.returncode == 0, q.stderr[-3000:]
    assert json.loads(q.stdout.strip().splitlines()[-1])["config"] == line["config"]
    # --dump-outputs: the headline leg's last step; the same arguments give the same outputs (the sub-blocks run after it)
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *small, "--no-extras", "--no-ess", "--no-cpu-baseline",
                        "--dump-outputs", str(tmp_path / "b")], capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-3000:]
    shapes = dict(samples=(512, 100), grads=(512, 100), logtarget=(512,), accept=(512,), chain_index=(512,))
    for name, shape in shapes.items():
        a, b = np.load(tmp_path / "a" / f"{name}.npy"), np.load(tmp_path / "b" / f"{name}.npy")
        assert a.shape == shape and a.dtype == np.float64 and np.all(np.isfinite(a)), name
        assert np.array_equal(a, b), name
    assert np.array_equal(np.load(tmp_path / "a" / "chain_index.npy"), np.arange(512))
    assert set(np.unique(np.load(tmp_path / "a" / "accept.npy"))) <= {0.0, 1.0}


@pytest.mark.parametrize("workload,nleaps,initial,d", [("smallN", 8, 0, 100), ("cfg2", 10, 1, 3)])
def test_bench_times_exactly_steps(tmp_path, workload, nleaps, initial, d):
    """--steps is the number of timed MCMC steps: the device counts nleaps gradient evaluations per chain and timed step, plus
    `initial` for the starting point (cfg2's fused run starts there; smallN's timed segment resumes after the warm-up)"""
    import json
    import numpy as np
    K, C = 6, 1024
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", workload, "--chains", str(C), "--steps", str(K),
                        "--warmup", "3", "--no-ess", "--no-cpu-baseline", "--dump-outputs", str(tmp_path)], capture_output=True, text=True,
                       timeout=900)
    assert p.returncode == 0, p.stderr[-3000:]
    line = json.loads(p.stdout.strip().splitlines()[-1])
    assert line["steps"] == K
    assert line["observed"]["grad_evals_per_chain_step"] == pytest.approx(nleaps + initial / K, rel=1e-12)
    samples = np.load(tmp_path / "samples.npy")
    assert samples.shape == (C, d) and np.all(np.isfinite(samples))


def test_c_abi_from_plain_c(tmp_path):
    """examples/c_abi_demo.c: the library driven from C exactly as a Julia ccall would (no Python in the loop)"""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from test_capi_and_host import _build_c_demo
    p = subprocess.run([_build_c_demo(tmp_path)], capture_output=True, text=True, timeout=300)
    assert p.returncode == 0 and "C_ABI_DEMO ok" in p.stdout, p.stdout + p.stderr
