"""CPU suite, part 4: bench.py's reference arm runs without a GPU and prints the contract's JSON line."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_json_line():
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload", "cfg2", "--steps", "1",
                        "--warmup", "1"], capture_output=True, text=True, timeout=300)
    assert p.returncode == 0, p.stderr[-2000:]
    line = json.loads(p.stdout.strip().splitlines()[-1])
    for key in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
                "dtype", "data", "config", "impl", "cpu_baseline", "e2e"):
        assert key in line, key
    assert line["impl"] == "reference" and line["metric"] == "chain-steps/s" and line["dtype"] == "f64" and line["value"] > 0
    assert line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["cores"] >= 1
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["e2e"]["value"] == line["value"]
    assert line["config"]["workload"] == "cfg2" and line["vs_baseline"] is None
    # the config object is built by one function for both arms, so the driver's `same_config` comparison holds
    sys.path.insert(0, ROOT)
    import bench
    assert line["config"] == bench.config_block("cfg2", bench.WORKLOADS["cfg2"], 1)
    for key in ("chains_per_gpu", "seed", "eps", "len", "parallelism", "N", "d", "sampler"):
        assert key in bench.config_block("cfg4", bench.WORKLOADS["cfg4"], 8)


def test_dump_last_step_whole_and_sampled(tmp_path, monkeypatch):
    """--dump-outputs writes the last step of every fetched array as float64; above the byte budget the same seeded sample of
    chains every time, listed in chain_index.npy"""
    import numpy as np
    sys.path.insert(0, ROOT)
    import bench
    C, S, d = 1000, 4, 7
    rng = np.random.default_rng(0)
    res = dict(samples=rng.standard_normal((C, S, d)), grads=rng.standard_normal((C, S, d)),
               accept=rng.integers(0, 2, (C, S), dtype=np.uint8), logtarget=rng.standard_normal((C, S)))

    def load(sub):
        out = {k: np.load(tmp_path / sub / f"{k}.npy") for k in (*res, "chain_index")}
        assert all(v.dtype == np.float64 for v in out.values())
        return out
    bench.dump_last_step(str(tmp_path / "whole"), res)
    whole = load("whole")
    assert np.array_equal(whole["chain_index"], np.arange(C))
    for k, v in res.items():
        assert np.array_equal(whole[k], v[:, -1])
    monkeypatch.setattr(bench, "DUMP_BYTES", 100 * 8 * (3 + 2 * d))
    bench.dump_last_step(str(tmp_path / "a"), res)
    bench.dump_last_step(str(tmp_path / "b"), res)
    a, b = load("a"), load("b")
    idx = a["chain_index"].astype(np.int64)
    assert len(idx) == 100 and np.all(np.diff(idx) > 0) and idx[-1] < C
    for k, v in res.items():
        assert np.array_equal(a[k], v[idx, -1]) and np.array_equal(a[k], b[k])


def test_bench_rejects_arguments_it_cannot_honour():
    """the reference arm has no device outputs to dump; a run needs a timed step (cfg2's summaries leg two)"""
    for args, flag in ((["--impl", "reference", "--dump-outputs", "unused"], "--dump-outputs"), (["--steps", "0"], "--steps"),
                       (["--workload", "cfg2", "--steps", "1"], "--steps")):
        p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True, timeout=300)
        assert p.returncode == 2 and flag in p.stderr, p.stderr[-2000:]
