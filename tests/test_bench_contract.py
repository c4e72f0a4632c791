"""The `bench.py --impl reference` arm (the reference's own CPU algorithm -- the oracle port, since the Rust crate
cannot be built here -- timed on the host cores) runs without a GPU: its JSON line must carry the keys the driver
reads, and under torchrun only rank 0 may work and print.  The `ours` arm needs a B200 and must refuse to run
without one (no CPU fallback)."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def run_bench(*argv, env=None):
    e = dict(os.environ)
    e.pop("RANK", None)
    e.pop("WORLD_SIZE", None)
    e.update(env or {})
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *argv], capture_output=True, text=True,
                          env=e, timeout=600)


def test_reference_arm_line_has_the_contract_keys():
    res = run_bench("--impl", "reference", "--workload", "tiny", "--steps", "2", "--warmup", "1")
    assert res.returncode == 0, res.stderr[-2000:]
    lines = [ln for ln in res.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, "stdout carries exactly one JSON line"
    d = json.loads(lines[0])
    assert d["impl"] == "reference"
    assert d["metric"] == "count_kmer_31mer_queries_per_sec" and d["unit"] == "queries/s"
    assert d["higher_is_better"] is True and d["scaling"] == "strong" and d["vs_baseline"] is None
    assert d["steps"] == 2 and d["warmup"] == 1 and d["n_gpus"] == 1
    assert d["dtype"] == "u64" and d["data"] == "synthetic" and d["gpu_launches"] == 0
    assert d["value"] > 0 and d["ms_per_step"] > 0
    assert d["config"]["workload"].startswith("tiny") and d["config"]["k"] == 31 and "model" not in d["config"]
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and "queries per step" in cb["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_reference_arm_other_ranks_exit_quietly():
    res = run_bench("--impl", "reference", "--workload", "tiny", "--gpus", "2", env={"RANK": "1", "WORLD_SIZE": "2"})
    assert res.returncode == 0, res.stderr[-2000:]
    assert res.stdout.strip() == ""


def test_our_arm_refuses_to_run_without_a_device():
    import torch
    if torch.cuda.is_available():
        import pytest
        pytest.skip("a GPU is present")
    res = run_bench("--workload", "tiny", "--steps", "1", "--warmup", "1")
    assert res.returncode != 0
    assert "no CPU fallback" in (res.stderr + res.stdout)


def test_bench_helpers_on_cpu():
    """encode_u64 (the packed-integer input format of msbwt_count_kmers_u64: first symbol most significant, A,C,G,T =
    0..3) and the `config` object, which must be identical in both arms"""
    import numpy as np
    import torch
    sys.path.insert(0, ROOT)
    import bench
    q = torch.tensor([[1, 2, 3, 5], [5, 5, 5, 5], [1, 1, 1, 1]], dtype=torch.uint8)
    assert bench.encode_u64(q, 4).tolist() == [0b00011011, 0b11111111, 0]
    rng = np.random.default_rng(0)
    q = rng.choice(np.array([1, 2, 3, 5], dtype=np.uint8), size=(1000, 31))
    want = np.zeros(1000, dtype=np.uint64)
    code = np.zeros(6, dtype=np.uint64)
    code[[1, 2, 3, 5]] = [0, 1, 2, 3]
    for j in range(31):
        want = (want << np.uint64(2)) | code[q[:, j]]
    assert (bench.encode_u64(torch.from_numpy(q), 31).numpy().view(np.uint64) == want).all()
    c = bench.workload_config(bench.WORKLOADS["cfg3"], 1_510_000_000, 4)
    assert c["workload"].startswith("configs[2]") and c["queries"] == 100_000_000 and c["k"] == 31
    assert bench.workload_config(bench.WORKLOADS["cfg5"], 3_020_000_000, 8)["queries"] == 1_000_000_000
    assert bench.HEADLINE == "cfg3" and bench.WORKLOADS["cfg3"]["scaling"] == "strong"


def test_steps_below_one_are_refused():
    res = run_bench("--impl", "reference", "--workload", "tiny", "--steps", "0")
    assert res.returncode != 0 and "--steps must be at least 1" in res.stderr


def test_dump_outputs_writes_a_fixed_sample_of_the_counts(tmp_path):
    """--dump-outputs: float64 counts with their batch positions; a large batch is sampled at the same positions every
    run, and the default run's three workloads stay within 64 MB"""
    import numpy as np

    import bench
    small = np.arange(1000, dtype=np.uint64) * np.uint64(3)
    bench.dump_outputs(str(tmp_path / "a"), "tiny", small, 0)
    c, i = np.load(tmp_path / "a" / "tiny_counts.npy"), np.load(tmp_path / "a" / "tiny_query_index.npy")
    assert c.dtype == np.float64 and i.dtype == np.float64
    assert (i == np.arange(1000)).all() and (c == 3 * np.arange(1000)).all()

    n = 3 * bench.DUMP_SAMPLE + 5
    big = np.arange(n, dtype=np.uint64) + np.uint64(2**40)
    for run in ("b", "c"):
        bench.dump_outputs(str(tmp_path / run), "cfg3", big, 7)
    c, i = np.load(tmp_path / "b" / "cfg3_counts.npy"), np.load(tmp_path / "b" / "cfg3_query_index.npy")
    assert c.shape == i.shape == (bench.DUMP_SAMPLE,)
    assert (np.diff(i) > 0).all() and i[0] >= 7 and i[-1] < n + 7
    assert (c == i - 7 + 2**40).all()
    assert (np.load(tmp_path / "c" / "cfg3_query_index.npy") == i).all()
    per_workload = sum(os.path.getsize(tmp_path / "b" / f) for f in os.listdir(tmp_path / "b"))
    assert 3 * per_workload <= 64 << 20


def test_clock_sampler_keeps_the_samples_inside_the_timed_region(tmp_path):
    """bench.py's `clocks` object: nvidia-smi lines carry their own time stamps; only those inside the timed region count
    (the region is ~40 ms on the headline workload), with explicit fallbacks when none falls inside"""
    import datetime
    import time

    import bench

    def stamp(t):
        return datetime.datetime.fromtimestamp(t).strftime("%Y/%m/%d %H:%M:%S.%f")[:-3]

    class Done:
        def terminate(self):
            pass

        def wait(self, timeout=0):
            pass

    now = time.time()

    def sampler(lines):
        c = bench.ClockSampler(0)
        p = tmp_path / f"s{len(lines)}_{lines[0][0]}.csv"
        p.write_text("".join(f"{stamp(now + dt)}, 0, {mhz}, 1965, 512.3, 0x0, Not Active, Not Active, Not Active, {cap}\n" for dt, mhz, cap in lines))
        c.proc, c.path = Done(), str(p)
        return c

    lines = [(-0.30, 1200, "Not Active"), (0.010, 1965, "Not Active"), (0.030, 1950, "Active"), (0.200, 900, "Not Active")]
    got = sampler(lines).stop(now, now + 0.040)
    assert got == {"sm_mhz": 1957.5, "sm_max_mhz": 1965.0, "reasons": ["sw_power_cap"], "samples": 2, "window": "timed region"}
    near = sampler([(-0.02, 1965, "Not Active"), (0.5, 900, "Not Active")]).stop(now, now + 0.010)
    assert near["samples"] == 1 and near["sm_mhz"] == 1965.0 and near["window"] == "timed region +- 50 ms"
    far = sampler([(-1.0, 1800, "Not Active")]).stop(now, now + 0.010)
    assert far["samples"] == 1 and far["window"] == "warm-up + timed region"
    assert bench.ClockSampler(0).stop(now, now + 1)["sm_mhz"] is None   # never started: no clocks, no crash
