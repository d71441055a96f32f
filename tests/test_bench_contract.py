"""bench.py keeps the driver's JSON contract (both arms)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BASE_KEYS = {"metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better",
             "scaling", "vs_baseline", "dtype", "data", "config", "e2e", "gpu_launches"}


def run_bench(*args, timeout=300):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True,
                         text=True, timeout=timeout, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1, out.stdout
    return json.loads(lines[0])


def test_reference_arm_contract():
    d = run_bench("--impl", "reference", "--workload", "C2", "--steps", "3", "--warmup", "1")
    assert BASE_KEYS <= set(d)
    assert d["impl"] == "reference" and d["higher_is_better"] is True and d["vs_baseline"] is None
    assert d["unit"] == "decisions/s" and d["value"] > 0 and d["steps"] == 3
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and "requests per step" in cb["sample"]
    assert d["repo_libraries_loaded"] == ["liblig_oracle.so"]            # the reference arm never loads the product
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"] and "model" not in d["config"]


def test_reference_arm_other_ranks_exit_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2",
                          "--workload", "C2", "--steps", "2", "--warmup", "1"], capture_output=True, text=True,
                         timeout=120, cwd=ROOT, env=env)
    assert out.returncode == 0 and out.stdout.strip() == ""


@pytest.mark.gpu
def test_gpu_arm_contract():
    d = run_bench("--workload", "C3", "--steps", "20", "--warmup", "3", "--min-seconds", "0.05",
                  "--cpu-seconds", "0.5", "--stream-seconds", "2")
    assert BASE_KEYS <= set(d) and "impl" not in d
    assert d["n_gpus"] == 1 and d["steps"] == 20 and d["warmup"] == 3 and d["scaling"] == "weak"
    assert d["value"] > 1e8 and d["gpu_launches"] == 1                   # a queue of K steps is ONE launch
    par = d["parity"]
    assert par["ranks_checked"] == 1 and par["picks_checked_per_rank"] == 65536 and par["port_sample_per_rank"] > 0
    rf = d["roofline"]
    assert rf["bound"] == "hbm" and rf["unit"] == "GB/s" and abs(rf["frac"] - rf["achieved"] / rf["peak"]) < 1e-9
    assert rf["kernel"].startswith("lig_pick_persistent_kernel")
    assert d["details"]["kernel"]["tables_in_smem"] is True
    assert rf["algorithmic_bytes_per_step"] == int(24 * 65536 + (16 * 512 + 4 * 256 * 16) / 20)
    assert rf["algorithmic_bytes_per_launch"] == rf["algorithmic_bytes_per_step"] * 20
    assert rf["traffic"] is None and "capture" in rf["traffic_note"]     # the committed capture is of C4, not C3
    e = d["e2e"]
    assert e["value"] > 0 and e["h2d_bytes_per_step"] >= 4 * 65536 and e["d2h_bytes_per_step"] == 4 * 65536
    assert e["value"] < d["value"] and e["descriptor_call"]["d2h_bytes_per_step"] == 8 * 65536
    assert {"1", "20", "200"} <= set(d["k_sweep"]) and d["strong"]["requests_per_gpu"] == 65536
    assert d["snapshot_tick"]["us"] > 0 and d["adapter_dist_uniform"]["value"] > 0 and d["model_requests"]["value"] > 0
    assert d["k_sweep"]["launch_floor_us"] > 0 and d["strong"]["k200"]["value"] > 0
    fb = d["load_feedback"]
    assert fb["max_picks_per_pod"]["with_feedback"] <= fb["max_picks_per_pod"]["default"]
    assert fb["pods_used"]["with_feedback"] >= fb["pods_used"]["default"]
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] > 0
    assert cb["class_table_cpu"]["value"] > cb["optimised_cpu"]["value"] > cb["single_thread"]["value"]
    assert set(d["clocks"]) >= {"sm_mhz", "sm_max_mhz", "reasons"}
    assert d["streaming"]["errors"] == 0 and d["streaming"]["latency_us"]["p99"] > 0


def test_dump_picks_samples_rows_above_the_cap(tmp_path, monkeypatch):
    import bench
    from llm_instance_gateway_b200.packer import PICK_DTYPE
    picks = np.zeros(1000, dtype=PICK_DTYPE)
    picks["pod_idx"] = np.arange(1000) - 1
    picks["status"] = np.arange(1000) % 4
    picks["n_survivors"] = np.arange(1000) % 65536
    bench.dump_picks(str(tmp_path / "whole"), picks)
    assert sorted(os.listdir(tmp_path / "whole")) == ["n_survivors.npy", "pod_idx.npy", "status.npy"]
    for name in PICK_DTYPE.names:
        got = np.load(tmp_path / "whole" / f"{name}.npy")
        assert got.dtype == np.float32 and np.array_equal(got, picks[name])
    monkeypatch.setattr(bench, "DUMP_BYTES", 2000)
    for d in ("a", "b"):
        bench.dump_picks(str(tmp_path / d), picks)
    rows = np.load(tmp_path / "a" / "row.npy")
    assert rows.dtype == np.float64 and len(rows) == 2000 // 20 and np.all(np.diff(rows) > 0)
    for name in ("row",) + PICK_DTYPE.names:                                # the sample is seeded
        assert np.array_equal(np.load(tmp_path / "a" / f"{name}.npy"), np.load(tmp_path / "b" / f"{name}.npy"))
    assert np.array_equal(np.load(tmp_path / "a" / "pod_idx.npy"), picks["pod_idx"][rows.astype(np.int64)])


@pytest.mark.gpu
def test_dump_outputs_are_the_last_timed_step(tmp_path, oracle):
    """K timed steps over a ring of the 4 host-generated batches: step K-1 reads batch (K-1) % 4 with
    seed 1000 + K-1, and --dump-outputs writes exactly its picks."""
    from llm_instance_gateway_b200 import workload as WL
    K = 7
    d = run_bench("--workload", "C3", "--steps", str(K), "--warmup", "3", "--ring", "4", "--min-seconds", "0",
                  "--no-extras", "--no-streaming", "--no-cpu-baseline", "--dump-outputs", str(tmp_path))
    assert d["steps"] == K and d["details"]["timed_steps"] == K
    c = WL.CONFIGS["C3"]
    pk = WL.make_snapshot(c["P"], c["A"]).packed
    reqs = WL.make_requests(c["R"], c["A"], seed=WL.REQUEST_SEED + (K - 1) % 4)
    tab = oracle.ClassTable(pk.P, pk.A, pk.kv, pk.q, pk.n_active, pk.max_active, pk.bitmap)
    want = tab.schedule_batch(reqs, 1000 + K - 1)
    assert sorted(os.listdir(tmp_path)) == ["n_survivors.npy", "pod_idx.npy", "status.npy"]
    for name in want.dtype.names:
        got = np.load(tmp_path / f"{name}.npy")
        assert got.dtype == np.float32 and np.array_equal(got, want[name])


@pytest.mark.gpu
def test_committed_traffic_capture_matches_the_default_kernel():
    """profiles/traffic.json vouches for the kernel bench.py launches by default on C4."""
    from llm_instance_gateway_b200 import workload as WL
    from llm_instance_gateway_b200.engine import Engine
    t = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))["C4"]
    c = WL.CONFIGS["C4"]
    with Engine(0, max_pods=c["P"], max_adapters=c["A"], max_batch=1024) as e:
        e.upload_snapshot(1, WL.make_snapshot(c["P"], c["A"]).packed)
        info = e.pick_kernel_info(1)
    assert (t["capture"]["kernel"], t["capture"]["grid"], t["capture"]["threads"]) == (info["kernel"], info["grid"], info["threads"])
    assert 0.85 * 24 * c["R"] < t["bytes_per_step"] < 1.1 * 24 * c["R"]      # no wasted re-reads
