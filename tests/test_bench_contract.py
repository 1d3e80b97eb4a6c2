"""The reference arm of bench.py runs on CPU (it times the oracle), so its half of the driver's contract can be checked here:
one JSON line with the keys the driver reads, the same metric/unit/config as the B200 arm, and no work on ranks other than 0."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def run(env=None, *args):
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", *args], capture_output=True, text=True,
                          env={**os.environ, **(env or {})}, timeout=900, cwd=ROOT)


def check_dump(directory, golden_key):
    """--dump-outputs: the last timed step's GFA (cfg1's fits whole) and graph counts, against the oracle's committed values."""
    import hashlib
    import numpy as np
    g = json.load(open(os.path.join(ROOT, "tests", "golden", "config_goldens.json")))[golden_key]
    gfa = np.load(os.path.join(directory, "gfa.npy"))
    assert gfa.dtype == np.float32 and hashlib.sha256(gfa.astype(np.uint8).tobytes()).hexdigest() == g["sha256"]
    assert np.load(os.path.join(directory, "gfa_size.npy")).tolist() == [g["gfa_bytes"]]
    counts = np.load(os.path.join(directory, "graph_counts.npy"))
    assert counts.dtype == np.float64 and counts[:3].tolist() == [g["n_kmers"], g["unitigs_after"], g["links_after"]]


def test_reference_arm_line(tmp_path):
    r = run(None, "--steps", "2", "--warmup", "1", "--workload", "cfg1", "--dump-outputs", str(tmp_path / "out"))      # the default (full cfg2) takes minutes per pass on one core
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for key in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
                "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert key in d, key
    assert d["impl"] == "reference" and d["unit"] == "Mbp/s" and d["higher_is_better"] is True and d["vs_baseline"] is None
    assert d["metric"] == json.load(open(os.path.join(ROOT, "BASELINE.json")))["metric"] or "Mbp/sec" in d["metric"]
    assert d["value"] > 0 and d["e2e"] == {"value": d["value"], "unit": "Mbp/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] == 1 and d["cpu_baseline"]["value"] == d["value"]
    assert "-march=native" in d["cpu_baseline"]["build"] and d["cpu_baseline"]["host_cores"] >= 1
    assert "workload" in d["config"] and "sample" in d["config"] and d["config"]["input_bases"] == 299982
    assert d["steps_timed"] == 2 and d["parity"]["ok"] is True and d["parity"]["golden_key"] == "cfg1_k51"      # the timed output is the committed oracle output
    check_dump(tmp_path / "out", "cfg1_k51")


def test_workload_selection_matches_the_committed_goldens():
    """N = 1 runs cfg2, N > 1 the first 8N assemblies of cfg5; both arms name the same golden."""
    import argparse
    import sys
    sys.path.insert(0, ROOT)
    import bench
    goldens = json.load(open(os.path.join(ROOT, "tests", "golden", "config_goldens.json")))
    for n, key in [(1, "cfg2_k51"), (2, "cfg5_k51_n16"), (4, "cfg5_k51_n32"), (8, "cfg5_k51_n64")]:
        wl, per_rank, n_asm, golden_key, label = bench.workload_for(argparse.Namespace(workload=None, k=51), n)
        assert golden_key == key and per_rank == 8 and n_asm == 8 * n
        assert key in goldens, f"no committed oracle hash for {key}"


def test_reference_arm_other_ranks_do_nothing():
    r = run({"RANK": "1", "WORLD_SIZE": "2", "LOCAL_RANK": "1"}, "--gpus", "2", "--steps", "1", "--warmup", "0")
    assert r.returncode == 0 and r.stdout.strip() == ""


@pytest.mark.gpu
def test_b200_arm_line(tmp_path):
    """The B200 arm on the smallest BASELINE config (a second or two on the GPU): one JSON line with the driver's keys, the timed output
    equal to the oracle's committed hash, kernels of this library counted, the roofline entry for the insert kernel timed on its own."""
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "cfg1", "--steps", "3", "--warmup", "3", "--no-cpu-baseline",
                        "--dump-outputs", str(tmp_path / "out")], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for key in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype", "data",
                "config", "e2e", "gpu_launches", "parity", "clocks", "roofline", "stage_ms"):
        assert key in d, key
    assert d["n_gpus"] == 1 and d["steps"] == 3 and d["unit"] == "Mbp/s" and d["higher_is_better"] is True and d["vs_baseline"] is None
    assert d["parity"]["ok"] is True and d["parity"]["golden_key"] == "cfg1_k51"
    assert d["value"] > 0 and d["e2e"]["value"] > 0 and d["e2e"]["h2d_bytes_per_step"] > 0 and d["e2e"]["d2h_bytes_per_step"] > 0
    assert d["gpu_launches"] >= 3 * 30
    rf = d["roofline"]
    assert rf["bound"] == "hbm" and rf["unit"] == "GB/s" and 0 < rf["frac"] < 1 and abs(rf["frac"] - rf["achieved"] / rf["peak"]) < 1e-3
    assert 0 < rf["kernel_ms"] <= d["stage_ms"]["insert"] + 1e-3 and d["stage_ms"]["host_simplify"] == 0 and d["stage_ms"]["host_gfa"] == 0
    check_dump(tmp_path / "out", "cfg1_k51")
