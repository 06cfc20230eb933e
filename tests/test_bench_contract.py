"""bench.py contract: the reference arm prints exactly ONE JSON line on stdout with the agreed keys (CPU), and
--dump-outputs writes what the timed path returned (GPU)."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_json_line():
    from oracle import oracle as O
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1",
                        "--nv-per-gpu", "16384"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert p.returncode == 0, p.stderr[-2000:]
    lines = [ln for ln in p.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, p.stdout
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "louvain_phase_edges_per_sec" and d["unit"] == "edges/s"
    assert d["higher_is_better"] is True and d["n_gpus"] == 1 and d["steps"] == 1 and d["warmup"] == 1
    assert d["value"] > 0 and d["ms_per_step"] > 0
    assert d["cpu_baseline"]["kind"] == ("reference" if O.have_reference() else "port")
    assert d["cpu_baseline"]["value"] == d["value"] and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"] == {"value": d["value"], "unit": "edges/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"] and d["config"]["nv"] == 16384 and d["config"]["ne"] == 129456
    assert d["cpu_baseline"]["same_graph_as_gpu_arm"] is True and d["reference_runs_timed"] >= 1


def test_both_arms_describe_the_same_workload():
    """`config` is built by one function from (N, nv, ne) only: the two arms' JSON lines carry identical dictionaries."""
    sys.path.insert(0, ROOT)
    import bench
    a = bench.workload_config(2, 2 * 16777216, 378438414)
    assert a == bench.workload_config(2, 2 * 16777216, 378438414) and a["strips"] == 2 and "33554432" in a["workload"]
    g, name = bench.load_golden(33554432, 2)
    assert g is not None and g["ne"] == 378438414 and name.endswith("golden_full_33554432_p2.json")
    for n in (1, 2, 4, 8):
        assert bench.load_golden(16777216 * n, n)[0] is not None
    import numpy as np
    from oracle import oracle as O
    comm = np.arange(1000, dtype=np.int64)[::-1].copy()
    assert bench.comm_hash_np(7, comm) == O.comm_hash(7, comm)


def test_reference_arm_other_ranks_exit_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1",
                        "--warmup", "1"], capture_output=True, text=True, timeout=120, cwd=ROOT, env=env)
    assert p.returncode == 0 and p.stdout.strip() == ""


@pytest.mark.gpu
def test_dump_outputs_hold_the_last_timed_result(tmp_path, golden):
    """At 16384 vertices the dump is the whole assignment: the graph of `miniVite -n 16384`, so the reference's
    golden (rgg_n16384_p1) pins iterations, modularity and the final assignment hash."""
    import numpy as np
    from oracle import oracle as O
    out = tmp_path / "out"
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "2", "--warmup", "0", "--nv-per-gpu",
                        "16384", "--no-cpu-baseline", "--dump-outputs", str(out)], capture_output=True, text=True,
                       timeout=600, cwd=ROOT)
    assert p.returncode == 0, p.stderr[-2000:]
    d = json.loads(p.stdout)
    assert d["steps"] == 2
    files = {f.name: np.load(f) for f in out.iterdir()}
    assert set(files) == {"modularity.npy", "iterations.npy", "communities.npy", "community_vertices.npy"}
    assert all(a.dtype == np.float64 for a in files.values())
    case = golden["rgg_n16384_p1"]
    assert files["iterations.npy"][0] == case["iters"] == d["result"]["iterations"]
    assert files["modularity.npy"][0] == float(case["modularity"]) == d["result"]["modularity"]
    assert np.array_equal(files["community_vertices.npy"], np.arange(16384))
    assert "%016x" % O.comm_hash(0, files["communities.npy"].astype(np.int64)) == case["final_chash"]
