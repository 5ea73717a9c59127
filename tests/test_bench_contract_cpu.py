"""CPU: the bench.py output contract.  (1) the committed B200 lines under profiles/ carry every key the driver and the
judge read; (2) the reference arm (`--impl reference`: the oracle port of the reference's PyTorch CPU path, the one
leg that runs without a GPU) produces a well-formed line here."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BASE_KEYS = {"metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
             "vs_baseline", "dtype", "data", "config", "e2e", "gpu_launches"}


def _line(path):
    with open(path) as fp:
        return json.loads(fp.read().strip().splitlines()[-1])


@pytest.mark.parametrize("name,n_gpus", [("r01b_bench_wg.json", 1), ("r01b_bench_wg_2gpu.json", 2), ("r01b_bench_wg_8gpu.json", 8),
                                         ("r01b_bench_c1.json", 1), ("r02_bench_wg_1gpu.json", 1), ("r02_bench_wg_4gpu.json", 4),
                                         ("r02_bench_wg_8gpu.json", 8), ("r02_bench_c1_1gpu.json", 1)])
def test_committed_bench_lines_follow_the_contract(name, n_gpus):
    d = _line(os.path.join(ROOT, "profiles", name))
    assert BASE_KEYS <= set(d), BASE_KEYS - set(d)
    base = json.load(open(os.path.join(ROOT, "BASELINE.json")))
    assert d["metric"].split(" (")[0] in base["metric"] and d["unit"] == "GE/s"
    assert d["n_gpus"] == n_gpus and d["warmup"] >= 3 and d["higher_is_better"] is True and d["vs_baseline"] is None
    assert d["dtype"] == "f32" and d["data"] == "synthetic" and "workload" in d["config"] and "model" not in d["config"]
    assert abs(d["value"] - d["config"]["total_stored_entries"] / (d["ms_per_step"] * 1e-3) / 1e9) <= 1e-9 * d["value"]
    e = d["e2e"]
    assert {"value", "unit", "h2d_bytes_per_step", "d2h_bytes_per_step"} <= set(e)
    assert e["h2d_bytes_per_step"] > 0 and e["d2h_bytes_per_step"] > 0 and 0 < e["value"] < d["value"]
    assert d["gpu_launches"] > 0
    c = d["clocks"]
    assert {"sm_mhz", "sm_max_mhz", "reasons"} <= set(c)
    assert not set(c["reasons"]) & {"hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown"}
    r = d["roofline"]
    assert {"bound", "achieved", "peak", "unit", "frac", "traffic"} <= set(r) and r["bound"] == "hbm" and r["unit"] == "GB/s"
    assert abs(r["frac"] - r["achieved"] / r["peak"]) <= 1e-9
    if n_gpus == 1 and "WG" in d["config"]["workload"]:
        assert r["traffic"] and r["traffic"] < r["algorithmic_bytes_per_launch"]      # no wasted re-reads
        b = d["cpu_baseline"]
        assert {"value", "unit", "cores", "kind", "sample"} <= set(b) and b["kind"] in ("port", "reference") and b["cores"] >= 1
    if name.startswith("r02") and n_gpus == 1 and "WG" in d["config"]["workload"]:
        # round 2: the cache-served algorithmic fraction is reported next to the honest ones
        assert 0 < r["compulsory_frac"] < 1 and 0 < r["time_bound_frac"] <= 1 and r["l2_read_peak"] > r["peak"]
        assert 0 < r["spmm"]["time_bound_frac"] <= 1
        g = d["gpu_baseline"]
        assert g["kind"] == "port" and 0 < g["e2e"] < g["value"] < d["value"]


def test_permuted_graph_keeps_degrees_and_symmetry():
    """bench.py --graph permuted: P A P^T of a symmetric pattern (the locality sensitivity line)."""
    import numpy as np
    from scipy import sparse
    sys.path.insert(0, ROOT)
    import bench
    a = sparse.random(300, 300, 0.03, format="csr", random_state=3)
    a = ((a + a.T) > 0).astype(np.float32).tocsr()
    a.sort_indices()
    ip, ix = bench.permute_pattern(a.indptr.astype(np.int32), a.indices.astype(np.int32), 9)
    b = sparse.csr_matrix((np.ones(ix.shape[0]), ix, ip), shape=a.shape)
    assert ix.shape[0] == a.nnz and (b != b.T).nnz == 0
    assert sorted(np.diff(ip).tolist()) == sorted(np.diff(a.indptr).tolist())
    assert all(np.all(np.diff(ix[ip[i]:ip[i + 1]]) > 0) for i in range(300))          # rows column-sorted
    assert not np.array_equal(ix, a.indices)


def test_steps_below_one_are_refused():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload", "c1", "--steps", "0"],
                         capture_output=True, text=True, timeout=120, cwd=ROOT)
    assert out.returncode != 0 and "--steps" in out.stderr


def test_dump_row_sample_is_fixed_and_within_budget():
    """--dump-outputs writes the same rows of every probability matrix on every run and build, 64 MB at most in all:
    whole-genome graphs share the probability budget, and so do the ranks' row blocks of the st graph."""
    import numpy as np
    sys.path.insert(0, ROOT)
    import bench
    from chromegcn_b200 import synthetic
    from chromegcn_b200.dist import row_partition
    chroms = synthetic.WHOLE_GENOME
    rows = {c: bench.dump_rows(synthetic.num_windows(c), len(chroms), synthetic.chrom_index(c)) for c in chroms}
    for c, r in rows.items():
        assert np.all(np.diff(r) > 0) and 0 <= r[0] and r[-1] < synthetic.num_windows(c)
    assert rows["chr1"][:4].tolist() == [9, 97, 111, 197] and rows["chr22"][:4].tolist() == [2, 13, 14, 28]
    assert sum(r.size for r in rows.values()) * bench.NCLASS * 4 <= bench.DUMP_PROB_BYTES <= 48 << 20
    for world in (1, 2, 8):
        st = [bench.dump_rows(e - b, world, rank) for rank, (b, e) in enumerate(row_partition(bench.ST_ROWS, world))]
        assert sum(r.size for r in st) * bench.NCLASS * 4 <= bench.DUMP_PROB_BYTES
    assert bench.dump_rows(bench.ST_ROWS // 2, 2, 1)[:4].tolist() == [5, 7, 9, 22]
    assert np.array_equal(bench.dump_rows(10, 23, 0), np.arange(10))          # small graphs are written whole


def test_reference_arm_runs_on_the_host_and_prints_one_line():
    env = dict(os.environ, OMP_NUM_THREADS="4")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload", "c1", "--steps", "1",
                          "--warmup", "0"], capture_output=True, text=True, timeout=600, cwd=ROOT, env=env)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "GE/s" and d["value"] > 0 and d["gpu_launches"] == 0
    assert d["e2e"] == {"value": d["value"], "unit": "GE/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    b = d["cpu_baseline"]
    assert b["kind"] == "port" and b["cores"] >= 1 and b["value"] == d["value"] and "sample" in b
    # ranks other than 0 print nothing and exit 0
    env["RANK"] = "1"
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload", "c1", "--steps", "1"],
                         capture_output=True, text=True, timeout=120, cwd=ROOT, env=env)
    assert out.returncode == 0 and not [l for l in out.stdout.splitlines() if l.startswith("{")]
