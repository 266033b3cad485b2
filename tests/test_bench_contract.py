"""bench.py contract (task statement, sections "Measurement" and "How to work"), checked on the CPU:
the reference arm really runs here (it is the reference's CPU implementation, no GPU involved), and
the committed bench lines under profiles/ carry every key the driver and the judge read."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BASE_KEYS = {"metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better",
             "scaling", "vs_baseline", "dtype", "data", "config"}


def _line(path):
    with open(path) as f:
        return json.loads([l for l in f if l.startswith("{")][0])


def test_reference_arm_runs_on_the_host_and_prints_one_json_line():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "2",
                        "--warmup", "1", "--ref-step", "200000"], capture_output=True, text=True, timeout=600,
                       cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, "stdout must hold exactly one JSON line"
    d = json.loads(lines[0])
    assert BASE_KEYS <= set(d) and d["impl"] == "reference" and d["steps"] == 2 and d["warmup"] == 1
    assert d["metric"] == "incr_mops_c2" and d["unit"] == "Mops/s" and d["higher_is_better"] is True
    assert "workload" in d["config"] and d["value"] > 0
    cb = d["cpu_baseline"]
    assert cb["kind"] in ("reference", "port") and cb["cores"] >= 1 and cb["sample"] and cb["value"] == d["value"]
    e = d["e2e"]
    assert e["value"] == d["value"] and e["unit"] == d["unit"]
    assert e["h2d_bytes_per_step"] == 0 and e["d2h_bytes_per_step"] == 0


@pytest.mark.parametrize("n", [1, 2, 4, 8])
def test_committed_bench_lines_carry_the_contract_keys(n):
    d = _line(os.path.join(ROOT, "profiles", f"r1_bench_n{n}.json"))
    assert BASE_KEYS <= set(d)
    assert d["metric"] == "incr_mops_c2" and d["unit"] == "Mops/s" and d["n_gpus"] == n
    assert d["scaling"] == "weak" and d["vs_baseline"] is None and d["data"] == "synthetic" and d["dtype"] == "u32"
    assert d["warmup"] >= 3 and abs(d["ms_per_step"] * d["steps"] * d["value"] * 1e3
                                    - d["config"]["timed_ops"]) < 1e-6 * d["config"]["timed_ops"]
    assert d["gpu_launches"] > 0
    c = d["clocks"]
    assert c["sm_mhz"] > 0.9 * c["sm_max_mhz"]
    assert not set(c["reasons"]) & {"hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown"}
    r = d["roofline"]
    assert r["bound"] == "hbm" and r["unit"] == "GB/s" and abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-9
    assert r["traffic"] is None or r["traffic"] > 0
    k = d["checks"]                   # full-size invariants: every op added 1, odd queries all miss
    assert k["value_sum_ok"] and k["hit_fraction_exact"] and k["rows_ok"] and k["value_sum"] == k["ops_applied"]
    if n == 1:
        e = d["e2e"]
        assert e["h2d_bytes_per_step"] == 8 * d["config"]["ops_per_step"] and e["d2h_bytes_per_step"] > 0
        assert 0 < e["value"] < d["value"]         # host buffers can only be slower than resident ones
        cb = d["cpu_baseline"]
        assert cb["kind"] == "reference" and cb["cores"] >= 1 and cb["value"] > 0 and cb["sample"]
        assert r["random_sector"]["incr_frac"] > 0.4          # north_star: >= 40 % of the random-sector roofline


ROUND2 = [("r2_bench_n1.json", "incr_mops_c2", 1), ("r2_bench_n1_steps20.json", "incr_mops_c2", 1),
          ("r2_bench_c3_n1.json", "incr_mops_c3", 1), ("r2_bench_c4_n1.json", "getrow_mpairs_c4", 1),
          ("r2_bench_n2.json", "incr_mops_c2", 2), ("r2_bench_n8.json", "incr_mops_c2", 8),
          ("r2_bench_c5_n2.json", "incr_mops_c5", 2), ("r2_bench_c5_n8.json", "incr_mops_c5", 8),
          # the final build of the round (256-slice write chunks, slice-ordered point reads)
          ("r2h_bench_n1_steps20.json", "incr_mops_c2", 1), ("r2h_bench_c3_n1.json", "incr_mops_c3", 1)]


@pytest.mark.parametrize("name,metric,n", ROUND2)
def test_round2_bench_lines(name, metric, n):
    """Every committed round-2 line: the contract keys, zero parity mismatches against the CPU reference
    (incl. sharded getrow at N > 1), the size-independent checks, roofline + e2e + cpu_baseline present."""
    path = os.path.join(ROOT, "profiles", name)
    if not os.path.exists(path):
        pytest.skip(f"{name} not recorded yet")
    d = _line(path)
    assert BASE_KEYS <= set(d) and d["metric"] == metric and d["n_gpus"] == n
    assert d["vs_baseline"] is None and d["data"] == "synthetic" and d["dtype"] == "u32" and d["warmup"] >= 3
    assert "workload" in d["config"] and d["gpu_launches"] > 0 and d["value"] > 0
    c = d["clocks"]
    assert not set(c["reasons"]) & {"hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown"}
    p = d["parity"]
    assert p["mismatches"] == 0 and p["ranks"] == n and p["checker"] == "reference"
    assert p["gets"] > 0 and p["rowlens"] > 0 and p["getrow_pairs"] > 0
    assert all(v for k, v in d["checks"].items() if k.endswith("_ok") or k.endswith("_exact"))
    r = d["roofline"]
    assert r["bound"] == "hbm" and r["unit"] == "GB/s" and abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-9
    e = d["e2e"]
    assert e["value"] > 0 and e["h2d_bytes_per_step"] > 0 and e["d2h_bytes_per_step"] > 0 and e["value"] < d["value"]
    cb = d["cpu_baseline"]
    assert cb["kind"] == "reference" and cb["cores"] >= 1 and cb["value"] > 0 and cb["sample"]
    if n > 1:
        assert r["nvlink"]["remote_bytes_per_rank_per_step"] > 0 and d["scaling"] in ("weak", "strong")
    if metric == "incr_mops_c2" and n == 1:
        assert r["random_sector"]["incr_frac"] > 0.4          # north_star: >= 40 % of the random-sector roofline
    if name.startswith("r2h_"):
        g = r["get"]        # the slice-ordered look-ups answered every query, with the answers of the input order, faster
        assert g["sliced_fraction"] == 1.0 and g["input_order"]["same_answers"] and d["checks"]["get_orders_agree"]
        assert d["get_mops"] > 1.5 * g["input_order"]["get_mops"]


def _bench_dump(tmp_path, *args):
    out = tmp_path / "dump"
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--warmup", "1", "--no-e2e", "--no-cpu",
                        "--no-probes", "--no-parity", "--dump-outputs", str(out), *args],
                       capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    d = json.loads(r.stdout.strip().splitlines()[-1])
    assert sum(f.stat().st_size for f in out.iterdir()) <= 64 << 20
    import numpy as np
    got = {f.name[:-4]: np.load(f) for f in out.iterdir()}
    assert all(a.dtype == np.float64 for a in got.values())
    return d, got


def _counts(keys, q):
    """How often every query key occurs in the build stream = its cell value (every op adds 1)."""
    import numpy as np
    uk, cnt = np.unique(keys, return_counts=True)
    pos = np.minimum(np.searchsorted(uk, q), len(uk) - 1)
    return np.where(uk[pos] == q, cnt[pos], 0)


@pytest.mark.gpu
@pytest.mark.parametrize("wl", ["c2", "c3"])
def test_dump_outputs_of_the_write_workloads_are_the_streams_answers(tmp_path, wl):
    """--dump-outputs on a small write workload with --steps past the workload's own length (c2: 20 batches,
    c3: 11): the step count is honoured, and the dumped cells of the last batch and the sampled get answers equal
    the counts of their keys in the whole build stream, generated again on the host by the CPU checker."""
    import numpy as np
    sys.path.insert(0, ROOT)
    import bench
    from libsmatrix_b200.workloads import zipf_thresholds
    from oracle import cpu
    B, K = 1 << 20, {"c2": 24, "c3": 12}[wl]
    d, got = _bench_dump(tmp_path, "--workload", wl, "--steps", str(K), "--scale", "0.01", "--batch", str(B))
    assert set(got) == {"incr_values", "get_values"}
    assert d["steps"] == K and d["checks"]["ops_applied"] == K * B and d["checks"]["value_sum_ok"]
    cfg, rows, G = bench.WORKLOADS[wl], d["config"]["rows"], d["config"]["gets"]
    if wl == "c2":
        xs, ys = cpu.gen_c2_ops(cfg["seed"], 0, K * B, rows, cfg["ycols"])
        qx, qy = cpu.gen_c2_queries(cfg["seed_get"], cfg["seed"], 0, G, K * B, rows, cfg["ycols"])
    else:
        thr = zipf_thresholds(rows, cfg["zipf_s"])
        xs, ys = cpu.gen_c3_ops(cfg["seed"], 0, K * B, thr)
        qx, qy = cpu.gen_c3_queries(cfg["seed_get"], cfg["seed"], 0, G, K * B, thr)
    keys = xs.astype(np.uint64) << np.uint64(32) | ys
    last = keys[(K - 1) * B:][bench.dump_index(B)]
    assert (got["incr_values"] == _counts(keys, last)).all() and (got["incr_values"] >= 1).all()
    idx = bench.dump_index(G)
    q = (qx.astype(np.uint64) << np.uint64(32) | qy)[idx]
    assert (got["get_values"] == _counts(keys, q)).all()
    assert (got["get_values"][idx % 2 == 1] == 0).all() and (got["get_values"][idx % 2 == 0] >= 1).all()


@pytest.mark.gpu
def test_dump_outputs_of_the_read_workload_are_the_last_steps_rows(tmp_path):
    """--dump-outputs on a small c4 run: the last step's rowlens are the generated row lengths, and the sampled
    rows' getrow pairs, column-sorted, are the (column, value) ops the host generator wrote into them."""
    import numpy as np
    sys.path.insert(0, ROOT)
    import bench
    from libsmatrix_b200.workloads import zipf_thresholds
    from oracle import cpu
    K = 4
    d, got = _bench_dump(tmp_path, "--workload", "c4", "--steps", str(K), "--scale", "0.02")
    assert set(got) == {"rowlen", "getrow_lengths", "getrow_pairs"} and d["steps"] == K
    cfg, R = bench.WORKLOADS["c4"], d["config"]["rows"]
    thr = zipf_thresholds(d["config"]["kmax"], cfg["zipf_s"])
    lens = cpu.gen_c4_lens(cfg["seed"], 0, R, thr).astype(np.uint64)
    offs = np.concatenate([[0], np.cumsum(lens)]).astype(np.uint64)
    lo, hi = (K - 1) * R // K, R
    assert (got["rowlen"] == lens[lo:hi][bench.dump_index(hi - lo)]).all()
    rows = lo + bench.dump_index(hi - lo, 1 << 16)[:len(got["getrow_lengths"])]
    assert len(rows) > 0 and (got["getrow_lengths"] == lens[rows]).all()
    _, ys, vs = cpu.gen_c4_ops(cfg["seed"], int(offs[lo]), int(offs[hi] - offs[lo]), offs)
    at = np.concatenate([np.arange(offs[r], offs[r + 1]) for r in rows]).astype(np.int64) - int(offs[lo])
    row_of = np.repeat(np.arange(len(rows)), lens[rows].astype(np.int64))
    order = np.lexsort((ys[at], row_of))
    assert (got["getrow_pairs"] == np.stack([ys[at][order], vs[at][order]], 1)).all()


def test_full_scale_parity_record():
    d = json.load(open(os.path.join(ROOT, "profiles", "r2_fullscale_parity.json")))
    assert d["ok"] and d["row_digest_mismatches"] == 0 and d["get_mismatches"] == 0
    assert d["rows_checked"] == 13_000_000 and d["pairs_compared"] == d["gpu_nnz"] == 1_510_576_950
    d = json.load(open(os.path.join(ROOT, "profiles", "r1_fullscale_parity.json")))
    assert d["ok"] and d["row_digest_mismatches"] == 0 and d["get_mismatches"] == 0
    assert d["rows_checked"] == 13_000_000 and d["pairs_compared"] == d["gpu_nnz"] == 1_510_576_950
