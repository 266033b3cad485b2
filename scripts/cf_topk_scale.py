"""Top-k recommender queries on the config-3 table (bench size: 4 M items, 2^24 baskets, built on the device).

For the 10 000 hottest items and 100 000 random ones, after a warm-up call of each kind, times with CUDA events
on the library's stream:
  1. cf_topk_batch with device outputs;
  2. the baseline: cf_neighbors_batch with device outputs, then a torch segmented ranking of its output
     (three stable sorts; timed with events on torch's stream);
  3. both with host outputs (wall clock around the synchronous calls), with the bytes that came down.
Writes one JSON to profiles/ (or the path given as argv[1]) with the card's name and power limit read in the same run.

    python scripts/cf_topk_scale.py [out.json]
"""
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np  # noqa: E402
import torch  # noqa: E402

from libsmatrix_b200 import SparseMatrix  # noqa: E402
from test_cf_topk import build_c3, rank_segments  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q[0] if q else "unknown"


def lib_ms(m, fn):
    m.timer_start()
    fn()
    return m.timer_stop_ms()


def main():
    out = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "profiles", "cf_topk_scale.json")
    res = {"card": card(), "table": "config 3: 4 M items, 2^24 baskets of 8 (Zipf 1.1), built on the device"}
    m = SparseMatrix(arena_gib=40)
    t0 = time.perf_counter()
    build_c3(m)
    m.sync()
    res["build_s"] = round(time.perf_counter() - t0, 2)
    res["rowlen_item1"] = int(m.rowlen(1))
    rng = np.random.default_rng(12)
    sets = {"hottest_10k": np.arange(1, 10_001, dtype=np.uint32),
            "random_100k": rng.integers(1, 4_000_001, 100_000).astype(np.uint32)}
    for name, items in sets.items():
        d_items = torch.from_numpy(items.view(np.int32)).cuda()
        n = len(items)
        off = torch.empty(n + 1, dtype=torch.int64, device="cuda")
        total = int(m._lib.smatrix_cf_neighbors_batch(m._handle(), d_items.data_ptr(), n, off.data_ptr(), None, None, 0))
        nb = torch.empty(total, dtype=torch.int32, device="cuda")
        sc = torch.empty(total, dtype=torch.float64, device="cuda")
        for k in (10, 100):
            r = {"items": n, "k": k, "pairs": total}
            c = torch.empty(n, dtype=torch.int32, device="cuda")
            ids = torch.empty((n, k), dtype=torch.int32, device="cuda")
            s = torch.empty((n, k), dtype=torch.float64, device="cuda")
            topk = lambda: m._lib.smatrix_cf_topk_batch(m._handle(), d_items.data_ptr(), n, k, c.data_ptr(),
                                                        ids.data_ptr(), s.data_ptr())
            neigh = lambda: m._lib.smatrix_cf_neighbors_batch(m._handle(), d_items.data_ptr(), n, off.data_ptr(),
                                                              nb.data_ptr(), sc.data_ptr(), total)
            topk(); neigh()                                              # warm-up: scratch sized, modules loaded
            a0 = m.stat("allocs")
            r["topk_device_ms"] = [round(lib_ms(m, topk), 3) for _ in range(3)]
            r["allocs_in_timed_calls"] = m.stat("allocs") - a0
            r["neighbors_device_ms"] = [round(lib_ms(m, neigh), 3) for _ in range(3)]
            rank_segments(m, d_items, k)                                 # warm-up of the torch ranking
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); want = rank_segments(m, d_items, k); e1.record(); torch.cuda.synchronize()
            r["baseline_neighbors_plus_torch_rank_ms"] = round(e0.elapsed_time(e1), 3)
            got = (c, ids, s.view(torch.int64))
            r["equal_to_baseline"] = all(torch.equal(g, w) for g, w in zip(got, (want[0], want[1], want[2].view(torch.int64))))
            h0 = m.stat("d2h_bytes"); t1 = time.perf_counter()
            m.cf_topk_batch(items, k)
            r["topk_host_ms"] = round((time.perf_counter() - t1) * 1e3, 3)
            r["topk_host_d2h_bytes"] = m.stat("d2h_bytes") - h0
            h0 = m.stat("d2h_bytes"); t1 = time.perf_counter()
            m.cf_neighbors_batch(items)
            r["neighbors_host_ms"] = round((time.perf_counter() - t1) * 1e3, 3)
            r["neighbors_host_d2h_bytes"] = m.stat("d2h_bytes") - h0
            r["topk_big"], r["topk_passes"] = m.stat("topk_big"), m.stat("topk_passes")
            res[f"{name}_k{k}"] = r
            print(json.dumps(r), flush=True)
        del nb, sc
    m.close()
    os.makedirs(os.path.dirname(out), exist_ok=True)
    with open(out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({"card": res["card"], "out": out}))


if __name__ == "__main__":
    main()
