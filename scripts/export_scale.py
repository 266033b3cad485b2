"""Matrix enumeration at bench size on one GPU: the config-2 table (13 M rows, 2 * 10^9 incr ops over 256 columns)
and the config-4 table (13 M rows with Zipf(1.7) lengths up to 10^6, about 1.4 * 10^9 pairs, half of them in rows
longer than 10^5 columns), both built on the device.

For each table, after a warm-up call of each kind, the script reports:
  - list_rows of all rows into a device tensor (rows(device=True));
  - getrow of every row, device to device, unsorted (smatrix_getrow_batch) and sorted (smatrix_getrow_sorted_batch),
    the same rows in the same order into the same buffer, in Gpairs/s; 10^4 sampled sorted rows are checked against
    the unsorted ones sorted on the host;
  - the sort pass alone per size class: smatrix_b200_sort_rows over the CSR of the rows of one class (warp: <= 256
    pairs, block: <= 4096, radix: longer), in Gpairs/s;
  - the full paged export (iter_rows, pages of 2^20 rows) device to device, and into host memory (numpy).
Call times come from the library's CUDA-event timer on its own stream; the calls end in a synchronise, so the paged
exports are timed with the host clock.  Writes one JSON to profiles/export_scale.json (or argv[1]) with the card's
name and power limit read in the same run.

    python scripts/export_scale.py [out.json]
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
from test_export import build_c4  # noqa: E402

CLASSES = {"warp": (2, 256), "block": (257, 4096), "radix": (4097, 1 << 32)}   # pairs per row (1-pair rows: no sort)
PAGE = 1 << 20


def log(*a):
    print(*a, flush=True)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q[0] if q else "unknown"


def lib_ms(m, fn, reps=1):
    fn()                                             # warm-up: scratch, module load
    m.timer_start()
    for _ in range(reps):
        fn()
    return m.timer_stop_ms() / reps


def build_c2(m, rows=13_000_000, ycols=256, total=2_000_000_000, seed=2):
    B = 1 << 26
    xs = torch.empty(B, dtype=torch.int32, device="cuda")
    ys = torch.empty(B, dtype=torch.int32, device="cuda")
    for first in range(0, total, B):
        n = min(B, total - first)
        m.gen_c2_ops(seed, first, n, rows, ycols, xs.data_ptr(), ys.data_ptr())
        m.incr_batch(xs[:n], ys[:n], None)


def getrow_into(m, fn, keys, off, pairs):
    total = int(fn(m._handle(), keys.data_ptr(), keys.numel(), off.data_ptr(), pairs.data_ptr(), pairs.numel() // 2))
    assert total * 2 <= pairs.numel()
    return total


def measure(m, name):
    r = {"table": name, "rows": m.stat("rows"), "nnz": m.stat("nnz")}
    lib = m._lib
    keys = m.rows(device=True)
    assert keys.numel() == r["rows"]
    r["list_rows_ms"] = lib_ms(m, lambda: m.rows(device=True), reps=5)
    n = keys.numel()
    off = torch.empty(n + 1, dtype=torch.int64, device="cuda")
    total = int(lib.smatrix_getrow_batch(m._handle(), keys.data_ptr(), n, None, None, 0))
    assert total == r["nnz"]
    pairs = torch.empty(2 * total, dtype=torch.int32, device="cuda")
    t_u = lib_ms(m, lambda: getrow_into(m, lib.smatrix_getrow_batch, keys, off, pairs))
    rng = np.random.default_rng(1)
    pick = np.sort(rng.choice(n, 10_000, replace=False))
    h_off = off.cpu().numpy()
    unsorted = [pairs[2 * h_off[i]:2 * h_off[i + 1]].cpu().numpy().view(np.uint32).reshape(-1, 2) for i in pick]
    b0 = m.stat("sort_big")
    t_s = lib_ms(m, lambda: getrow_into(m, lib.smatrix_getrow_sorted_batch, keys, off, pairs))
    r["sort_big_per_call"] = (m.stat("sort_big") - b0) // 2
    for i, u in zip(pick, unsorted):
        got = pairs[2 * h_off[i]:2 * h_off[i + 1]].cpu().numpy().view(np.uint32).reshape(-1, 2)
        assert (got == u[np.argsort(u[:, 0], kind="stable")]).all(), f"row {i}"
    r["getrow_all"] = {"pairs": total, "unsorted_ms": t_u, "sorted_ms": t_s,
                       "unsorted_gpairs_s": total / t_u / 1e6, "sorted_gpairs_s": total / t_s / 1e6,
                       "checked_rows": len(pick)}
    lens = (off[1:] - off[:-1]).cpu().numpy()
    del pairs
    torch.cuda.empty_cache()
    r["classes"] = {}
    for cname, (lo, hi) in CLASSES.items():
        sel = np.flatnonzero((lens >= lo) & (lens <= hi))
        if not len(sel):
            continue
        ck = keys[torch.from_numpy(sel).cuda()]
        coff = torch.empty(len(sel) + 1, dtype=torch.int64, device="cuda")
        ctotal = int(lib.smatrix_getrow_batch(m._handle(), ck.data_ptr(), len(sel), None, None, 0))
        cpairs = torch.empty(2 * ctotal, dtype=torch.int32, device="cuda")
        getrow_into(m, lib.smatrix_getrow_batch, ck, coff, cpairs)
        ms = lib_ms(m, lambda: lib.smatrix_b200_sort_rows(m._handle(), len(sel), coff.data_ptr(), cpairs.data_ptr()),
                    reps=3)
        r["classes"][cname] = {"rows": len(sel), "pairs": ctotal, "sort_ms": ms, "gpairs_s": ctotal / ms / 1e6}
        log(name, cname, r["classes"][cname])
        del ck, coff, cpairs
        torch.cuda.empty_cache()
    for dev in (True, False):
        sum(k.shape[0] for k, _, _ in m.iter_rows(0, PAGE, device=dev))       # warm-up
        t0 = time.perf_counter()
        rows = pairs_n = 0
        for k, o, p in m.iter_rows(0, PAGE, device=dev):
            rows += k.shape[0]
            pairs_n += p.shape[0]
        if dev:
            torch.cuda.synchronize()
        s = time.perf_counter() - t0
        assert rows == r["rows"] and pairs_n == r["nnz"]
        r["paged_export_" + ("device" if dev else "host")] = {"page_rows": PAGE, "s": s, "gpairs_s": pairs_n / s / 1e9}
    log(json.dumps(r))
    return r


def main():
    out = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "profiles", "export_scale.json")
    res = {"card": card(), "tables": []}
    log(res["card"])
    for name, build, arena in (("config-2", build_c2, 40), ("config-4", build_c4, 48)):
        m = SparseMatrix(arena_gib=arena)
        t0 = time.perf_counter()
        build(m)
        m.sync()
        log(name, "built in", round(time.perf_counter() - t0, 1), "s")
        res["tables"].append(measure(m, name))
        m.close()
        torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(out), exist_ok=True)
    with open(out, "w") as f:
        json.dump(res, f, indent=1)
    log("wrote", out)


if __name__ == "__main__":
    main()
