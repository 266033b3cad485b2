"""Basket recommendations on the config-3 table (bench size: 4 M items, 2^24 baskets, built on the device).

Two sets of baskets: 2^10 of the config-3 stream's own (basket i = the 8 Zipf items of build ops 64 i .. 64 i + 63:
item 1 is in about two thirds of them, so one call aggregates some 10^9 pairs; 2^16 of them would be some 10^11 pairs
per call) and 2^16 baskets of 8 uniform random items.  For k = 10 and 100, after a warm-up call,
the script reports:
  - cf_recommend_batch with device outputs, timed with CUDA events on the library's stream, and the aggregated input
    pairs (the rows of every position) per second; cudaMalloc calls during the timed calls (`allocs`);
  - the split of one call's kernel time between rows + scores, aggregation and ranking (torch.profiler, a run of
    its own; the prefix scans are shared by the stages and listed apart);
  - the same call with host outputs (wall clock) and the bytes that came down;
  - the baseline on the first BASELINE baskets: cf_neighbors_batch with device outputs, then a torch segmented sum
    (index_add_, whose additions are not in a fixed order) and ranking; compared by counts and id sets only.
Writes one JSON to profiles/ (or the path given as argv[1]) with the card's name and power limit read in the same run.

    python scripts/cf_recommend_scale.py [out.json]
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
from test_cf_recommend import stream_baskets  # noqa: E402
from test_cf_topk import build_c3  # noqa: E402

SETS = {"stream": 1 << 10, "uniform": 1 << 16}                     # baskets per set
BASELINE = 256


def log(*a):
    print(*a, flush=True)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q[0] if q else "unknown"


def lib_ms(m, fn):
    m.timer_start()
    fn()
    return m.timer_stop_ms()


def baseline(m, off, items, k, chunk=32):
    """cf_neighbors_batch into device tensors, then a torch segmented sum by (basket, id) and ranking."""
    n = len(off) - 1
    counts = torch.zeros(n, dtype=torch.int32, device="cuda")
    ids = torch.full((n, k), -1, dtype=torch.int32, device="cuda")
    scores = torch.full((n, k), -1.0, dtype=torch.float64, device="cuda")
    for b0 in range(0, n, chunk):
        b1 = min(n, b0 + chunk)
        it = torch.from_numpy(items[off[b0]:off[b1]].view(np.int32)).cuda()
        npos = it.numel()
        loff = torch.empty(npos + 1, dtype=torch.int64, device="cuda")
        total = int(m._lib.smatrix_cf_neighbors_batch(m._handle(), it.data_ptr(), npos, loff.data_ptr(), None, None, 0))
        nb = torch.empty(max(total, 1), dtype=torch.int32, device="cuda")
        sc = torch.empty(max(total, 1), dtype=torch.float64, device="cuda")
        m._lib.smatrix_cf_neighbors_batch(m._handle(), it.data_ptr(), npos, loff.data_ptr(), nb.data_ptr(),
                                          sc.data_ptr(), max(total, 1))
        nb, sc = nb[:total].to(torch.int64) & 0xFFFFFFFF, sc[:total]
        bl = torch.from_numpy(np.diff(off[b0:b1 + 1]).astype(np.int64)).cuda()
        pos_basket = torch.repeat_interleave(torch.arange(b1 - b0, device="cuda"), bl)
        pair_basket = torch.repeat_interleave(pos_basket, loff[1:] - loff[:-1])
        keys, inv = torch.unique(pair_basket * (1 << 32) + nb, return_inverse=True)
        sums = torch.zeros(keys.numel(), dtype=torch.float64, device="cuda").index_add_(0, inv, sc)
        own = pos_basket * (1 << 32) + (it.to(torch.int64) & 0xFFFFFFFF)
        keep = ((keys & 0xFFFFFFFF) != 0) & ~torch.isin(keys, own)
        keys, sums = keys[keep], sums[keep]
        kb, kid = keys >> 32, keys & 0xFFFFFFFF
        o = torch.argsort(kid, stable=True)
        o = o[torch.argsort(-sums[o], stable=True)]
        o = o[torch.argsort(kb[o], stable=True)]
        kb, kid, sums = kb[o], kid[o], sums[o]
        cnt = torch.bincount(kb, minlength=b1 - b0)
        start = torch.cumsum(cnt, 0) - cnt
        rank = torch.arange(kb.numel(), device="cuda") - start[kb]
        sel = rank < k
        ids[b0 + kb[sel], rank[sel]] = kid[sel].to(torch.int32)
        scores[b0 + kb[sel], rank[sel]] = sums[sel]
        counts[b0:b1] = torch.clamp(cnt, max=k).to(torch.int32)
    return counts, ids, scores


def compare_baseline(m, r, off, items, k):
    """The library and the baseline on the first BASELINE baskets: times, counts, id sets."""
    boff, bitems = off[:BASELINE + 1], items[:8 * BASELINE]
    sub = lambda: m.cf_recommend_batch(torch.from_numpy(boff.astype(np.int64)).cuda(),
                                       torch.from_numpy(bitems.view(np.int32)).cuda(), k)
    sub(); baseline(m, boff, bitems, k)                          # warm-ups
    torch.cuda.synchronize(); t1 = time.perf_counter(); lc, li, ls = sub(); torch.cuda.synchronize()
    r["subset_library_ms"] = round((time.perf_counter() - t1) * 1e3, 3)
    torch.cuda.synchronize(); t1 = time.perf_counter(); bc, bi, bs = baseline(m, boff, bitems, k)
    torch.cuda.synchronize()
    r["subset_baseline_ms"] = round((time.perf_counter() - t1) * 1e3, 3)
    lc, li, ls, bc, bi, bs = (x.cpu().numpy() for x in (lc, li, ls, bc, bi, bs))
    same_sets = [set(li[j][:lc[j]].tolist()) == set(bi[j][:bc[j]].tolist()) for j in range(BASELINE)]
    r["subset_counts_equal"] = bool((lc == bc).all())
    r["subset_id_sets_equal_fraction"] = round(float(np.mean(same_sets)), 5)
    both = [j for j in range(BASELINE) if same_sets[j] and (li[j][:lc[j]] == bi[j][:bc[j]]).all()]
    diff = max([float(np.abs(ls[j][:lc[j]] - bs[j][:bc[j]]).max()) for j in both if lc[j]] or [0.0])
    r["subset_max_abs_score_diff_same_order"] = diff


def kernel_split(m, fn):
    """Kernel time of one call by stage (torch.profiler with CUDA activities)."""
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    split = {"rows_scores_ms": 0.0, "aggregation_ms": 0.0, "ranking_ms": 0.0, "scans_ms": 0.0, "other_ms": 0.0}
    for e in prof.key_averages():
        t = e.device_time_total / 1e3 if hasattr(e, "device_time_total") else e.cuda_time_total / 1e3
        name = e.key
        if "k_rec_" in name or "RadixSort" in name or "Onesweep" in name:
            split["aggregation_ms"] += t
        elif "k_topk_" in name:
            split["ranking_ms"] += t
        elif "k_row_counts" in name or "k_getrow" in name or "k_cf_scores" in name:
            split["rows_scores_ms"] += t
        elif "k_scan_" in name:
            split["scans_ms"] += t
        elif name.startswith("k_") or "Kernel" in name or "kernel" in name:
            split["other_ms"] += t
    return {a: round(b, 3) for a, b in split.items()}


def main():
    out = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "profiles", "cf_recommend_scale.json")
    res = {"card": card(), "table": "config 3: 4 M items, 2^24 baskets of 8 (Zipf 1.1), built on the device",
           "baskets": SETS, "baseline_baskets": BASELINE}
    m = SparseMatrix(arena_gib=40)
    t0 = time.perf_counter()
    build_c3(m)
    m.sync()
    res["build_s"] = round(time.perf_counter() - t0, 2)
    log("built", res["build_s"], "s")
    rng = np.random.default_rng(17)
    sets = {"stream": stream_baskets(m, 0, SETS["stream"]),
            "uniform": rng.integers(1, 4_000_001, 8 * SETS["uniform"]).astype(np.uint32)}
    for name, items in sets.items():
        N_BASKETS = SETS[name]
        off = np.arange(0, 8 * N_BASKETS + 1, 8, dtype=np.uint64)
        d_off = torch.from_numpy(off.astype(np.int64)).cuda()
        d_items = torch.from_numpy(items.view(np.int32)).cuda()
        loff = torch.empty(len(items) + 1, dtype=torch.int64, device="cuda")
        pairs = int(m._lib.smatrix_cf_neighbors_batch(m._handle(), d_items.data_ptr(), len(items), loff.data_ptr(),
                                                      None, None, 0))
        log(name, N_BASKETS, "baskets,", pairs, "input pairs")
        for k in (10, 100):
            r = {"baskets": N_BASKETS, "k": k, "input_pairs": pairs,
                 "baskets_with_item_1": int((items.reshape(-1, 8) == 1).any(1).sum())}
            c = torch.empty(N_BASKETS, dtype=torch.int32, device="cuda")
            ids = torch.empty((N_BASKETS, k), dtype=torch.int32, device="cuda")
            s = torch.empty((N_BASKETS, k), dtype=torch.float64, device="cuda")
            call = lambda: m._lib.smatrix_cf_recommend_batch(m._handle(), d_off.data_ptr(), d_items.data_ptr(),
                                                             N_BASKETS, k, c.data_ptr(), ids.data_ptr(), s.data_ptr())
            b0 = m.stat("rec_big")
            call()                                                       # warm-up: scratch sized, modules loaded
            r["rec_big_per_call"] = m.stat("rec_big") - b0
            log(name, k, "warm-up done")
            a0 = m.stat("allocs")
            r["device_ms"] = [round(lib_ms(m, call), 3) for _ in range(3)]
            r["allocs_in_timed_calls"] = m.stat("allocs") - a0
            r["input_pairs_per_s"] = round(pairs / (min(r["device_ms"]) / 1e3), 1)
            log(name, k, "device", r["device_ms"])
            if k == 10:
                r["kernel_split"] = kernel_split(m, call)
                log(name, k, "split", r["kernel_split"])
            h0 = m.stat("d2h_bytes"); t1 = time.perf_counter()
            got = m.cf_recommend_batch(off, items, k)
            r["host_ms"] = round((time.perf_counter() - t1) * 1e3, 3)
            r["host_d2h_bytes"] = m.stat("d2h_bytes") - h0
            r["host_answer_bytes"] = N_BASKETS * (12 * k + 4)
            r["host_equals_device"] = bool((got[0] == c.cpu().numpy().view(np.uint32)).all()
                                           and (got[1] == ids.cpu().numpy().view(np.uint32)).all()
                                           and (got[2].view(np.uint64) == s.cpu().numpy().view(np.uint64)).all())
            # the baseline on the first BASELINE baskets, and the library on the same baskets
            log(name, k, "host", r["host_ms"])
            try:
                compare_baseline(m, r, off, items, k)
            except Exception as e:                                       # noqa: BLE001 - recorded, the run goes on
                r["baseline_error"] = repr(e)
            res[f"{name}_k{k}"] = r
            print(json.dumps(r), flush=True)
            save(res, out)                                               # after every result: a cut-short run keeps them
    m.close()
    print(json.dumps({"card": res["card"], "out": out}))


def save(res, out):
    os.makedirs(os.path.dirname(os.path.abspath(out)), exist_ok=True)
    with open(out, "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
