#!/usr/bin/env python
"""bench.py — the BASELINE.json workloads on B200 through the C-ABI (SURVEY.md 8d).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload c2|c3|c4|c5]
                    [--dump-outputs DIR]

One JSON line on stdout (rank 0).  Default = the headline, config 2.

  c2  uniform-random batched incr building ~1.5 B nnz over 13 M rows per GPU, then 500 M point gets
      at 50 % hits.  A step = one batch of 2^26 incr ops per GPU; the timed steps are the LAST K
      batches of the 2 B-op stream (K = 30: the whole build from empty; smaller K: the first batches
      are applied untimed, so the timed region still ends at ~1.5 B nnz; larger K: the stream goes on).
  c3  co-occurrence build (examples/cf_recommender.c:35-47): Zipf(1.1) baskets of 8 over 4 M items,
      all-pairs incr + column-0 totals, 2^24 baskets = 1.07 B ops in 16 steps of 2^26; then gets.
  c4  read path: 13 M rows with Zipf(1.7) row lengths 1 .. 10^6 (~1.4 B nnz) are built, then every
      step is rowlen_batch + getrow_batch over 1/K of ALL rows; value = pairs/s.
  c5  row-sharded: 52 M rows in total, y = 1 + r % 170, 10 B incr ops in total over the N >= 2 GPUs.

  value      the metric with all inputs resident in HBM before the timed region starts
  e2e        the same through the C-ABI with HOST (pinned) buffers: H2D of every batch / D2H of every
             answer inside the timed region; byte counts come from the library's own copy counters
  roofline   dominant kernel (k_upsert / k_getrow_fill): algorithmic bytes / launch time measured with
             CUDA events on the library's stream, against MEASURED_PEAKS.json hbm_gbs
  parity     after the timed region: a prefix of the same stream is applied to a fresh matrix through
             the same product path (sharded at N > 1) and compared with the CPU reference op for op:
             gets, rowlens and column-sorted getrows — mismatch counts must be 0
  cpu_baseline / --impl reference   the unmodified reference (the compiled checker under oracle/) on
             the box's host cores over a bounded sample of the same stream
N > 1 (torchrun): rows are hash-partitioned by owner rank; the C router (include/smatrix_shard.h) moves
every rank's slice of a batch to the owners with stores over NVLink; torch.distributed is used only for
the barrier / max-over-ranks around the timed regions.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

SCRAMBLE = 2654435761
GET_BYTES = 76                             # 2 sectors + 8 B in + 4 B out, SURVEY.md 8(d)
INCR_SECTORS, GET_SECTORS = 3, 2           # random 32 B sectors per op
WORKLOADS = {
    # rows / ycols / total ops are PER GPU for c2 (weak scaling) and IN TOTAL for c5 (strong scaling)
    "c2": dict(metric="incr_mops_c2", rows=13_000_000, ycols=256, total_ops=2_000_000_000, gets=500_000_000,
               seed=2, seed_get=3, scaling="weak"),
    "c3": dict(metric="incr_mops_c3", items=4_000_000, zipf_s=1.1, baskets=1 << 24, gets=1 << 28,
               seed=4, seed_get=7, scaling="weak"),
    "c4": dict(metric="getrow_mpairs_c4", rows=13_000_000, zipf_s=1.7, kmax=1_000_000, seed=5, scaling="weak"),
    "c5": dict(metric="incr_mops_c5", rows=52_000_000, ycols=170, total_ops=10_000_000_000, gets=1 << 28,
               seed=6, seed_get=8, scaling="strong"),
}


def parse():
    p = argparse.ArgumentParser()
    p.add_argument("--gpus", type=int, default=1)
    p.add_argument("--steps", type=int, default=None,
                   help="timed steps (default: the whole workload); past the workload's own length the stream goes on and "
                        "the arena grows with it, and all K batches (8 B per op) are resident at once, so device memory "
                        "bounds K (c2 at full scale: 0.5 GiB of batches + 1.7 GiB of arena per step)")
    p.add_argument("--warmup", type=int, default=3)
    p.add_argument("--impl", default="ours", choices=["ours", "reference"])
    p.add_argument("--workload", default="c2", choices=sorted(WORKLOADS))
    p.add_argument("--batch", type=int, default=1 << 26, help="ops per step per GPU")
    p.add_argument("--scale", type=float, default=1.0, help="shrink the workload (rows, ops, gets) for quick checks; "
                   "a scaled run says so in config and is not a headline number")
    p.add_argument("--arena-gib", type=int, default=None,
                   help="slab memory each table reserves at smatrix_open (SMATRIX_ARENA_GIB); default per workload, 0 = on demand")
    p.add_argument("--no-e2e", action="store_true")
    p.add_argument("--no-cpu", action="store_true")
    p.add_argument("--no-probes", action="store_true")
    p.add_argument("--no-parity", action="store_true")
    p.add_argument("--phase-series", action="store_true", help="diagnostic: host phase split of every step on stderr")
    p.add_argument("--cpu-secs", type=float, default=12.0, help="target seconds of CPU work for cpu_baseline")
    p.add_argument("--ref-step", type=int, default=None, help="ops (c4: rows) per step of the reference arm")
    p.add_argument("--parity-ops", type=int, default=3_000_000, help="ops of the parity prefix (whole job)")
    p.add_argument("--dump-outputs", metavar="DIR", default=None,
                   help="after the timed steps, write what the timed path computed in its last step as DIR/<name>.npy "
                        "(float64, fixed seeded samples, at most 64 MB) so that two builds can be compared output for output")
    a = p.parse_args()
    if a.dump_outputs and a.impl != "ours":
        p.error("--dump-outputs records the GPU path: use it with --impl ours")
    return a


# ------------------------------------------------------------------------------ clocks
class ClockSampler:
    """nvidia-smi clocks + throttle reasons DURING the timed region (B200_PROFILING.md)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.rows, self.proc = [], None
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i",
                 str(index), "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [c.strip() for c in line.split(",")]))

    def window(self, t0, t1):
        sel = [r for (t, r) in self.rows if t0 <= t <= t1 and len(r) >= 7] or \
              [r for (_, r) in self.rows[-3:] if len(r) >= 7]
        if not sel:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        sm = sorted(float(r[0]) for r in sel)
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for k, n in enumerate(names) if any(r[3 + k].lower().startswith("active") for r in sel)]
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": float(sel[0][1]), "reasons": reasons,
                "samples": len(sel), "power_w_max": max(float(r[2]) for r in sel)}

    def stop(self):
        if self.proc:
            self.proc.terminate()


def measured_peak_gbs():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


def committed_traffic(key):
    """DRAM bytes per unit of the dominant kernel from the committed ncu capture (profiles/), or None."""
    for name in ("traffic_r2.json", "traffic_r1.json"):
        try:
            with open(os.path.join(ROOT, "profiles", name)) as f:
                d = json.load(f)
            if key in d:
                return float(d[key]), f"profiles/{name}"
        except Exception:
            pass
    return None, None


def thread_candidates():
    n = os.cpu_count() or 1
    return [t for t in (1, 2, 4, 8, 16, 32) if t <= n] or [1]


def scaled(a, v):
    return max(1, int(v * a.scale))


DUMP_SAMPLE = 1 << 21        # entries per dumped array over the whole job (N ranks: 1/N each): 16 MB in float64


def dump_index(n: int, k: int = DUMP_SAMPLE) -> np.ndarray:
    """Sorted positions of a fixed, seeded sample of k out of n outputs (all n when n <= k)."""
    if n <= k:
        return np.arange(n, dtype=np.int64)
    return np.unique(np.random.default_rng(20240611).integers(0, n, k))


def write_dump(job, arrays: dict):
    """--dump-outputs: every array as DIR/<name>.npy in float64 (u32 values and i64 offsets are exact there);
    at N > 1 every rank writes its own share as <name>.rank<r>.npy."""
    os.makedirs(job.a.dump_outputs, exist_ok=True)
    sfx = f".rank{job.rank}" if job.world > 1 else ""
    for name, arr in arrays.items():
        if not isinstance(arr, np.ndarray):
            arr = arr.cpu().numpy()
        if arr.dtype == np.int32:
            arr = arr.view(np.uint32)
        np.save(os.path.join(job.a.dump_outputs, f"{name}{sfx}.npy"), arr.astype(np.float64))


# ====================================================================================================
# CPU legs: cpu_baseline, the reference arm and the parity checker.  The ONLY code that touches oracle/.
# ====================================================================================================
def _host_stream(wl, cfg, first, count, rows_total, tables):
    """ops [first, first + count) of the workload's build stream, generated on the host (the CPU
    checker's own generators — the same counter-based definitions as the device kernels)."""
    from oracle import cpu
    if wl in ("c2", "c5"):
        xs, ys = cpu.gen_c2_ops(cfg["seed"], first, count, rows_total, cfg["ycols"])
        return xs, ys, None
    if wl == "c3":
        xs, ys = cpu.gen_c3_ops(cfg["seed"], first, count, tables["thr"])
        return xs, ys, None
    raise ValueError(wl)


def _host_queries(wl, cfg, first, count, n_build, rows_total, tables):
    from oracle import cpu
    if wl in ("c2", "c5"):
        return cpu.gen_c2_queries(cfg["seed_get"], cfg["seed"], first, count, n_build, rows_total, cfg["ycols"])
    return cpu.gen_c3_queries(cfg["seed_get"], cfg["seed"], first, count, n_build, tables["thr"])


def cpu_write_baseline(wl, cfg, rows_total, tables, n_steps, warm_steps, step_ops, get_ops):
    """The unmodified reference on the host cores: ONE matrix, consecutive prefixes of the build
    stream, `step_ops` per step; the warm-up steps double as the thread-count sweep (the reference
    scales negatively, BASELINE.md 2); then gets.  Arrays are generated outside the timed calls."""
    from oracle import cpu
    cpu.build(ref=True)
    kind = "reference" if cpu.have_reference() else "port"
    m = cpu.CpuMatrix(kind)
    cands = thread_candidates() if kind == "reference" else [1]
    first, sweep = 0, {}
    for w in range(max(warm_steps, len(cands))):
        t = cands[w % len(cands)]
        xs, ys, _ = _host_stream(wl, cfg, first, step_ops, rows_total, tables)
        s = m.bench_apply("incr", t, xs, ys, None)
        sweep.setdefault(t, []).append(step_ops / s / 1e6)
        first += step_ops
    best_t = max(sweep, key=lambda t: max(sweep[t]))
    secs = 0.0
    for _ in range(n_steps):
        xs, ys, _ = _host_stream(wl, cfg, first, step_ops, rows_total, tables)
        secs += m.bench_apply("incr", best_t, xs, ys, None)
        first += step_ops
    qx, qy = _host_queries(wl, cfg, 0, get_ops, first, rows_total, tables)
    gs = m.bench_get(best_t, qx, qy)
    m.close()
    return {"kind": kind, "cores": best_t, "host_cores": os.cpu_count(), "value": n_steps * step_ops / secs / 1e6,
            "get_mops": get_ops / gs / 1e6, "secs": secs, "unit": "Mops/s",
            "sweep_mops": {str(t): round(max(v), 3) for t, v in sweep.items()},
            "sample": f"{wl} stream prefix on one matrix: {n_steps} timed steps x {step_ops} incr ops after "
                      f"{first - n_steps * step_ops} warm-up ops (thread sweep), then {get_ops} gets"}


def c4_tables(cfg, a):
    from libsmatrix_b200.workloads import zipf_thresholds
    return {"thr": zipf_thresholds(scaled(a, cfg["kmax"]) if a.scale < 1 else cfg["kmax"], cfg["zipf_s"])}


def cpu_read_baseline(cfg, tables, rows_sample, n_steps, warm_steps):
    """c4 on the CPU: the reference holds `rows_sample` rows of the same length distribution (it cannot
    build 1.4 B nnz in bench time); every step is rowlen + getrow (full-size buffers) over 1/steps of them."""
    from oracle import cpu
    cpu.build(ref=True)
    kind = "reference" if cpu.have_reference() else "port"
    m = cpu.CpuMatrix(kind)
    lens = cpu.gen_c4_lens(cfg["seed"], 0, rows_sample, tables["thr"])
    offs = np.concatenate([[0], np.cumsum(lens.astype(np.uint64))]).astype(np.uint64)
    xs, ys, vs = cpu.gen_c4_ops(cfg["seed"], 0, int(offs[-1]), offs)
    t0 = time.perf_counter()
    m.bench_apply("incr", 1, xs, ys, vs)
    build_s = time.perf_counter() - t0
    ids = (np.arange(rows_sample, dtype=np.uint64) * SCRAMBLE).astype(np.uint32)
    cands = thread_candidates() if kind == "reference" else [1]
    sweep = {}
    for w in range(max(warm_steps, len(cands))):
        t = cands[w % len(cands)]
        s, pairs = m.bench_getrow(t, ids)
        sweep.setdefault(t, []).append(pairs / s / 1e6)
    best_t = max(sweep, key=lambda t: max(sweep[t]))
    secs, pairs_total = 0.0, 0
    for j in range(n_steps):
        part = ids[j * rows_sample // n_steps:(j + 1) * rows_sample // n_steps]
        s, pairs = m.bench_getrow(best_t, part)
        secs += s
        pairs_total += pairs
    m.close()
    return {"kind": kind, "cores": best_t, "host_cores": os.cpu_count(), "value": pairs_total / secs / 1e6,
            "unit": "Mpairs/s", "secs": secs, "build_mops": len(xs) / build_s / 1e6,
            "sweep_mpairs": {str(t): round(max(v), 3) for t, v in sweep.items()},
            "sample": f"c4 length distribution on {rows_sample} rows ({len(xs)} nnz) held by the reference; "
                      f"{n_steps} timed steps of rowlen + getrow over all of them ({pairs_total} pairs)"}


def main_reference(a):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    wl, cfg = a.workload, WORKLOADS[a.workload]
    K = a.steps or 4
    if wl == "c4":
        tables = c4_tables(cfg, a)
        r = cpu_read_baseline(cfg, tables, a.ref_step or scaled(a, 400_000), K, a.warmup)
        config = {"workload": "c4 read path (rowlen + getrow over all rows), reference CPU path, bounded sample",
                  "rows": a.ref_step or scaled(a, 400_000)}
    else:
        from libsmatrix_b200.workloads import zipf_thresholds
        tables = {"thr": zipf_thresholds(scaled(a, cfg["items"]), cfg["zipf_s"])} if wl == "c3" else {}
        per_gpu = wl == "c2"
        rows_total = scaled(a, cfg.get("rows", 0)) * (a.gpus if per_gpu else 1)
        step = a.ref_step or (2_000_000 if wl != "c3" else 1_000_000)
        r = cpu_write_baseline(wl, cfg, rows_total, tables, K, a.warmup, step, min(2 * step, 4_000_000))
        config = {"workload": f"{wl} build stream (SURVEY.md 8d), reference CPU path, bounded sample",
                  "rows": rows_total, "ops_per_step": step}
    line = {
        "impl": "reference", "metric": cfg["metric"], "value": r["value"], "unit": r["unit"],
        "n_gpus": a.gpus, "steps": K, "warmup": a.warmup, "ms_per_step": r["secs"] / K * 1e3,
        "higher_is_better": True, "scaling": cfg["scaling"], "vs_baseline": None, "dtype": "u32",
        "data": "synthetic", "config": config,
        "cpu_baseline": {k: r[k] for k in r if k != "secs"},
        "e2e": {"value": r["value"], "unit": r["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    if "get_mops" in r:
        line["get_mops"] = r["get_mops"]
    print(json.dumps(line), flush=True)


# ====================================================================================================
# our arm
# ====================================================================================================
class Job:
    """Process-level plumbing shared by the workloads: ranks, device, barrier, matrix factory."""

    def __init__(self, a):
        import torch
        import torch.distributed as dist
        self.a, self.torch, self.dist = a, torch, dist
        self.rank = int(os.environ.get("RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        if self.world != a.gpus and self.world == 1 and a.gpus > 1:
            raise SystemExit("launch N>1 with torchrun (one rank per GPU)")
        torch.cuda.set_device(self.local)
        self.dev = torch.device("cuda", self.local)
        os.environ.pop("SMATRIX_ARENA_GIB", None)
        os.environ.setdefault("SMATRIX_SHARD_TIMEOUT", "1800")
        if self.world > 1:
            os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
            dist.init_process_group("nccl", device_id=self.dev)
        self.sampler = ClockSampler(self.local)
        self.gen = None

    def ibuf(self, n):
        return self.torch.empty(n, dtype=self.torch.int32, device=self.dev)

    def pinned(self, n):
        return self.torch.empty(n, dtype=self.torch.int32, pin_memory=True)

    def barrier(self):
        self.torch.cuda.synchronize()
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max_over_ranks(self, x: float) -> float:
        if self.world == 1:
            return x
        t = self.torch.tensor([x], dtype=self.torch.float64, device=self.dev)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def sum_over_ranks(self, *vals):
        if self.world == 1:
            return [int(v) for v in vals]
        t = self.torch.tensor([int(v) for v in vals], dtype=self.torch.int64, device=self.dev)
        self.dist.all_reduce(t)
        return [int(v) for v in t.tolist()]

    def make_matrix(self, arena_gib: int):
        """The product handle: SparseMatrix at N = 1, the C router's sharded matrix at N > 1.  Only
        handles that hold a table reserve the slab arena."""
        from libsmatrix_b200 import SparseMatrix
        if self.world > 1:
            from libsmatrix_b200.sharded import open_sharded
            return open_sharded(self.rank, self.world, self.local, arena_gib=arena_gib)
        return SparseMatrix(device=self.local, arena_gib=arena_gib)

    def generator(self, m):
        """A single-GPU handle whose stream runs the synthetic-stream kernels (N > 1: a helper handle)."""
        if self.world == 1:
            return m
        if self.gen is None:
            from libsmatrix_b200 import SparseMatrix
            self.gen = SparseMatrix(device=self.local)
        return self.gen

    def finish(self):
        self.sampler.stop()
        if self.gen is not None:
            self.gen.close()
        if self.world > 1:
            self.dist.destroy_process_group()


class WriteWorkload:
    """c2 / c3 / c5: a counter-based stream of incr ops + a query stream over it."""

    def __init__(self, job: Job, name: str):
        a, cfg = job.a, WORKLOADS[name]
        self.job, self.name, self.cfg = job, name, cfg
        self.B = a.batch
        W = job.world
        self.tables, self.d_thr = {}, None
        if name == "c3":
            from libsmatrix_b200.workloads import zipf_thresholds
            self.items = scaled(a, cfg["items"])
            self.tables["thr"] = zipf_thresholds(self.items, cfg["zipf_s"])
            self.d_thr = job.torch.from_numpy(self.tables["thr"].view(np.int64)).to(job.dev)
            total = scaled(a, cfg["baskets"]) * 64 * W           # weak scaling: every GPU adds its own baskets
            self.rows_total = self.items
            self.ordered = True                                  # column-0 ops: order matters for rowlen (Q1)
            self.arena = 40
        elif name == "c2":
            self.rows_total = scaled(a, cfg["rows"]) * W
            total = scaled(a, cfg["total_ops"]) * W
            self.ordered = False
            self.arena = 52
        else:                                                    # c5: fixed total work, N >= 2
            if W < 2:
                raise SystemExit("c5 is the row-sharded workload: run it with --gpus 2, 4 or 8 (6 B nnz do not fit one GPU)")
            self.rows_total = scaled(a, cfg["rows"])
            total = scaled(a, cfg["total_ops"])
            self.ordered = False
            self.arena = {2: 120, 4: 60, 8: 32}.get(W, 32)
        if a.scale < 1:
            self.arena = max(2, int(self.arena * a.scale) + 1)
        if a.arena_gib is not None:
            self.arena = a.arena_gib
        self.n_batches = max(1, -(-total // (self.B * W)))       # batches per rank
        if a.steps and a.steps > self.n_batches:                 # more steps than the workload has: the stream goes on
            if a.arena_gib is None:                              # and the arena grows with the ops it has to hold
                self.arena = -(-self.arena * a.steps // self.n_batches)
            self.n_batches = a.steps
        self.K = a.steps or self.n_batches
        self.prefill = self.n_batches - self.K
        self.gets = scaled(a, cfg["gets"])
        self.n_build = self.n_batches * self.B * W
        self.bytes_per_op = 96 + 8                               # 3 sectors + x, y streamed (vals == NULL: all ones)

    def first_of(self, k):                                       # global op index of (rank, batch k): ranks interleave batch-wise
        return (k * self.job.world + self.job.rank) * self.B

    def gen_ops(self, g, first, count, xs, ys):
        c = self.cfg
        if self.name == "c3":
            g.gen_c3_ops(c["seed"], first, count, self.d_thr.data_ptr(), self.items, xs.data_ptr(), ys.data_ptr())
        else:
            g.gen_c2_ops(c["seed"], first, count, self.rows_total, c["ycols"], xs.data_ptr(), ys.data_ptr())

    def gen_warm(self, g, first, count, xs, ys):
        c = self.cfg
        if self.name == "c3":
            g.gen_c3_ops(99, first, count, self.d_thr.data_ptr(), self.items, xs.data_ptr(), ys.data_ptr())
        else:
            g.gen_c2_ops(99, first, count, self.rows_total, c["ycols"], xs.data_ptr(), ys.data_ptr())

    def gen_queries(self, g, first, count, xs_ptr, ys_ptr):
        c = self.cfg
        if self.name == "c3":
            g.gen_c3_queries(c["seed_get"], c["seed"], first, count, self.n_build, self.d_thr.data_ptr(), self.items,
                             xs_ptr, ys_ptr)
        else:
            g.gen_c2_queries(c["seed_get"], c["seed"], first, count, self.n_build, self.rows_total, c["ycols"],
                             xs_ptr, ys_ptr)

    def incr(self, m, xs, ys):
        if self.job.world > 1:
            m.incr_batch(xs, ys, None, ordered=self.ordered)
        else:
            m.incr_batch(xs, ys, None)

    def describe(self):
        W = self.job.world
        if self.name == "c2":
            return ("C2: uniform-random batched incr, 2^26 ops/step/GPU, building ~1.5 B nnz over 13 M rows per GPU, "
                    "then point gets at 50 % hits (SURVEY.md 8d)")
        if self.name == "c3":
            return ("C3: co-occurrence build (examples/cf_recommender.c:35-47), Zipf(1.1) baskets of 8 over 4 M items, "
                    "all-pairs incr + column-0 totals, 2^24 baskets per GPU, then point gets at 50 % hits")
        return (f"C5: row-sharded uniform incr, 52 M rows and 10 B ops in total over {W} GPUs, y = 1 + r % 170 "
                "(~6 B nnz), then point gets at 50 % hits")


def run_write_workload(job: Job, name: str):
    a, torch = job.a, job.torch
    wl = WriteWorkload(job, name)
    B, K, W, world, rank = wl.B, wl.K, a.warmup, job.world, job.rank
    mk = lambda: job.make_matrix(wl.arena)

    # ---- warm-up on a scratch matrix (W full-size batches from a different seed)
    scratch = mk()
    g = job.generator(scratch)
    wx, wy = job.ibuf(B), job.ibuf(B)
    for w in range(W):
        wl.gen_warm(g, (rank * W + w) * B, B, wx, wy)
        wl.incr(scratch, wx, wy)
    del_me = scratch.get_batch(wx, wy)
    del del_me
    # how large an inbox the warm-up batches needed: a hash-sharded skewed stream (c3) sends the hottest rows'
    # ops to ONE owner, which then receives more than a batch's worth
    inbox_ops = max(B, scratch.route_stats()["max_inbox_ops"]) if world > 1 else B
    scratch.close()

    m = mk()
    if world > 1:
        m.reserve_route(inbox_ops)      # inboxes + IPC exchange: communicator-style set-up, untimed
    g = job.generator(m)

    # ---- prefill (untimed, measured separately)
    t_prefill = 0.0
    for k in range(wl.prefill):
        wl.gen_ops(g, wl.first_of(k), B, wx, wy)
        job.barrier()
        t0 = time.perf_counter()
        wl.incr(m, wx, wy)
        job.barrier()
        t_prefill += time.perf_counter() - t0
    del wx, wy

    # ---- timed build: all K batches resident in HBM first
    xs = [job.ibuf(B) for _ in range(K)]
    ys = [job.ibuf(B) for _ in range(K)]
    for j in range(K):
        wl.gen_ops(g, wl.first_of(wl.prefill + j), B, xs[j], ys[j])
    m.set_kernel_timing(True)
    launches0, rounds0 = m.stat("launches"), m.stat("rounds")
    if world > 1:
        m.route_stats(reset=True)
    job.barrier()
    wall0 = time.time()
    m.timer_start()
    step_ms, kern_ms, prev_k = [], [], 0
    PHASES = ("partition", "upsert", "grow_plan", "slab", "migrate", "dir")
    prev_ph = [0.0] * len(PHASES) + [m.stat("rounds"), m.stat("launches")]
    alloc0 = prev_alloc = m.stat("ns_alloc") / 1e6     # cudaMalloc time inside the timed steps (0 with an arena)
    for j in range(K):
        t_s = time.perf_counter()
        wl.incr(m, xs[j], ys[j])                # synchronous: returns when the device is done
        step_ms.append(round((time.perf_counter() - t_s) * 1e3, 2))
        k_now = m.stat("kernel_ns")
        kern_ms.append(round((k_now - prev_k) / 1e6, 2))
        prev_k = k_now
        if a.phase_series and rank == 0:
            now = [m.stat("ns_" + k) / 1e6 for k in PHASES] + [m.stat("rounds"), m.stat("launches")]
            al = m.stat("ns_alloc") / 1e6
            print(f"step {j}: {step_ms[-1]} ms; " + ", ".join(f"{k} {now[i] - prev_ph[i]:.2f}" for i, k in enumerate(PHASES))
                  + f"; rounds {now[-2] - prev_ph[-2]}, launches {now[-1] - prev_ph[-1]}, cudaMalloc {al - prev_alloc:.2f} ms",
                  file=sys.stderr)
            prev_ph, prev_alloc = now, al
    ms_build = m.timer_stop_ms()
    job.barrier()
    wall1 = time.time()
    ms_build = job.max_over_ranks(ms_build)
    launches = m.stat("launches") - launches0
    rounds = m.stat("rounds") - rounds0
    upsert_ns = m.stat("kernel_ns")
    phases = {k: round(m.stat("ns_" + k) / 1e6 / K, 3) for k in PHASES}
    phases["cudaMalloc"] = round((m.stat("ns_alloc") / 1e6 - alloc0) / K, 3)
    route = m.route_stats() if world > 1 else None
    m.set_kernel_timing(False)
    clocks = job.sampler.window(wall0, wall1)
    value = K * B * world / (ms_build * 1e-3) / 1e6
    dump = {}
    if a.dump_outputs:      # incr_batch hands nothing back: its result is the cells it wrote, read back before close
        pick = torch.from_numpy(dump_index(B, DUMP_SAMPLE // world)).to(job.dev)
        dump_keys = xs[K - 1][pick].contiguous(), ys[K - 1][pick].contiguous()
    del xs, ys
    nnz_local, rows_local = m.stat("nnz"), m.stat("rows")
    vsum_local = m.stat("value_sum")     # every op added 1: the table-wide sum must equal the op count
    stats = {k: m.stat(k) for k in ("dir_cap", "slab_bytes", "device_bytes", "row_grows", "dir_grows", "recycled",
                                    "bucket_bytes", "live_bucket_bytes", "free_bytes")}
    stats["buckets_over_live"] = round(stats["bucket_bytes"] / max(1, stats["live_bucket_bytes"]), 3)

    # ---- timed gets (50 % hits): all queries resident first
    G = wl.gets
    qx, qy, out = job.ibuf(G), job.ibuf(G), job.ibuf(G)
    for off in range(0, G, B):
        cnt = min(B, G - off)
        wl.gen_queries(g, rank * G + off, cnt, qx[off:].data_ptr(), qy[off:].data_ptr())
    m.set_kernel_timing(True)
    job.barrier()
    m.timer_start()
    for off in range(0, G, B):
        cnt = min(B, G - off)
        m.get_batch(qx[off:off + cnt], qy[off:off + cnt], out[off:off + cnt])
    ms_get = job.max_over_ranks(m.timer_stop_ms())
    job.barrier()
    get_ns = m.stat("kernel_ns")
    m.set_kernel_timing(False)
    get_mops = G * world / (ms_get * 1e-3) / 1e6
    sliced = m.stat("sliced_gets")
    # the same queries looked up in input order (smatrix_b200_set_get_slices(0)): the A side of the slice-order A/B;
    # $SMX_BENCH_GET_VARIANTS = further set_get_slices() values to time on the same table (measurement switches)
    ref_out = out.clone()
    get_variants = {}
    get_same = True
    for variant in [0] + [int(v, 0) for v in os.environ.get("SMX_BENCH_GET_VARIANTS", "").split(",") if v]:
        m.set_get_slices(variant)
        out.zero_()
        m.set_kernel_timing(True)
        job.barrier()
        m.timer_start()
        for off in range(0, G, B):
            cnt = min(B, G - off)
            m.get_batch(qx[off:off + cnt], qy[off:off + cnt], out[off:off + cnt])
        ms_v = job.max_over_ranks(m.timer_stop_ms())
        job.barrier()
        ns_v = m.stat("kernel_ns")
        m.set_kernel_timing(False)
        same = bool((out == ref_out).all().item())
        get_same = get_same and same
        get_variants[variant] = {"get_mops": G * world / (ms_v * 1e-3) / 1e6, "get_ms": ms_v, "kernels_ms": ns_v / 1e6,
                                 "same_answers": same}
    ms_get0, get0_ns = get_variants[0]["get_ms"], get_variants[0]["kernels_ms"] * 1e6
    # $SMX_BENCH_GET_BATCHES: 2^27 of the queries again in batches of these sizes, input order (0) vs always by slice (2):
    # where the slice order starts to pay as a function of queries per call / rows in the table
    get_sweep = {}
    for bs in [int(v, 0) for v in os.environ.get("SMX_BENCH_GET_BATCHES", "").split(",") if v]:
        tot = min(G, 1 << 27)
        for mode in (0, 2):
            m.set_get_slices(mode)
            job.barrier()
            m.timer_start()
            for off in range(0, tot, bs):
                cnt = min(bs, tot - off)
                m.get_batch(qx[off:off + cnt], qy[off:off + cnt], out[off:off + cnt])
            ms_v = job.max_over_ranks(m.timer_stop_ms())
            get_sweep[f"{bs}:{mode}"] = round(tot * world / (ms_v * 1e-3) / 1e6, 1)
        get_same = get_same and bool((out[:tot] == ref_out[:tot]).all().item())
    m.set_get_slices(int(os.environ.get("SMATRIX_GET_SLICES", "1"), 0))
    if a.dump_outputs:
        dump["get_values"] = ref_out[torch.from_numpy(dump_index(G, DUMP_SAMPLE // world)).to(job.dev)]
    del ref_out
    hits = int((out != 0).sum().item())
    first_q = rank * G
    odd = out[1::2] if first_q % 2 == 0 else out[0::2]
    odd_hits = int((odd != 0).sum().item())
    del qx, qy, out

    # ---- read path on the same table (N = 1, c2): rowlen over all rows, getrow of 2 M rows
    reads = None
    if world == 1 and name == "c2":
        ids = ((torch.arange(wl.rows_total, device=job.dev, dtype=torch.int64) * SCRAMBLE) & 0xFFFFFFFF)
        ids = torch.where(ids >= 2**31, ids - 2**32, ids).to(torch.int32)
        m.rowlen_batch(ids[:1 << 20])                                   # warm
        m.timer_start(); rl = m.rowlen_batch(ids); ms_rl = m.timer_stop_ms()
        sample = ids[: min(wl.rows_total, 1 << 21)].contiguous()
        offs = torch.empty(sample.numel() + 1, dtype=torch.int64, device=job.dev)
        lib, h = m._lib, m._handle()
        total = int(lib.smatrix_getrow_batch(h, sample.data_ptr(), sample.numel(), offs.data_ptr(), None, 0))
        pairs = torch.empty(2 * total, dtype=torch.int32, device=job.dev)
        m.timer_start()
        got = int(lib.smatrix_getrow_batch(h, sample.data_ptr(), sample.numel(), offs.data_ptr(), pairs.data_ptr(), total))
        ms_gr = m.timer_stop_ms()
        reads = {"rowlen_mops": wl.rows_total / (ms_rl * 1e-3) / 1e6, "rowlen_sum": int(rl.to(torch.int64).sum().item()),
                 "getrow_rows": sample.numel(), "getrow_pairs": got, "getrow_ms": ms_gr,
                 "getrow_gpairs_per_s": got / (ms_gr * 1e-3) / 1e9,
                 "getrow_algorithmic_gbs": (32 * sample.numel() + 16 * got) / (ms_gr * 1e-3) / 1e9,
                 "getrow_value_sum": int(pairs[1::2].to(torch.int64).sum().item())}
        del pairs, offs, ids, sample

    if a.dump_outputs:
        dump["incr_values"] = m.get_batch(*dump_keys, job.ibuf(dump_keys[0].numel()))
        write_dump(job, dump)
        del dump, dump_keys
    m.close()
    torch.cuda.empty_cache()      # the timed batches are back with the driver before the next tables reserve their arenas

    # ---- roofline probes in the same process (random 32 B sector reads / 4 B atomics over 32 GiB), after the
    # table is gone: the probe buffer and a 120 GiB arena do not fit one GPU together
    probes = None
    if not a.no_probes and rank == 0:
        from libsmatrix_b200 import SparseMatrix
        pm = SparseMatrix(device=job.local)
        foot, acc = 32 << 30, 1 << 30
        probes = {"footprint_gib": 32,
                  "random_read_32B_per_s": pm.probe_random_read(foot, acc, 32),
                  "random_read_8B_per_s": pm.probe_random_read(foot, acc, 8),
                  "random_atomic_4B_per_s": pm.probe_random_atomic(foot, acc)}
        pm.close()

    e2e = None if a.no_e2e else run_e2e_writes(job, wl, mk, inbox_ops)
    parity = None if a.no_parity else run_parity_writes(job, wl)

    nnz_total, rows_seen, vsum_total = job.sum_over_ranks(nnz_local, rows_local, vsum_local)
    applied = wl.n_batches * B * world
    checks = {"value_sum": vsum_total, "ops_applied": applied, "value_sum_ok": vsum_total == applied,
              "hit_fraction_exact": (odd_hits == 0 and hits == G - G // 2) if world == 1 else (odd_hits == 0),
              "rows_ok": rows_seen <= wl.rows_total, "get_orders_agree": get_same}

    cpu = None
    if rank == 0 and not a.no_cpu:
        est = {"c2": 4.0e6, "c3": 0.5e6, "c5": 3.5e6}[name]            # reference ops/s, order of magnitude
        step = max(100_000, int(est * a.cpu_secs / 8))
        r = cpu_write_baseline(name, wl.cfg, wl.rows_total, wl.tables, 4, 0, step, min(2 * step, 4_000_000))
        cpu = {k: r[k] for k in r if k != "secs"}
    job.barrier()                                                        # the other ranks wait for rank 0's CPU leg

    if rank != 0:
        return None
    peak, peak_src = measured_peak_gbs()
    upsert_launches = max(rounds, 1)
    ops_per_launch = K * B / upsert_launches
    ach = wl.bytes_per_op * K * B / (upsert_ns * 1e-9) / 1e9 if upsert_ns else None
    per_op, tsrc = committed_traffic(f"upsert_dram_bytes_per_op_{name}")
    if per_op is None:
        per_op, tsrc = committed_traffic("upsert_dram_bytes_per_op")
    roofline = {"bound": "hbm", "kernel": "k_upsert<INCR>", "achieved": ach, "peak": peak, "unit": "GB/s",
                "frac": (ach / peak) if ach else None,
                "traffic": per_op * ops_per_launch if per_op else None, "traffic_source": tsrc,
                "peak_source": peak_src, "algorithmic_bytes_per_op": wl.bytes_per_op,
                "algorithmic_note": "3 random 32 B sectors + 8 B streamed (x, y; vals == NULL means all ones)",
                "ops_per_launch": ops_per_launch, "launches": upsert_launches,
                "avg_launch_ms": upsert_ns / upsert_launches / 1e6 if upsert_ns else None,
                "kernel_share_of_step": upsert_ns / 1e6 / ms_build if upsert_ns else None}
    get_ach = GET_BYTES * G / (get_ns * 1e-9) / 1e9 if get_ns else None
    roofline["get"] = {"kernel": "k_get (+ k_partition_count / _scatter, k_parts_prefix, k_gather when the batch is looked up "
                                 "in directory-slice order)", "achieved": get_ach, "frac": (get_ach / peak) if get_ach else None,
                       "algorithmic_bytes_per_op": GET_BYTES, "sliced_fraction": sliced / G,
                       "input_order": {"get_mops": G * world / (ms_get0 * 1e-3) / 1e6, "get_ms": ms_get0,
                                       "achieved": GET_BYTES * G / (get0_ns * 1e-9) / 1e9 if get0_ns else None,
                                       "same_answers": get_variants[0]["same_answers"]}}
    if len(get_variants) > 1:
        roofline["get"]["variants"] = get_variants
    if get_sweep:
        roofline["get"]["batch_sweep_mops"] = get_sweep
    if probes:
        r32 = probes["random_read_32B_per_s"]
        roofline["random_sector"] = {
            "R32_sectors_per_s": r32, "atomic_4B_per_s": probes["random_atomic_4B_per_s"],
            "read_8B_per_s": probes["random_read_8B_per_s"], "footprint_gib": probes["footprint_gib"],
            "incr_frac": INCR_SECTORS * (K * B / (upsert_ns * 1e-9)) / r32 if upsert_ns else None,
            "incr_frac_step": INCR_SECTORS * (K * B / (ms_build * 1e-3)) / r32,
            "get_frac": GET_SECTORS * (G / (get_ns * 1e-9)) / r32 if get_ns else None,
            "get_frac_input_order": GET_SECTORS * (G / (get0_ns * 1e-9)) / r32 if get0_ns else None,
            "note": "achieved = ops/s x algorithmic random sectors per op (3 incr, 2 get) / measured random 32 B read rate; "
                    "incr_frac: inside k_upsert, incr_frac_step: over the whole timed region; get_frac counts 2 sectors per query "
                    "although the slice-ordered look-up fetches a directory entry from DRAM once per row and batch, not once "
                    "per query (it can exceed 1); get_frac_input_order is the plain kernel"}
    if route:
        per_step = route["remote_bytes"] / max(K, 1)
        roofline["nvlink"] = {"bound": "nvlink", "peak": 900.0, "unit": "GB/s",
                              "remote_bytes_per_rank_per_step": per_step,
                              "min_ms_per_step": per_step / 900e9 * 1e3,
                              "route_ms_per_step": route["route_ms"] / max(K, 1),
                              "apply_ms_per_step": route["apply_ms"] / max(K, 1),
                              "achieved": per_step / (route["route_ms"] / max(K, 1) * 1e-3) / 1e9 if route["route_ms"] else None,
                              "note": "rank 0's view: bytes its partition kernel stored into the other ranks' inboxes per step / "
                                      "the NVLink 5 per-direction rate; route = count + count exchange + scatter + arrival barrier"}
    line = {
        "metric": wl.cfg["metric"], "value": value, "unit": "Mops/s", "n_gpus": world, "steps": K,
        "warmup": W, "ms_per_step": ms_build / K, "higher_is_better": True, "scaling": wl.cfg["scaling"],
        "vs_baseline": None, "dtype": "u32", "data": "synthetic",
        "parity": parity, "checks": checks,
        "config": {"workload": wl.describe(), "rows": wl.rows_total, "ops_per_step": B * world, "timed_ops": K * B * world,
                   "prefill_ops": wl.prefill * B * world, "gets": G * world, "scale": a.scale,
                   "l2": "inputs larger than L2 (512 MiB of keys per step, table >> 126 MB)",
                   "arena_gib": wl.arena, "arena_note": "slab arena reserved by smatrix_open (outside the timed region); "
                   "on-demand cudaMalloc is the fallback and costs 0.3-8 ms/step on this pool",
                   "chunk_ops": int(os.environ.get("SMATRIX_CHUNK", 1 << 26)),
                   "parallelism": f"row-hash shard x{world}, C router over peer memory" if world > 1 else "single GPU"},
        "get_mops": get_mops, "get_ms": ms_get, "get_hit_fraction": hits / G,
        "get_mops_input_order": G * world / (ms_get0 * 1e-3) / 1e6,   # the same queries with set_get_slices(0)
        "nnz": nnz_total, "rows_present": rows_seen, "prefill_s": t_prefill,
        "table": stats, "clocks": clocks, "gpu_launches": launches, "upsert_rounds": rounds,
        "host_phase_ms_per_step": phases, "step_ms": step_ms, "step_upsert_kernel_ms": kern_ms,
        "roofline": roofline,
    }
    if "ycols" in wl.cfg:
        line["config"]["ycols"] = wl.cfg["ycols"]
    if reads:
        line["reads"] = reads
    if e2e:
        line["e2e"] = e2e
    line["cpu_baseline"] = cpu
    return line


def run_e2e_writes(job: Job, wl: WriteWorkload, mk, inbox_ops=None):
    """Same stream, HOST buffers: each timed step is one incr_batch(host arrays) call per rank —
    H2D of the batch, (N > 1: the route,) the update, and the D2H reads of the control block.
    Per step: barrier, wall clock around the call, max over ranks.  Byte counts = the library's own
    copy counters over the timed steps."""
    a, B, K, rank, world = job.a, wl.B, wl.K, job.rank, job.world
    dx, dy = job.ibuf(B), job.ibuf(B)
    hx, hy = job.pinned(B), job.pinned(B)
    scratch = mk()                               # warm-up of the host-pointer path (W steps, other seed)
    g = job.generator(scratch)
    for w in range(a.warmup):
        wl.gen_warm(g, (rank * a.warmup + w + 7) * B, B, dx, dy)
        hx.copy_(dx); hy.copy_(dy)
        job.torch.cuda.synchronize()
        wl.incr(scratch, hx, hy)
    scratch.close()
    m = mk()
    if world > 1:
        m.reserve_route(inbox_ops or B)
    g = job.generator(m)
    for k in range(wl.prefill):
        wl.gen_ops(g, wl.first_of(k), B, dx, dy)
        wl.incr(m, dx, dy)
    h2d0, d2h0 = m.stat("h2d_bytes"), m.stat("d2h_bytes")
    secs, series = 0.0, []
    for j in range(K):
        wl.gen_ops(g, wl.first_of(wl.prefill + j), B, dx, dy)
        hx.copy_(dx); hy.copy_(dy)
        job.barrier()
        t0 = time.perf_counter()
        wl.incr(m, hx, hy)                       # returns after the device finished (synchronous API)
        dt = job.max_over_ranks(time.perf_counter() - t0)
        series.append(round(dt * 1e3, 2))
        secs += dt
    h2d, d2h = job.sum_over_ranks(m.stat("h2d_bytes") - h2d0, m.stat("d2h_bytes") - d2h0)
    incr = K * B * world / secs / 1e6
    # gets through host buffers: queries up, values down
    G = min(wl.gets, 4 * B)
    hq, hr = job.pinned(B), job.pinned(B)
    gsecs, done = 0.0, 0
    h2d1, d2h1 = m.stat("h2d_bytes"), m.stat("d2h_bytes")
    while done < G:
        cnt = min(B, G - done)
        wl.gen_queries(g, rank * G + done, cnt, dx.data_ptr(), dy.data_ptr())
        hx.copy_(dx); hq.copy_(dy)
        job.barrier()
        t0 = time.perf_counter()
        m.get_batch(hx[:cnt], hq[:cnt], hr[:cnt])
        gsecs += job.max_over_ranks(time.perf_counter() - t0)
        done += cnt
    gh2d, gd2h = job.sum_over_ranks(m.stat("h2d_bytes") - h2d1, m.stat("d2h_bytes") - d2h1)
    gsteps = -(-G // B)
    m.close()
    # the box's own ceiling for this step's upload: every rank copies its pinned batch (x, y) host -> device at the
    # same time, nothing else running — what e2e could reach if routing and updating were free
    job.barrier()
    t0 = time.perf_counter()
    for _ in range(4):
        dx.copy_(hx, non_blocking=True); dy.copy_(hy, non_blocking=True)
    job.torch.cuda.synchronize()
    ceil_s = job.max_over_ranks(time.perf_counter() - t0) / 4
    ceiling_mops = B * world / ceil_s / 1e6
    return {"value": incr, "unit": "Mops/s", "h2d_bytes_per_step": h2d // K, "d2h_bytes_per_step": d2h // K,
            "ms_per_step": secs / K * 1e3, "step_ms": series,
            "get_mops": G * world / gsecs / 1e6, "get_h2d_bytes_per_step": gh2d // gsteps,
            "get_d2h_bytes_per_step": gd2h // gsteps,
            "pcie_frac": (h2d / K / world) / (secs / K) / 55e9,
            "h2d_ceiling": {"mops": ceiling_mops, "gbs_per_gpu": 8 * B / ceil_s / 1e9, "ms_per_step": ceil_s * 1e3,
                            "frac": incr / ceiling_mops,
                            "note": "all ranks uploading one step's pinned (x, y) arrays concurrently, nothing else running"},
            "note": "pinned host arrays through incr_batch / get_batch (N = 1: the C-ABI smatrix_incr_batch / smatrix_get_batch "
                    "with host pointers; N > 1: smatrix_b200_shard_* stage each rank's slice piece by piece, then route); barrier, "
                    "wall clock around the call, max over ranks; bytes = the library's copy counters, summed over ranks; "
                    "pcie_frac = per-GPU H2D rate / 55 GB/s"}


def run_parity_writes(job: Job, wl: WriteWorkload):
    """Parity in the driver's own record: a prefix of the SAME stream (reduced key space so that rows
    fill up) goes into a fresh matrix through the same product path — sharded at N > 1, every rank its
    slice — plus a duplicate-heavy set batch and column-0 incrs; every rank then compares its share of
    gets, rowlens and column-sorted getrows with the CPU reference fed the whole prefix."""
    from oracle import cpu
    a, rank, world = job.a, job.rank, job.world
    cpu.build(ref=True)
    kind = "reference" if cpu.have_reference() else "port"
    n = a.parity_ops
    name, cfg = wl.name, wl.cfg
    if name == "c3":
        from libsmatrix_b200.workloads import zipf_thresholds
        tables = {"thr": zipf_thresholds(min(20_000, wl.items), cfg["zipf_s"])}
        rows_p = len(tables["thr"])
        xs, ys, _ = _host_stream(name, cfg, 0, n, rows_p, tables)
    else:
        rows_p, tables = 40_000 * world, {}
        xs, ys, _ = _host_stream(name, cfg, 0, n, rows_p, tables)
    rng = np.random.default_rng(12345)
    ns = n // 8                                          # set batch with duplicates + a few column-0 writes
    sx, sy = xs[rng.integers(0, n, ns)], rng.integers(0, 12, ns).astype(np.uint32)
    sv = rng.integers(1, 2**32, ns, dtype=np.uint64).astype(np.uint32)
    ref = cpu.CpuMatrix(kind)
    ref.apply("incr", xs, ys, np.ones(n, np.uint32))
    ref.apply("set", sx, sy, sv)
    m = job.make_matrix(0)
    sl = lambda k: slice(rank * k // world, (rank + 1) * k // world)
    if world > 1:
        m.incr_batch(xs[sl(n)], ys[sl(n)], None, ordered=True)
        m.set_batch(sx[sl(ns)], sy[sl(ns)], sv[sl(ns)])
    else:
        m.incr_batch(xs, ys, None)
        m.set_batch(sx, sy, sv)
    nq = min(n, 400_000)
    qx, qy = _host_queries(name, cfg, 0, nq, n, rows_p, tables)
    qx, qy = np.concatenate([qx, sx[:nq // 8]]), np.concatenate([qy, sy[:nq // 8]])
    mine = slice(rank, None, world)                      # every rank checks its share
    got = np.asarray(m.get_batch(qx[mine].copy(), qy[mine].copy())).view(np.uint32)
    get_mis = int((got != ref.get_many(qx[mine], qy[mine])).sum())
    rows = np.unique(xs)
    rows = np.concatenate([rows, np.array([0xFFFFFFF0, 0xFFFFFFF1], np.uint32)])[mine].copy()   # + rows nobody has
    rl_mis = int((np.asarray(m.rowlen_batch(rows)).view(np.uint32) != ref.rowlen_many(rows)).sum())
    o1, p1 = m.getrow_batch(rows)
    o2, p2 = ref.getrow_many(rows)
    if (o1 != o2).any():
        gr_mis = int((np.diff(o1.astype(np.int64)) != np.diff(o2.astype(np.int64))).sum()) or 1
    else:
        gr_mis = int((cpu.sort_rows(o1, p1) != cpu.sort_rows(o2, p2)).any(axis=1).sum())
    m.close(); ref.close()
    tot = job.sum_over_ranks(get_mis, rl_mis, gr_mis, len(got), len(rows), len(p2))
    return {"mismatches": tot[0] + tot[1] + tot[2], "get_mismatches": tot[0], "rowlen_mismatches": tot[1],
            "getrow_mismatches": tot[2], "gets": tot[3], "rowlens": tot[4], "getrow_rows": tot[4], "getrow_pairs": tot[5],
            "ops": n + ns, "checker": kind, "ranks": world,
            "what": f"first {n} ops of the {name} stream over a reduced key space ({rows_p} rows) + {ns} duplicate-heavy set ops "
                    "(incl. column 0), applied to a fresh matrix through the product path (ordered collective batches at N > 1); "
                    "gets / rowlens / column-sorted getrows of every row compared with the CPU reference, every rank its share"}


# ------------------------------------------------------------------------------ c4: the read path
def run_c4(job: Job):
    a, torch, rank, world = job.a, job.torch, job.rank, job.world
    cfg = WORKLOADS["c4"]
    from libsmatrix_b200.workloads import zipf_thresholds
    R = scaled(a, cfg["rows"]) * world                   # weak scaling: 13 M rows per GPU
    kmax = cfg["kmax"] if a.scale >= 1 else max(1000, scaled(a, cfg["kmax"]))
    thr = zipf_thresholds(kmax, cfg["zipf_s"])
    d_thr = torch.from_numpy(thr.view(np.int64)).to(job.dev)
    arena = a.arena_gib if a.arena_gib is not None else (max(2, int(48 * a.scale) + 1) if a.scale < 1 else 48)
    m = job.make_matrix(arena)
    g = job.generator(m)
    B = a.batch

    # ---- row lengths, offsets (exclusive prefix: plumbing), the build
    lens = job.ibuf(R)
    g.gen_c4_lens(cfg["seed"], 0, R, d_thr.data_ptr(), kmax, lens.data_ptr())
    offs = torch.zeros(R + 1, dtype=torch.int64, device=job.dev)
    torch.cumsum(lens.to(torch.int64), 0, out=offs[1:])
    nnz_expected = int(offs[-1].item())
    torch.cuda.synchronize()
    bx, by, bv = job.ibuf(B), job.ibuf(B), job.ibuf(B)
    n_batches = -(-nnz_expected // (B * world))
    if world > 1:
        m.reserve_route(B)
    job.barrier()
    t0 = time.perf_counter()
    for k in range(n_batches):                           # ranks interleave batch-wise over the op stream
        first = (k * world + rank) * B
        cnt = max(0, min(B, nnz_expected - first))
        if cnt:
            g.gen_c4_ops(cfg["seed"], first, cnt, offs.data_ptr(), R, bx.data_ptr(), by.data_ptr(), bv.data_ptr())
        if world > 1:
            m.incr_batch(bx[:cnt], by[:cnt], bv[:cnt], ordered=False)
        else:
            m.incr_batch(bx[:cnt], by[:cnt], bv[:cnt])
    job.barrier()
    build_s = time.perf_counter() - t0
    del bx, by, bv
    nnz_local, rows_local = m.stat("nnz"), m.stat("rows")
    stats = {k: m.stat(k) for k in ("dir_cap", "slab_bytes", "device_bytes", "row_grows", "recycled",
                                    "bucket_bytes", "live_bucket_bytes", "free_bytes")}
    stats["buckets_over_live"] = round(stats["bucket_bytes"] / max(1, stats["live_bucket_bytes"]), 3)

    # ---- steps: this rank asks for ITS 1/world of the rows (ids interleaved), 1/K of them per step
    K = a.steps or 13
    ids_all = (torch.arange(rank, R, world, device=job.dev, dtype=torch.int64) * SCRAMBLE) & 0xFFFFFFFF
    ids_all = torch.where(ids_all >= 2**31, ids_all - 2**32, ids_all).to(torch.int32)
    my_lens = lens[rank::world].to(torch.int64)
    n_mine = ids_all.numel()
    cut = [j * n_mine // K for j in range(K + 1)]
    step_pairs = [int(my_lens[cut[j]:cut[j + 1]].sum().item()) for j in range(K)]
    cap = max(step_pairs) + 16
    pairs = job.ibuf(2 * cap)
    offsets = torch.empty(max(cut[j + 1] - cut[j] for j in range(K)) + 1, dtype=torch.int64, device=job.dev)
    rl_out = job.ibuf(n_mine)
    lib = m._lib
    sharded = world > 1

    def getrow(ids, cap_pairs, p_off, p_pairs):
        if sharded:
            return m.getrow_batch_into(ids.data_ptr(), ids.numel(), p_off, p_pairs, cap_pairs)
        return int(lib.smatrix_getrow_batch(m._handle(), ids.data_ptr(), ids.numel(), p_off, p_pairs, cap_pairs))

    if sharded:
        m.reserve_route(max(cut[j + 1] - cut[j] for j in range(K)) + 1, job.max_over_ranks(cap))
    for w in range(a.warmup):                            # warm-up on the first slab
        ids = ids_all[cut[0]:cut[1]]
        m.rowlen_batch(ids, out=rl_out[cut[0]:cut[1]])
        getrow(ids, cap, offsets.data_ptr(), pairs.data_ptr())
    m.set_kernel_timing(True)
    launches0 = m.stat("launches")
    job.barrier()
    wall0 = time.time()
    m.timer_start()
    got_pairs, step_ms, rl_ms = 0, [], 0.0
    vsum = 0
    for j in range(K):
        ids = ids_all[cut[j]:cut[j + 1]]
        t_s = time.perf_counter()
        m.rowlen_batch(ids, out=rl_out[cut[j]:cut[j + 1]])
        rl_ms += (time.perf_counter() - t_s) * 1e3
        got = getrow(ids, cap, offsets.data_ptr(), pairs.data_ptr())
        step_ms.append(round((time.perf_counter() - t_s) * 1e3, 2))
        got_pairs += got
        assert got == step_pairs[j], (got, step_pairs[j])
    ms_read = m.timer_stop_ms()
    job.barrier()
    wall1 = time.time()
    ms_read = job.max_over_ranks(ms_read)
    fill_ns = m.stat("kernel_ns")
    launches = m.stat("launches") - launches0
    m.set_kernel_timing(False)
    clocks = job.sampler.window(wall0, wall1)
    if a.dump_outputs:
        dump_c4_last_step(job, rl_out[cut[K - 1]:cut[K]], offsets[:cut[K] - cut[K - 1] + 1], pairs)
    rowlen_ok = bool((rl_out.to(torch.int64) == my_lens).all().item())   # no column 0 here: rowlen = distinct columns
    last_val_sum = int(pairs[1:2 * step_pairs[-1]:2].to(torch.int64).sum().item())
    pairs_total, rows_asked = job.sum_over_ranks(got_pairs, n_mine)
    value = pairs_total / (ms_read * 1e-3) / 1e6

    # ---- e2e: host buffers for the answers (offsets + pairs come down inside the timed region)
    e2e = None
    if not a.no_e2e:
        h_ids = job.pinned(offsets.numel())
        h_off = torch.empty(offsets.numel(), dtype=torch.int64, pin_memory=True)
        h_pairs = job.pinned(2 * cap)
        h_rl = job.pinned(offsets.numel())
        KE = min(K, 4)
        for w in range(min(a.warmup, 2)):               # warm-up of the host-pointer path (staging buffer, pinned pages)
            nrow = cut[K] - cut[K - 1]
            h_ids[:nrow].copy_(ids_all[cut[K - 1]:cut[K]])
            job.torch.cuda.synchronize()
            getrow(h_ids[:nrow], cap, h_off.data_ptr(), h_pairs.data_ptr()) if not sharded else \
                m.getrow_batch_into(h_ids.data_ptr(), nrow, h_off.data_ptr(), h_pairs.data_ptr(), cap)
        h2d0, d2h0 = m.stat("h2d_bytes"), m.stat("d2h_bytes")
        secs, epairs, e_series = 0.0, 0, []
        for j in range(KE):
            nrow = cut[j + 1] - cut[j]
            h_ids[:nrow].copy_(ids_all[cut[j]:cut[j + 1]])
            job.barrier()
            t0 = time.perf_counter()
            if sharded:
                lib.smatrix_b200_shard_rowlen_batch(m._handle(), h_ids.data_ptr(), nrow, h_rl.data_ptr())
                epairs += m.getrow_batch_into(h_ids.data_ptr(), nrow, h_off.data_ptr(), h_pairs.data_ptr(), cap)
            else:
                lib.smatrix_rowlen_batch(m._handle(), h_ids.data_ptr(), nrow, h_rl.data_ptr())
                epairs += int(lib.smatrix_getrow_batch(m._handle(), h_ids.data_ptr(), nrow, h_off.data_ptr(),
                                                       h_pairs.data_ptr(), cap))
            dt = job.max_over_ranks(time.perf_counter() - t0)
            e_series.append(round(dt * 1e3, 2))
            secs += dt
        h2d, d2h, epairs = job.sum_over_ranks(m.stat("h2d_bytes") - h2d0, m.stat("d2h_bytes") - d2h0, epairs)
        e2e = {"value": epairs / secs / 1e6, "unit": "Mpairs/s", "h2d_bytes_per_step": h2d // KE,
               "d2h_bytes_per_step": d2h // KE, "ms_per_step": secs / KE * 1e3, "steps": KE, "step_ms": e_series,
               "pcie_frac": (d2h / KE / world) / (secs / KE) / 55e9,
               "note": "row ids, rowlens, offsets and pairs in pinned HOST buffers through smatrix_rowlen_batch + "
                       "smatrix_getrow_batch; the D2H of 8 B per pair is inside the timed region (PCIe-bound); bytes = the "
                       "library's copy counters"}

    # ---- parity: sampled rows (incl. the longest ones) rebuilt on the CPU reference
    parity = None
    if not a.no_parity:
        parity = run_parity_c4(job, m, cfg, lens, offs, R)
    m.close()
    nnz_total, rows_seen = job.sum_over_ranks(nnz_local, rows_local)

    cpu = None
    if rank == 0 and not a.no_cpu:
        r = cpu_read_baseline(cfg, {"thr": thr}, max(20_000, int(150_000 * a.cpu_secs / 12)), 4, 0)
        cpu = {k: r[k] for k in r if k != "secs"}
    job.barrier()
    if rank != 0:
        return None
    peak, peak_src = measured_peak_gbs()
    alg_bytes = 32 * rows_asked + 16 * pairs_total
    ach = (alg_bytes / world) / (fill_ns * 1e-9) / 1e9 if fill_ns else None
    per_pair, tsrc = committed_traffic("getrow_dram_bytes_per_pair")
    roofline = {"bound": "hbm", "kernel": "k_getrow_fill + k_getrow_big", "achieved": ach, "peak": peak, "unit": "GB/s",
                "frac": (ach / peak) if ach else None,
                "traffic": per_pair * pairs_total / world / max(K, 1) if per_pair else None, "traffic_source": tsrc,
                "peak_source": peak_src,
                "algorithmic_bytes": "32 B per row + 16 B per pair (8 read + 8 written), SURVEY.md 8(d)",
                "kernel_share_of_step": fill_ns / 1e6 / ms_read if fill_ns else None,
                "step_level_gbs": (alg_bytes / world) / (ms_read * 1e-3) / 1e9}
    return {
        "metric": cfg["metric"], "value": value, "unit": "Mpairs/s", "n_gpus": world, "steps": K, "warmup": a.warmup,
        "ms_per_step": ms_read / K, "higher_is_better": True, "scaling": cfg["scaling"], "vs_baseline": None,
        "dtype": "u32", "data": "synthetic", "parity": parity,
        "checks": {"nnz": nnz_total, "nnz_expected": nnz_expected, "nnz_ok": nnz_total == nnz_expected,
                   "rows_ok": rows_seen == R, "rowlen_equals_generated_length": rowlen_ok,
                   "pairs_ok": pairs_total == nnz_expected, "last_step_value_sum": last_val_sum},
        "config": {"workload": "C4 read path: rowlen_batch + getrow_batch over ALL rows of a table with Zipf(1.7) row lengths "
                               "1 .. 10^6 (SURVEY.md 8d), 13 M rows per GPU, 1/steps of the rows per step",
                   "rows": R, "kmax": kmax, "nnz": nnz_expected, "rows_per_step": rows_asked // K, "scale": a.scale,
                   "l2": "every step reads ~1 GB of buckets and writes ~0.8 GB of pairs: larger than L2",
                   "arena_gib": arena,
                   "parallelism": f"row-hash shard x{world}, C router over peer memory" if world > 1 else "single GPU"},
        "rowlen_mops": rows_asked / (rl_ms * 1e-3) / 1e6 if rl_ms else None,
        "build": {"seconds": build_s, "mops": nnz_expected / build_s / 1e6, "batches_per_rank": n_batches},
        "table": stats, "clocks": clocks, "gpu_launches": launches, "step_ms": step_ms,
        "roofline": roofline, "e2e": e2e, "cpu_baseline": cpu,
    }


def dump_c4_last_step(job: Job, rowlen, offsets, pairs):
    """The last step's answers: rowlens, and the getrow pairs of a seeded sample of its rows (at most
    DUMP_SAMPLE pairs over the job), each row sorted by column because a row's pairs come back in table order."""
    torch, k = job.torch, DUMP_SAMPLE // job.world
    offs = offsets.cpu().numpy()
    rows = dump_index(len(offs) - 1, (1 << 16) // job.world)
    lens = offs[rows + 1] - offs[rows]
    keep = np.cumsum(lens) <= k
    rows, lens = rows[keep], lens[keep]
    at = np.repeat(offs[rows] - np.cumsum(lens) + lens, lens) + np.arange(int(lens.sum()))
    got = pairs.view(-1, 2)[torch.from_numpy(at).to(job.dev)].cpu().numpy().view(np.uint32)
    row_of = np.repeat(np.arange(len(rows)), lens)
    write_dump(job, {"rowlen": rowlen[torch.from_numpy(dump_index(rowlen.numel(), k)).to(job.dev)],
                     "getrow_lengths": lens, "getrow_pairs": got[np.lexsort((got[:, 0], row_of))]})


def run_parity_c4(job: Job, m, cfg, lens, offs, R):
    from oracle import cpu
    cpu.build(ref=True)
    kind = "reference" if cpu.have_reference() else "port"
    torch, rank, world = job.torch, job.rank, job.world
    h_lens = lens.cpu().numpy().astype(np.int64)
    h_offs = offs.cpu().numpy().astype(np.uint64)
    rng = np.random.default_rng(777 + rank)
    longest = np.argsort(h_lens)[-2 - rank:][:1] if world > 1 else np.argsort(h_lens)[-3:]
    sample = np.unique(np.concatenate([rng.integers(0, R, 3000), longest]))
    ref = cpu.CpuMatrix(kind)
    for r in sample:                                     # only the sampled rows' ops: rows are independent
        x, y, v = cpu.gen_c4_ops(cfg["seed"], int(h_offs[r]), int(h_lens[r]), h_offs)
        ref.apply("incr", x, y, v)
    ids = (sample.astype(np.uint64) * SCRAMBLE).astype(np.uint32)
    ghost = 0xFFFFFFF3                                   # a row id nobody wrote (unless it is row r < R: skip it then)
    if (ghost * pow(SCRAMBLE, -1, 2**32)) % 2**32 >= R:
        ids = np.concatenate([ids, np.array([ghost], np.uint32)])
    rl_mis = int((np.asarray(m.rowlen_batch(ids)).view(np.uint32) != ref.rowlen_many(ids)).sum())
    o1, p1 = m.getrow_batch(ids)
    o2, p2 = ref.getrow_many(ids)
    if (o1 != o2).any():
        gr_mis = int((np.diff(o1.astype(np.int64)) != np.diff(o2.astype(np.int64))).sum()) or 1
    else:
        gr_mis = int((cpu.sort_rows(o1, p1) != cpu.sort_rows(o2, p2)).any(axis=1).sum())
    gq = min(len(p2), 200_000)
    pick = rng.integers(0, max(1, len(p2)), gq)
    row_of = np.repeat(np.arange(len(ids)), np.diff(o2.astype(np.int64)))
    qx, qy = ids[row_of[pick]], p2[pick, 0].copy()
    qy[::2] ^= np.uint32(0x5A5A5A5A)                    # half of them (almost surely) misses
    get_mis = int((np.asarray(m.get_batch(qx.copy(), qy.copy())).view(np.uint32) != ref.get_many(qx, qy)).sum())
    ref.close()
    tot = job.sum_over_ranks(get_mis, rl_mis, gr_mis, gq, len(ids), len(p2), int(h_lens[sample].max()))
    return {"mismatches": tot[0] + tot[1] + tot[2], "get_mismatches": tot[0], "rowlen_mismatches": tot[1],
            "getrow_mismatches": tot[2], "gets": tot[3], "rowlens": tot[4], "getrow_rows": tot[4], "getrow_pairs": tot[5],
            "checker": kind, "ranks": world,
            "what": "per rank ~3000 random rows + the longest rows of the FULL-SCALE table: their ops are replayed into the CPU "
                    "reference (rows are independent), then rowlen, column-sorted getrow and gets (half misses) are compared"}


def _json_only_stdout():
    """Everything that C libraries print to fd 1 (NCCL's version banner, ...) goes to stderr; the
    returned file object is the real stdout for the ONE JSON line."""
    sys.stdout.flush()
    real = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    return real


def main_ours(a):
    job = Job(a)
    try:
        line = run_c4(job) if a.workload == "c4" else run_write_workload(job, a.workload)
    finally:
        job.finish()
    if line is not None:
        print(json.dumps(line), flush=True)


if __name__ == "__main__":
    args = parse()
    _REAL_STDOUT = _json_only_stdout()
    _print = print

    def print(*a, **k):     # noqa: A001 - only the JSON line is printed with flush=True below
        k.setdefault("file", _REAL_STDOUT)
        _print(*a, **k)
    if args.impl == "reference":
        main_reference(args)
    else:
        main_ours(args)
