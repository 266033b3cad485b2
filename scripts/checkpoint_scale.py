"""Incremental checkpoints at scale on one GPU: a config-2 table (a fraction of 13 M rows and 2 * 10^9 incr ops over
256 columns, built on the device) in a file under /dev/shm.

Reported per line:
  - the full snapshot (smatrix_b200_snapshot: every row block to a temporary file, fsync, rename);
  - for f = 1 %, 10 % and 100 % of the rows: a snapshot first (the base, not timed), then gen_c2_ops with
    rows = f * R over the same id space (8 f R ops: nearly every one of the first f * R row ids is hit), then the
    timed checkpoint: rows written, bytes appended, whether it appended or fell back to a full snapshot (the file
    would have passed twice a full snapshot's size);
  - the reload of the final file: its time, and whether rows, nnz and value_sum equal the live table's.
With more than one GPU the sharded checkpoint is not measured here (no multi-process harness in this script).
Times are host wall clock around calls that end in a synchronise and an fsync.  Writes one JSON to
profiles/checkpoint_scale.json (or argv[2]) with the card's name and power limit read in the same run.

    python scripts/checkpoint_scale.py [fraction=0.25] [out.json] [dir=/dev/shm]
"""
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

from libsmatrix_b200 import SparseMatrix  # noqa: E402


def log(*a):
    print(*a, flush=True)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q[0] if q else "unknown"


def timed(fn):
    t0 = time.perf_counter()
    rc = fn()
    return rc, time.perf_counter() - t0


def head_ptr(path):
    with open(path, "rb") as f:
        f.seek(8)
        return int.from_bytes(f.read(8), "little")


def main():
    frac = float(sys.argv[1]) if len(sys.argv) > 1 else 0.25
    out = sys.argv[2] if len(sys.argv) > 2 else os.path.join(ROOT, "profiles", "checkpoint_scale.json")
    where = sys.argv[3] if len(sys.argv) > 3 else "/dev/shm"
    R, ops, B = int(13_000_000 * frac), int(2_000_000_000 * frac), 1 << 26
    path = os.path.join(where, f"smx_checkpoint_scale_{os.getpid()}.smx")
    os.environ["SMATRIX_ARENA_GIB"] = str(max(4, int(64 * frac) + 2))
    res = {"gpu": card(), "gpus": torch.cuda.device_count(), "fraction": frac, "rows": R, "ops": ops, "dir": where}
    m = SparseMatrix(path, device=0)
    xs = torch.empty(B, dtype=torch.int32, device="cuda")
    ys = torch.empty(B, dtype=torch.int32, device="cuda")

    def feed(rows, first, count):
        for at in range(0, count, B):
            n = min(B, count - at)
            m.gen_c2_ops(2, first + at, n, rows, 256, xs.data_ptr(), ys.data_ptr())
            m.incr_batch(xs[:n], ys[:n], None)
        m.sync()

    _, res["build_s"] = timed(lambda: feed(R, 0, ops))
    res["table_rows"], res["nnz"] = m.stat("rows"), m.stat("nnz")
    rc, s = timed(m.snapshot)
    assert rc == 0
    res["snapshot"] = {"s": round(s, 3), "file_bytes": os.path.getsize(path),
                       "gbs": round(os.path.getsize(path) / s / 1e9, 3)}
    log("snapshot", res["snapshot"])
    res["checkpoints"] = []
    first = ops
    for f in (0.01, 0.10, 1.00):
        assert m.snapshot() == 0                     # the base
        rows = max(1, int(f * R))
        count = 8 * rows
        feed(rows, first, count)
        first += count
        dirty = m.stat("dirty_rows")
        size0 = os.path.getsize(path)
        rc, s = timed(m.checkpoint)
        assert rc == 0 and m.stat("dirty_rows") == 0
        size1 = os.path.getsize(path)
        appended = head_ptr(path) != 512
        line = {"fraction_touched": f, "dirty_rows": dirty, "s": round(s, 3), "appended": appended,
                "bytes_appended": size1 - size0 if appended else None, "file_bytes": size1}
        res["checkpoints"].append(line)
        log("checkpoint", line)
    live = {k: m.stat(k) for k in ("rows", "nnz", "value_sum")}
    m2, s = timed(lambda: SparseMatrix(path, device=0))
    got = {k: m2.stat(k) for k in ("rows", "nnz", "value_sum")}
    res["reload"] = {"s": round(s, 3), "equal": got == live, "stats": got}
    log("reload", res["reload"])
    os.remove(path)
    with open(out, "w") as fh:
        json.dump(res, fh, indent=1)
    log(json.dumps(res))
    os._exit(0)                                      # no close-time snapshots of the two handles


if __name__ == "__main__":
    main()
