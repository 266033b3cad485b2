"""Worker for tests/test_gpu_checkpoint.py: one rank (= one GPU) of a file-backed sharded matrix.
usage: checkpoint_gpu_worker.py build|ck|load <file>; RANK / WORLD_SIZE / SMX_NAME in the environment.
`build` builds the table from a seeded stream (every rank its slice) and closes (= the full snapshot); `ck` touches
a seeded tenth of the rows, checkpoints, and rank 0 copies the checkpointed file to <file>.ck and writes the
answers of the live table to <file>.npz; `load` opens the file and compares with <file>.npz."""
import os
import shutil
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from libsmatrix_b200.sharded import ShardedSparseMatrix  # noqa: E402
from oracle import cpu  # noqa: E402

U32 = np.uint32


def stream(n=2_000_000, seed=777, rows=100_000):
    rng = np.random.default_rng(seed)
    xs = rng.integers(0, rows, n).astype(U32) * U32(2654435761)
    ys = rng.integers(1, 256, n).astype(U32)
    ys[rng.random(n) < 0.05] = 0                      # column-0 traffic
    vs = rng.integers(1, 1000, n).astype(U32)
    return xs, ys, vs


def update():
    return stream(200_000, seed=778, rows=10_000)    # the first tenth of the row ids, and some new columns


def answers(m, rows):
    o, p = m.getrow_batch(rows)
    stats = [m.sum(m.stat(k)) % 2**64 for k in ("rows", "nnz", "value_sum")]
    return {"rowlen": np.asarray(m.rowlen_batch(rows)).copy(), "offsets": o, "pairs": cpu.sort_rows(o, p),
            "stats": np.array(stats, dtype=np.uint64)}


def main():
    phase, path = sys.argv[1], sys.argv[2]
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    torch.cuda.set_device(rank)
    m = ShardedSparseMatrix(rank, world, rank, name=os.environ["SMX_NAME"], fname=path)
    rows = np.unique(np.r_[stream()[0], update()[0]])
    dev = torch.device("cuda", rank)
    t = lambda a: torch.from_numpy(a.view(np.int32).copy()).to(dev)
    if phase in ("build", "ck"):
        xs, ys, vs = stream() if phase == "build" else update()
        sl = slice(rank * len(xs) // world, (rank + 1) * len(xs) // world)
        m.incr_batch(t(xs[sl]), t(ys[sl]), t(vs[sl]))
    if phase == "ck":
        dirty = m.sum(m.stat("dirty_rows"))
        assert dirty == len(np.unique(update()[0])), dirty
        assert m.checkpoint() == 0
        assert m.sum(m.stat("dirty_rows")) == 0
        m.barrier()
        if rank == 0:
            shutil.copy(path, path + ".ck")
        got = answers(m, rows)
        if rank == 0:
            np.savez(path + ".npz", **got)
        m.barrier()
    elif phase == "load":
        got = answers(m, rows)
        if rank == 0:
            want = np.load(path + ".npz")
            for k in ("offsets", "pairs", "stats"):
                assert np.array_equal(got[k], want[k]), f"{k} differs after the reload at world {world}"
    m.close()
    print(f"rank {rank} ok", flush=True)


if __name__ == "__main__":
    main()
