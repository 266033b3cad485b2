"""Worker for tests/test_cf_topk.py::test_world2: one rank (= one GPU) of a world-2 sharded matrix (the C router);
its top-k answers must equal the CPU checker's ranking of the whole table."""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import topk_suite as ts  # noqa: E402
from libsmatrix_b200.sharded import ShardedSparseMatrix  # noqa: E402


def main():
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    m = ShardedSparseMatrix(rank, world, rank, name=os.environ["SMX_TOPK_NAME"])
    rows = ts.Rows(seed=9, pool=60000)
    for L in (0, 1, 9, 10, 11, 256, 257, 4096, 4097, 50000):
        rows.add(L)
    rows.add(20000, "tie")
    rows.add(30000, "straddle")
    ref = ts.checker()
    xs, ys, vs = (np.concatenate([o[i] for o in rows.ops]).astype(np.uint32) for i in range(3))
    ref.apply("set", xs, ys, vs)
    sl = lambda a: a[rank * len(a) // world:(rank + 1) * len(a) // world]
    m.set_batch(sl(xs), sl(ys), sl(vs))
    q = ts.query_items(rows, np.random.default_rng(2))
    for k in (10, 100, 1024):
        want = ts.oracle_topk(ref, q, k)
        ts.assert_same(m.cf_topk_batch(q[rank::world], k), tuple(a[rank::world] for a in want), f"rank {rank} k={k}")
    m.close(); ref.close()
    print(f"rank {rank} ok")


if __name__ == "__main__":
    main()
