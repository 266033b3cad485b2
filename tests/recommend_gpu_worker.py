"""Worker for tests/test_cf_recommend.py::test_world2: one rank (= one GPU) of a world-2 sharded matrix (the C router);
its basket recommendations must equal those of a single-GPU table with the same contents, bit for bit."""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import recommend_suite as rs  # noqa: E402
import topk_suite as ts  # noqa: E402
from libsmatrix_b200 import SparseMatrix  # noqa: E402
from libsmatrix_b200.sharded import ShardedSparseMatrix  # noqa: E402


def main():
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    m = ShardedSparseMatrix(rank, world, rank, name=os.environ["SMX_REC_NAME"])
    single = SparseMatrix(device=rank)
    ms, ref, t, baskets, named = rs.setup(lambda: single, 256, 4096)
    xs, ys, vs = t.ops()
    sl = lambda a: a[rank * len(a) // world:(rank + 1) * len(a) // world]
    m.set_batch(sl(xs), sl(ys), sl(vs))
    off, items = rs.flatten(baskets[rank::world])
    for k in (10, 100, 1024):
        want = single.cf_recommend_batch(off, items, k)
        ts.assert_same(want, rs.oracle(ref, off, items, k), f"single GPU k={k}")
        ts.assert_same(m.cf_recommend_batch(off, items, k), want, f"rank {rank} k={k}")
    m.close(); single.close(); ref.close()
    print(f"rank {rank} ok")


if __name__ == "__main__":
    main()
