"""Worker for tests/test_export.py::test_world2: one rank (= one GPU) of a world-2 sharded matrix (the C router); its
listing and sorted rows must equal those of a single-GPU table fed the same stream, and the checker's."""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import export_suite as es  # noqa: E402
from test_export import Recorder, replay  # noqa: E402
from libsmatrix_b200 import SparseMatrix  # noqa: E402
from libsmatrix_b200.sharded import ShardedSparseMatrix  # noqa: E402


def main():
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    m = ShardedSparseMatrix(rank, world, rank, name=os.environ["SMX_EXPORT_NAME"])
    single, ref, rec = SparseMatrix(device=rank), es.port(), Recorder()
    es.build_shapes(es.Stream([single, rec], ref), 256, 4096, 10**5)
    replay(m, rec.batches, rank, world)
    keys = single.rows()
    assert (keys == es.oracle_rows(ref)).all(), "single GPU"
    assert (m.rows() == keys).all(), f"rank {rank}: rows()"
    for per in (1, 7, 1000):
        got = np.concatenate([m.rows(int(s), per) for s in [0] + [int(k) + 1 for k in keys[per - 1:-1:per]]])
        assert (got == keys).all(), f"rank {rank}: pages of {per}"
    d_keys = m.rows(device=True)
    assert (d_keys.cpu().numpy().view(np.uint32) == keys).all(), f"rank {rank}: device rows()"
    mine = keys[rank::world]
    off, pairs = m.getrow_sorted_batch(mine)
    soff, spairs = single.getrow_sorted_batch(mine)
    assert (off == soff).all() and (pairs == spairs).all(), f"rank {rank}: sorted rows"
    es.assert_rows_equal(off, pairs, ref, mine, f"rank {rank}")
    m.close(); single.close(); ref.close()
    print(f"rank {rank} ok")


if __name__ == "__main__":
    main()
