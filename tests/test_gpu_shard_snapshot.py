"""File mode of the sharded matrix on B200s: a .smx file saved by one GPU or by W ranks (every rank writes its
part) reloads single-GPU and sharded at any world — the rows' row blocks expanded on each rank's GPU by the
loader's kernels — with the same cells, row lengths and totals; where the reference is built, it reads the file
too."""
import os
import shutil
import subprocess
import sys

import numpy as np
import pytest
import torch

from libsmatrix_b200 import SparseMatrix
from libsmatrix_b200.sharded import ShardedSparseMatrix
from oracle import cpu

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))
U32 = np.uint32


def _ngpu():
    try:
        return torch.cuda.device_count()
    except Exception:
        return 0


def _view(m, rows, sharded):
    o, p = m.getrow_batch(rows)
    stats = [m.stat(k) for k in ("rows", "nnz", "value_sum")]
    if sharded:
        stats = [m.sum(v) % 2**64 for v in stats]
    return np.asarray(m.rowlen_batch(rows)).copy(), o.copy(), cpu.sort_rows(o, p), stats


def test_world1_save_and_reload(tmp_path):
    """A config-2-shaped table (256 columns per row, column-0 traffic, a few million ops) on one B200."""
    rng = np.random.default_rng(4242)
    n = 4_000_000
    xs = rng.integers(0, 60_000, n).astype(U32) * U32(2654435761)
    ys = rng.integers(1, 257, n).astype(U32)
    ys[rng.random(n) < 0.03] = 0
    big = rng.integers(0, n, 300_000)
    xs[big] = U32(99)                                   # one row of ~2^18 cells: many tiles
    ys[big] = rng.integers(1, 2**32, len(big), dtype=np.uint64).astype(U32)
    dev = torch.device("cuda", 0)
    t = lambda a: torch.from_numpy(a.view(np.int32).copy()).to(dev)
    rows = np.unique(xs)
    f = str(tmp_path / "w1.smx")
    m = SparseMatrix(f, device=0)
    m.incr_batch(t(xs), t(ys), t(rng.integers(1, 1000, n).astype(U32)))
    want = _view(m, rows, False)
    m.close()
    g = shutil.copy(f, str(tmp_path / "single.smx"))
    m = SparseMatrix(g, device=0)
    single = _view(m, rows, False)
    for a, b in zip(single[1:3], want[1:3]):                # every cell comes back
        assert np.array_equal(a, b)
    assert single[3] == want[3]
    m.close()
    h = shutil.copy(f, str(tmp_path / "sharded.smx"))
    s = ShardedSparseMatrix(0, 1, 0, name=f"smx_snap_w1_{os.getpid()}", fname=h)
    got = _view(s, rows, True)
    for a, b in zip(got[:3], single[:3]):                   # and the row lengths are the single-GPU reload's:
        assert np.array_equal(a, b)                         # the reference's recount from the file's row sizes
    assert got[3] == want[3]
    assert s.snapshot() == 0
    s.close()


def _run(phase, path, world, tag):
    env = dict(os.environ, WORLD_SIZE=str(world), SMX_NAME=f"smx_snap_{os.getpid()}_{tag}")
    procs = [subprocess.Popen([sys.executable, os.path.join(HERE, "shard_snapshot_gpu_worker.py"), phase, path],
                              env=dict(env, RANK=str(r)), stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
             for r in range(world)]
    outs = [p.communicate(timeout=900)[0] for p in procs]
    for r, (p, o) in enumerate(zip(procs, outs)):
        assert p.returncode == 0, f"{phase} at world {world}, rank {r} failed:\n{o[-3000:]}"
        assert f"rank {r} ok" in o


@pytest.mark.parametrize("world", [2, 4, 8])
def test_save_at_w_reload_at_any_world(world, tmp_path):
    if _ngpu() < world:
        pytest.skip(f"needs {world} GPUs, this machine has {_ngpu()}")
    other = {2: 1, 4: 2, 8: 3}[world]
    f = str(tmp_path / "m.smx")
    _run("save", f, world, f"save{world}")
    for w in (world, other):
        g = str(tmp_path / f"at{w}.smx")
        shutil.copy(f, g)
        shutil.copy(f + ".npz", g + ".npz")
        _run("load", g, w, f"load{world}_{w}")
    if cpu.have_reference():                            # the reference reads the sharded file
        want = np.load(f + ".npz")
        r = cpu.CpuMatrix("reference", shutil.copy(f, str(tmp_path / "ref.smx")))
        xs = np.unique(np.asarray(__import__("shard_snapshot_gpu_worker").stream()[0]))
        assert (r.rowlen_many(xs) == want["rowlen"]).all()
        o, p = r.getrow_many(xs)
        assert (o == want["offsets"]).all() and (cpu.sort_rows(o, p) == want["pairs"]).all()
        r.close()
