"""Incremental checkpoints on B200s: the scenarios of tests/test_checkpoint.py at the library's full thresholds, a
config-2-shaped table with a 2^18-cell row checkpointed after touching about 1 % and then 30 % of its rows, and
sharded checkpoints at worlds 2 / 4 / 8 where the machine has the GPUs, reloaded at another world and read by the
C checker (and the reference, where it is built)."""
import os
import shutil
import subprocess
import sys

import numpy as np
import pytest
import torch

from libsmatrix_b200 import SparseMatrix
from oracle import cpu
import checkpoint_suite as cs
import smx_file

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))
U32 = np.uint32


def _make(f):
    return SparseMatrix(f, device=0)


def test_gpu_equivalence(tmp_path):
    cs.scenario_equivalence(_make, tmp_path, exact=False)


def test_gpu_generations(tmp_path):
    cs.scenario_generations(_make, tmp_path, exact=False)


def test_gpu_dirty_counts(tmp_path):
    cs.scenario_dirty_counts(_make, tmp_path)


def test_gpu_fallbacks(tmp_path):
    cs.scenario_fallbacks(_make, tmp_path)


def test_gpu_foreign(tmp_path):
    cs.scenario_foreign(_make, tmp_path)


def _view(m, rows):
    o, p = m.getrow_batch(rows)
    return (np.asarray(m.rowlen_batch(rows)).copy(), o.copy(), cpu.sort_rows(o, p),
            [m.stat(k) for k in ("rows", "nnz", "value_sum")])


def _loaded(path, tmp, rows, tag):
    m = SparseMatrix(shutil.copy(path, os.path.join(tmp, f"load_{tag}.smx")), device=0)
    try:
        return _view(m, rows)
    finally:
        m.close()


def test_world1_config2_shaped(tmp_path):
    """4 M ops over 60 000 rows of up to 256 columns with column-0 traffic and one row of ~2^18 cells; checkpoints
    after touching ~1 % and then ~30 % of the rows load like full snapshots taken at the same moments."""
    tmp = str(tmp_path)
    rng = np.random.default_rng(4242)
    n, n_rows = 4_000_000, 60_000
    keys = np.arange(n_rows, dtype=U32) * U32(2654435761)
    xs = keys[rng.integers(0, n_rows, n)]
    ys = rng.integers(1, 257, n).astype(U32)
    ys[rng.random(n) < 0.03] = 0
    big = rng.integers(0, n, 300_000)
    xs[big] = keys[99]                                  # one row of ~2^18 cells
    ys[big] = rng.integers(1, 2**32, len(big), dtype=np.uint64).astype(U32)
    dev = torch.device("cuda", 0)
    t = lambda a: torch.from_numpy(a.view(np.int32).copy()).to(dev)
    f = os.path.join(tmp, "c2.smx")
    m = SparseMatrix(f, device=0)
    m.incr_batch(t(xs), t(ys), t(rng.integers(1, 1000, n).astype(U32)))
    assert m.snapshot() == 0
    rows = np.unique(xs)
    for frac, seed in ((0.01, 1), (0.30, 2)):
        r2 = np.random.default_rng(seed)
        touched = np.unique(keys[r2.choice(n_rows, int(frac * n_rows), replace=False)])
        touched = np.unique(np.r_[touched, keys[99]])   # and the big row
        k = 20 * len(touched)
        ux = touched[r2.integers(0, len(touched), k)]
        uy = r2.integers(0, 300, k).astype(U32)        # new columns too, and column 0
        m.incr_batch(t(ux), t(uy), t(r2.integers(1, 50, k).astype(U32)))
        assert m.stat("dirty_rows") == len(touched)
        size0 = os.path.getsize(f)
        assert m.checkpoint() == 0
        assert cs.head_ptr(f) != 512 and os.path.getsize(f) > size0, "appended"
        ck = shutil.copy(f, os.path.join(tmp, f"ck{seed}.smx"))
        assert m.snapshot() == 0                        # the full snapshot of the same moment
        got, want = _loaded(ck, tmp, rows, f"ck{seed}"), _loaded(f, tmp, rows, f"full{seed}")
        for a, b in zip(got[:3], want[:3]):
            assert np.array_equal(a, b)
        assert got[3] == want[3]
        for x, (size, cells) in smx_file.read(ck).items():
            if x in set(touched[:200].tolist()):
                smx_file.check_row(x, size, cells)
    m.close()


def _ngpu():
    try:
        return torch.cuda.device_count()
    except Exception:
        return 0


def _run(phase, path, world, tag):
    env = dict(os.environ, WORLD_SIZE=str(world), SMX_NAME=f"smx_ck_{os.getpid()}_{tag}")
    procs = [subprocess.Popen([sys.executable, os.path.join(HERE, "checkpoint_gpu_worker.py"), phase, path],
                              env=dict(env, RANK=str(r)), stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
             for r in range(world)]
    outs = [p.communicate(timeout=900)[0] for p in procs]
    for r, (p, o) in enumerate(zip(procs, outs)):
        assert p.returncode == 0, f"{phase} at world {world}, rank {r} failed:\n{o[-3000:]}"
        assert f"rank {r} ok" in o


@pytest.mark.parametrize("world", [2, 4, 8])
def test_sharded_checkpoint_reloads_at_any_world(world, tmp_path):
    if _ngpu() < world:
        pytest.skip(f"needs {world} GPUs, this machine has {_ngpu()}")
    other = {2: 1, 4: 2, 8: 3}[world]
    f = str(tmp_path / "m.smx")
    _run("build", f, world, f"build{world}")
    _run("ck", f, world, f"ck{world}")
    ck = f + ".ck"
    assert cs.head_ptr(ck) != 512
    g = str(tmp_path / "other.smx")
    shutil.copy(ck, g)
    shutil.copy(f + ".npz", g + ".npz")
    _run("load", g, other, f"load{world}")
    for x, (size, cells) in smx_file.read(ck).items():
        smx_file.check_row(x, size, cells)
    import checkpoint_gpu_worker as w
    rows = np.unique(np.r_[w.stream()[0], w.update()[0]])
    want = np.load(f + ".npz")
    kinds = ["port"] + (["reference"] if cpu.have_reference() else [])
    for kind in kinds:
        c = cpu.CpuMatrix(kind, shutil.copy(ck, str(tmp_path / f"{kind}.smx")))
        o, p = c.getrow_many(rows)
        assert (o == want["offsets"]).all() and (cpu.sort_rows(o, p) == want["pairs"]).all(), kind
        c.close()
