"""Incremental checkpoints (smatrix_b200_checkpoint, smatrix_b200_shard_checkpoint) on the 1-lane and 32-lane
simulators: the dirty marks of the update kernel, the keep filter over the old directory, the appended blocks and
directory, the header switch and the fall-backs to a full snapshot; ranks of a sharded matrix are threads of this
process.  The scenarios are in tests/checkpoint_suite.py; tests/test_gpu_checkpoint.py runs them on a B200."""
import os
import threading

import pytest

from libsmatrix_b200.matrix import SparseMatrix
from libsmatrix_b200.sharded import ShardedSparseMatrix
import checkpoint_suite as cs

_seq = [0]


@pytest.fixture(scope="module")
def sim():
    from hostsim import build as hb
    return hb.build()


@pytest.fixture(scope="module")
def sim32():
    from hostsim import build as hb
    return hb.build(defines=["-DSMX_SIM_WARP32"], suffix="_warp32")


@pytest.fixture(autouse=True)
def knobs(monkeypatch):
    """a small directory, and loads cut into many windows, pieces and tiles; small router pieces, so that the old
    directory's entries are routed to their owners in several rounds"""
    monkeypatch.setenv("SMATRIX_DIR_LOG2", "8")
    monkeypatch.setenv("SMATRIX_LOAD_WINDOW", "4096")
    monkeypatch.setenv("SMATRIX_LOAD_CELLS", "700")
    monkeypatch.setenv("SMATRIX_SHARD_INBOX", "1024")
    monkeypatch.setenv("SMATRIX_SHARD_PIECE", "1024")
    monkeypatch.setenv("SMATRIX_SHARD_TIMEOUT", "60")


def sharded_opener(lib):
    """open_sharded(world, fname, fn) -> [fn(m, rank) for every rank], closed collectively"""
    def open_sharded(world, fname, fn):
        _seq[0] += 1
        name = f"smxck_{os.getpid()}_{_seq[0]}"
        out, errors = [None] * world, []

        def main(r):
            try:
                m = ShardedSparseMatrix(r, world, 0, name=name, _lib_path=lib, fname=fname)
                try:
                    out[r] = fn(m, r)
                finally:
                    m.close()
            except BaseException as e:                   # noqa: BLE001 - reported below
                import traceback
                errors.append(f"rank {r}: {e!r}\n{traceback.format_exc()}")
        ts = [threading.Thread(target=main, args=(r,)) for r in range(world)]
        for t in ts:
            t.start()
        for t in ts:
            t.join(timeout=600)
        assert not errors, "\n".join(errors)
        assert not any(t.is_alive() for t in ts), "a rank hangs"
        return out
    return open_sharded


def _make(lib):
    return lambda f: SparseMatrix(f, _lib_path=lib)


@pytest.mark.parametrize("which", ["sim", "sim32"])
def test_checkpoint_loads_like_a_snapshot_and_appends_only_dirty_rows(request, which, tmp_path):
    cs.scenario_equivalence(_make(request.getfixturevalue(which)), tmp_path)


@pytest.mark.parametrize("which", ["sim", "sim32"])
def test_generations_and_the_size_bound(request, which, tmp_path):
    cs.scenario_generations(_make(request.getfixturevalue(which)), tmp_path)


def test_dirty_rows_counts_every_write_api(sim, tmp_path):
    cs.scenario_dirty_counts(_make(sim), tmp_path)


def test_replaced_file_failure_and_missing_file(sim, tmp_path):
    cs.scenario_fallbacks(_make(sim), tmp_path)


@pytest.mark.parametrize("which", ["sim", "sim32"])
def test_foreign_files(request, which, tmp_path):
    cs.scenario_foreign(_make(request.getfixturevalue(which)), tmp_path)


@pytest.mark.parametrize("world", [2, 3, "2-warp32"])
def test_sharded_checkpoint(request, world, tmp_path):
    lib = request.getfixturevalue("sim")
    if world == "2-warp32":      # the keep filter's flags and prefix on the 32-lane lock-step simulator
        lib, world = request.getfixturevalue("sim32"), 2
    cs.scenario_sharded(_make(lib), sharded_opener(lib), tmp_path, world, {2: 3, 3: 1}[world])


@pytest.mark.parametrize("world", [2, 3])
def test_sharded_fallbacks_and_failure(sim, world, tmp_path):
    cs.scenario_sharded_fallbacks(_make(sim), sharded_opener(sim), tmp_path, world)
