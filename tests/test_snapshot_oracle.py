""".smx snapshot and load kernels (k_snap_*, k_load_*) against the CPU checker's file mode and the independent
file reader, on the 1-lane and 32-lane simulators and (-m gpu) on a B200 at the library's full thresholds.
The scenarios are in tests/snapshot_oracle_suite.py."""
import os
import threading

import pytest

from libsmatrix_b200.matrix import SparseMatrix
from libsmatrix_b200.sharded import ShardedSparseMatrix
import snapshot_oracle_suite as so

_seq = [0]


@pytest.fixture(scope="module")
def sim():
    from hostsim import build as hb
    return hb.build()


@pytest.fixture(scope="module")
def sim32():
    from hostsim import build as hb
    return hb.build(defines=["-DSMX_SIM_WARP32"], suffix="_warp32")


@pytest.fixture
def knobs(monkeypatch):
    """simulator settings: a small directory, and loads cut into many windows, pieces and tiles"""
    monkeypatch.setenv("SMATRIX_DIR_LOG2", "8")
    monkeypatch.setenv("SMATRIX_LOAD_WINDOW", "4096")
    monkeypatch.setenv("SMATRIX_LOAD_CELLS", "700")
    monkeypatch.setenv("SMATRIX_SHARD_INBOX", "1024")
    monkeypatch.setenv("SMATRIX_SHARD_TIMEOUT", "60")


def sharded_opener(lib):
    """open_sharded(world, fname, fn) -> [fn(m, rank) for every rank]: ranks are threads of this process,
    each with its part of a file-backed sharded matrix, closed collectively (= the file is written)."""
    def open_sharded(world, fname, fn):
        _seq[0] += 1
        name = f"smxso_{os.getpid()}_{_seq[0]}"
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


def _lib(request, which):
    return request.getfixturevalue(which)


# ------------------------------------------------------------------ the simulators
@pytest.mark.parametrize("which", ["sim", "sim32"])
def test_save_side_and_reload_then_continue(request, knobs, which, tmp_path):
    lib = _lib(request, which)
    so.scenario_save_then_reload(lambda f: SparseMatrix(f, _lib_path=lib), tmp_path)


@pytest.mark.parametrize("which", ["sim", "sim32"])
def test_each_library_reloads_its_own_file(request, knobs, which, tmp_path):
    lib = _lib(request, which)
    so.scenario_each_reloads_its_own(lambda f: SparseMatrix(f, _lib_path=lib), tmp_path)


@pytest.mark.parametrize("which,worlds", [("sim", (1, 2, 3)), ("sim32", (2,))])
def test_checker_files_load_single_and_sharded(request, knobs, which, worlds, tmp_path):
    lib = _lib(request, which)
    so.scenario_load_checker_files(lambda f: SparseMatrix(f, _lib_path=lib), sharded_opener(lib), tmp_path, worlds)


@pytest.mark.parametrize("world", [2, 3])
def test_sharded_snapshot_is_the_checkers_file(sim, knobs, world, tmp_path):
    so.scenario_sharded_save(lambda f: SparseMatrix(f, _lib_path=sim), sharded_opener(sim), tmp_path, world)


def test_positional_load_hides_cells_only_where_the_reader_says(sim, knobs, tmp_path):
    so.scenario_hidden_cells(lambda f: SparseMatrix(f, _lib_path=sim), tmp_path)


# ------------------------------------------------------------------ B200, full thresholds
@pytest.mark.gpu
def test_gpu_save_side_and_reload_then_continue(tmp_path):
    """with rows of ~7 * 10^4 and 10^6 columns: k_snap_big over buckets of millions of cells"""
    so.scenario_save_then_reload(lambda f: SparseMatrix(f, device=0), tmp_path, huge=(70_000, 1_000_000))


@pytest.mark.gpu
def test_gpu_each_library_reloads_its_own_file(tmp_path):
    so.scenario_each_reloads_its_own(lambda f: SparseMatrix(f, device=0), tmp_path)


@pytest.mark.gpu
@pytest.mark.parametrize("small", [False, True], ids=["default-window", "small-window"])
def test_gpu_checker_files_load_single_and_sharded(monkeypatch, small, tmp_path):
    if small:
        monkeypatch.setenv("SMATRIX_LOAD_WINDOW", "65536")
        monkeypatch.setenv("SMATRIX_LOAD_CELLS", "5000")
    so.scenario_load_checker_files(lambda f: SparseMatrix(f, device=0), sharded_opener(None), tmp_path, worlds=(1,))


@pytest.mark.gpu
def test_gpu_positional_load_hides_cells_only_where_the_reader_says(tmp_path):
    so.scenario_hidden_cells(lambda f: SparseMatrix(f, device=0), tmp_path)
