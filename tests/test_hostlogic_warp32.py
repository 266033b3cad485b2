"""The host logic AND the warp-cooperative device code on the CPU: the kernel sources compiled against the 32-lane
lock-step variant of the simulator (tests/hostsim/warp_sched.cpp — every thread of a block is a fiber, collectives
exchange values as the hardware primitives are specified).  Unlike the 1-lane simulator of test_hostlogic.py this
runs the __match_any_sync pre-aggregation, the shuffle scans, the ballots of the getrow compaction, the per-warp
prefix tables of the partition scatter and every shared-memory stage behind a barrier.  Slow (a context switch per
collective), so the scenarios are small; the parity tests proper stay tests/test_gpu_parity.py."""
import ctypes as C

import pytest

import parity_suite as ps
from libsmatrix_b200 import SparseMatrix


@pytest.fixture(scope="module")
def sim32():
    from hostsim import build as hb
    return hb.build(defines=["-DSMX_SIM_WARP32"], suffix="_warp32")


@pytest.fixture
def make(sim32, monkeypatch):
    monkeypatch.setenv("SMATRIX_DIR_LOG2", "8")             # directory growth on every test
    monkeypatch.setenv("SMATRIX_CHUNK", "5000")             # multi-chunk batches
    monkeypatch.setenv("SMATRIX_PARTITION_MIN", "16")       # chunks re-ordered by directory slice
    monkeypatch.setenv("SMATRIX_SLICE_LOG2", "3")
    monkeypatch.setenv("SMATRIX_GET_SLICE_MIN", "16")       # point reads in slice order
    return lambda: SparseMatrix(_lib_path=sim32)


def test_primitives_selftest(sim32):
    lib = C.CDLL(sim32)
    assert lib.smx_sim_warp_selftest() == 0


def test_java_cases_and_quirks(make):
    ps.scenario_java_cases(make, grid=200)
    ps.scenario_quirks(make)
    ps.scenario_empty_and_ragged(make)


def test_random_stream(make):
    ps.scenario_random(make, 3, n=12000)


def test_set_last_writer(make):
    ps.scenario_set_last_writer(make)


def test_col0_ordering(make):
    ps.scenario_col0_ordering(make)


def test_preaggregation_of_hot_keys(make):
    ps.scenario_cf(make, n_baskets=600, n_items=120)        # duplicate (x, y) inside warps: __match_any_sync + segmented sum


def test_growth_and_recycling(make):
    ps.scenario_recycling_churn(make, waves=4, rows_per_wave=120)
    ps.scenario_big_row(make, n_cols=12000)


def test_read_path(make):
    ps.scenario_read_path_zipf(make, n_rows=1200, max_len=6000)
    ps.scenario_sliced_gets(make, n_rows=300, n_cols=40, n_ops=6000, sizes=(1, 7, 17, 600, 5001))


def test_batch_out_and_cf_read_side(make):
    ps.scenario_batch_out(make, n=9000)
    ps.scenario_cf_read_side(make, n_baskets=500, n_items=100)


def test_chunks_without_column0(make, monkeypatch):
    monkeypatch.setenv("SMATRIX_WIDE_SLICES", "1")
    ps.scenario_no_column0(make, n=9000, n_rows=2500)


def test_snapshot_export_kernels(sim32, tmp_path, monkeypatch):
    """K9: the row blocks of the .smx file are laid out by k_snap_* (one warp per row, linear probing in the reference's
    y % size layout) — both directions against the reference's own file mode."""
    import snapshot_suite as ss
    monkeypatch.setenv("SMATRIX_DIR_LOG2", "6")
    ss.scenario_snapshot_interchange(lambda f: SparseMatrix(f, _lib_path=sim32), tmp_path)


def test_snapshot_export_kernels_roundtrip(sim32, tmp_path, monkeypatch):
    """K9: the same kernels, ours -> ours with big rows (no reference build needed)."""
    import snapshot_suite as ss
    monkeypatch.setenv("SMATRIX_DIR_LOG2", "6")
    ss.scenario_snapshot_roundtrip_big(lambda f: SparseMatrix(f, _lib_path=sim32), tmp_path, n_rows=1500)
