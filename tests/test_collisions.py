"""Colliding row and column hashes, tile spills and staged host batches (tests/collision_suite.py): at reduced size
on the simulator builds of tests/hostsim/ (always), at full size on the CUDA library under the knobs that select
the other paths (`pytest -m gpu`)."""
import pytest

import collision_suite as cs
from libsmatrix_b200 import SparseMatrix


def test_mixers_invert():
    cs.check_mixers()


# ------------------------------------------------------------------ CPU: the simulator builds
@pytest.fixture(scope="module")
def sim():
    from hostsim import build as hb
    return hb.build()


@pytest.fixture(scope="module")
def sim_small_tiles():
    from hostsim import build as hb
    return hb.build(defines=["-DMIG_TILE_LOG=3u"], suffix="_smalltiles")


@pytest.fixture(scope="module")
def sim32():
    from hostsim import build as hb
    return hb.build(defines=["-DSMX_SIM_WARP32"], suffix="_warp32")


def _sim_env(monkeypatch):
    monkeypatch.setenv("SMATRIX_DIR_LOG2", "6")            # small directory floor: the shrink after a chunk can happen
    monkeypatch.setenv("SMATRIX_PARTITION_MIN", "16")      # chunks re-ordered by directory slice
    monkeypatch.setenv("SMATRIX_SLICE_LOG2", "3")
    monkeypatch.setenv("SMATRIX_GET_SLICE_MIN", "16")


@pytest.mark.parametrize("lib", ["sim", "sim32"])
def test_row_chains_sim(lib, request, monkeypatch):
    so = request.getfixturevalue(lib)
    _sim_env(monkeypatch)
    st = cs.scenario_row_chains(lambda: SparseMatrix(_lib_path=so), n_rows=300, low_bits=10)
    assert st["dir_grows"] > 0 and st["sliced_gets"] > 0


def test_chain_resizes_sim(sim, monkeypatch):
    _sim_env(monkeypatch)
    cs.scenario_chain_resizes(lambda: SparseMatrix(_lib_path=sim), n_rows=300, low_bits=12)


def test_column_runs_sim(sim, monkeypatch):
    _sim_env(monkeypatch)
    st = cs.scenario_column_runs(lambda: SparseMatrix(_lib_path=sim), n_cols=(20000, 30000, 40000), tile_log=10)
    assert st["spilled"] > 0


@pytest.mark.parametrize("spill_cap", [2, 1 << 16], ids=["spill-list-regrows", "spill-list-fits"])
def test_column_runs_small_tiles(sim_small_tiles, monkeypatch, spill_cap):
    _sim_env(monkeypatch)
    monkeypatch.setenv("SMATRIX_SPILL_CAP", str(spill_cap))
    st = cs.scenario_column_runs(lambda: SparseMatrix(_lib_path=sim_small_tiles), n_cols=(8000, 10000, 12000),
                                 tile_log=3)
    assert st["spilled"] > 0


def test_staged_host_batches_sim(sim, monkeypatch):
    _sim_env(monkeypatch)
    monkeypatch.setenv("SMATRIX_STAGE", "1024")
    cs.scenario_staged_host_batches(lambda: SparseMatrix(_lib_path=sim), pieces=13)


# ------------------------------------------------------------------ GPU: full size, one variant per knob
VARIANTS = {
    "default": {},
    "spill-cap-2": {"SMATRIX_SPILL_CAP": "2"},            # the spill list is too short: enlarged, tiles re-run
    "tiles-off": {"SMATRIX_MIGRATE_TILES": "0"},          # big rows re-placed by k_migrate_big (one global CAS per cell)
    "recycle-off": {"SMATRIX_RECYCLE": "0"},
    "presize-off": {"SMATRIX_PRESIZE": "0"},
    "arena": {"SMATRIX_ARENA_GIB": "2"},                  # directory, buckets and scratch carved from a reserved arena
}


@pytest.fixture(params=list(VARIANTS))
def variant(request, monkeypatch):
    for k, v in VARIANTS[request.param].items():
        monkeypatch.setenv(k, v)
    return VARIANTS[request.param]


def _common_asserts(st, env):
    if env.get("SMATRIX_RECYCLE") == "0":
        assert st["recycled"] == 0


@pytest.mark.gpu
def test_row_chains(variant):
    st = cs.scenario_row_chains(lambda: SparseMatrix(), n_rows=700, low_bits=22)
    assert st["dir_grows"] > 0
    assert st["sliced_gets"] > 0                          # the directory has many slices: mode 2 ordered the reads
    _common_asserts(st, variant)


@pytest.mark.gpu
def test_chain_resizes(variant):
    cs.scenario_chain_resizes(lambda: SparseMatrix(), n_rows=300, low_bits=22)


@pytest.mark.gpu
def test_column_runs(variant):
    st = cs.scenario_column_runs(lambda: SparseMatrix(), n_cols=(20000, 30000, 40000), tile_log=10)
    if variant.get("SMATRIX_MIGRATE_TILES") == "0":
        assert st["spilled"] == 0
    else:
        assert st["spilled"] > 0
    _common_asserts(st, variant)


@pytest.mark.gpu
def test_staged_host_batches(variant, monkeypatch):
    monkeypatch.setenv("SMATRIX_STAGE", "1024")
    cs.scenario_staged_host_batches(lambda: SparseMatrix(), pieces=13)
