"""Device scratch of the host shim (smx_host.c), on the 1-lane simulator build of tests/hostsim/.

Scratch buffers live on the handle and grow on demand with slack, so repeating a call with the same sizes makes
no cudaMalloc; a buffer that grows in the middle of a sequence (between two pieces of one top-k call, too) must
not be read after it was replaced (the simulator fills fresh allocations with 0xCD, so that shows up as a wrong
answer).  The copy and launch counters of a fixed call script are pinned to the values they have always had."""
import os

import numpy as np
import pytest

import topk_suite as ts
from oracle import cpu
from libsmatrix_b200 import SparseMatrix

U32 = np.uint32
OUT_ROW0 = 3_000_000_000          # rows of the *_batch_out ops: far from the item and neighbour rows


@pytest.fixture(scope="module")
def sim():
    from hostsim import build as hb
    return hb.build()


def _table(make, big_times=2):
    """-> (matrices, checker, Rows): the top-k boundary table (rows of every length class, ties, absent ids)."""
    return ts.build(make, 256, 4096, ks=(7,), big_times=big_times)


def _by_row(off, ids, scores):
    """cf_neighbors_batch answers in a fixed order: by item, then neighbour id (rows come in table order)."""
    seg = np.repeat(np.arange(len(off) - 1), np.diff(off.astype(np.int64)))
    o = np.lexsort((ids, seg))
    return ids[o], scores[o].view(np.uint64)


def check_cf_neighbors(m, ref, q):
    off, ids, sc = m.cf_neighbors_batch(q)
    w_off, w_ids, w_sc = ts.scores_of(ref, q)
    assert (off.astype(np.int64) == w_off).all(), "cf_neighbors: offsets differ"
    got, want = _by_row(off, ids, sc), _by_row(w_off, w_ids, w_sc)
    assert (got[0] == want[0]).all() and (got[1] == want[1]).all(), "cf_neighbors: neighbours or scores differ"


def check_getrow_batch(m, ref, q):
    off, pairs = m.getrow_batch(q)
    w_off, w_pairs = ref.getrow_many(q)
    assert (off == w_off).all(), "getrow_batch: row sizes differ"
    assert (cpu.sort_rows(off, pairs) == cpu.sort_rows(w_off, w_pairs)).all(), "getrow_batch: pairs differ"


def check_getrow(m, ref, xs):
    for x in xs:
        assert m.getRow(int(x)) == dict(ref.getrow(int(x))), f"getrow {x}"


def check_topk(m, ref, q, k):
    ts.assert_same(m.cf_topk_batch(q, k), ts.oracle_topk(ref, q, k), f"cf_topk k={k}")


def check_batch_out(m, ref, n, seed):
    rng = np.random.default_rng(seed)
    xs = (OUT_ROW0 + rng.integers(0, 64, n)).astype(U32)
    ys = rng.integers(1, 500, n).astype(U32)
    vs = rng.integers(1, 1000, n).astype(U32)
    got = m.incr_batch_out(xs, ys, vs)
    assert (got == ref.apply("incr", xs, ys, vs, want_out=True)).all(), f"incr_batch_out n={n}"


def test_repeated_calls_make_no_cudamalloc(sim):
    """The same calls twice: the second round allocates nothing (cf_neighbors_batch with host outputs included)."""
    ms, ref, rows = _table(lambda: SparseMatrix(_lib_path=sim))
    m = ms[0]
    q = ts.query_items(rows, np.random.default_rng(21))
    biggest = max(rows.items, key=lambda a: len(ref.getrow_many([a])[1]))
    allocs = []
    for _ in range(2):
        check_cf_neighbors(m, ref, q)
        check_getrow_batch(m, ref, q)
        check_getrow(m, ref, [biggest, rows.items[0], ts.ABSENT[0]])
        check_topk(m, ref, q, 7)
        check_batch_out(m, ref, 5000, seed=1)
        allocs.append(m.stat("allocs"))
    assert allocs[1] == allocs[0], f"the second round made {allocs[1] - allocs[0]} cudaMalloc calls"
    m.close(); ref.close()


def test_growth_inside_a_sequence(sim, monkeypatch):
    """Calls of increasing size: every read-side buffer regrows on the way, and on a table whose top-k calls are cut
    into many pieces (SMATRIX_TOPK_PAIRS small), between the pieces of one call (items ordered by row length)."""
    monkeypatch.setenv("SMATRIX_TOPK_PAIRS", "2055")
    ms, ref, rows = _table(lambda: SparseMatrix(_lib_path=sim), big_times=3)
    m = ms[0]
    lens = {a: len(ref.getrow_many([a])[1]) for a in rows.items}
    by_len = np.array(sorted(rows.items, key=lambda a: (lens[a], a)), U32)
    grew = 0
    for i, hi in enumerate((4, 12, 24, len(by_len))):
        q = by_len[:hi]
        a0 = m.stat("allocs")
        check_getrow_batch(m, ref, q)
        check_cf_neighbors(m, ref, q)
        for k in (1, 32, 1024):
            check_topk(m, ref, q, k)
        check_getrow(m, ref, [int(q[-1])])
        check_batch_out(m, ref, 3000 * 4 ** i, seed=10 + i)
        grew += m.stat("allocs") > a0
    assert grew == 4, "every step should have grown some buffer"
    assert m.stat("topk_big") > 0
    m.close(); ref.close()


# launches, h2d_bytes, d2h_bytes after each step of _script, as the host shim has always counted them (recorded
# before its scratch handling was unified; no step may change them)
COUNTERS = [("set_batch", 12, 54072, 8040), ("getrow_batch", 21, 54128, 20248), ("cf_neighbors", 31, 54184, 38356),
            ("cf_topk", 44, 54212, 38836), ("incr_batch_out", 53, 60212, 44052), ("get_batch", 54, 62612, 45252),
            ("rowlen_batch", 55, 62640, 45280), ("single ops", 69, 62688, 54948), ("getrow", 75, 62696, 54964),
            ("value_sum", 77, 62696, 58184), ("snapshot", 85, 62696, 569132)]


def _script(m):
    rows = ts.Rows(seed=2, pool=1500)
    for L in (0, 1, 5, 300, 1200):
        rows.add(L)
    xs, ys, vs = (np.concatenate([o[i] for o in rows.ops]).astype(U32) for i in range(3))
    q = np.array(rows.items + rows.items[:2], U32)
    steps = [
        ("set_batch", lambda: m.set_batch(xs, ys, vs)),
        ("getrow_batch", lambda: m.getrow_batch(q)),
        ("cf_neighbors", lambda: m.cf_neighbors_batch(q)),
        ("cf_topk", lambda: m.cf_topk_batch(q, 5)),
        ("incr_batch_out", lambda: m.incr_batch_out(xs[:500], ys[:500], vs[:500])),
        ("get_batch", lambda: m.get_batch(xs[:300], ys[:300])),
        ("rowlen_batch", lambda: m.rowlen_batch(q)),
        ("single ops", lambda: (m.set(5, 6, 7), m.incr(5, 6, 1), m.decr(5, 7, 0), m.get(5, 6), m.rowlen(int(q[3])))),
        ("getrow", lambda: m.getRow(int(q[4]))),
        ("value_sum", lambda: m.stat("value_sum")),
        ("snapshot", lambda: m._lib.smatrix_b200_snapshot(m._handle())),
    ]
    out = []
    for name, f in steps:
        f()
        out.append((name, m.stat("launches"), m.stat("h2d_bytes"), m.stat("d2h_bytes")))
    return out


def test_counters_unchanged(sim, tmp_path):
    m = SparseMatrix(str(tmp_path / "t.smx"), _lib_path=sim)
    got = _script(m)
    m.close()
    assert os.path.getsize(tmp_path / "t.smx") > 0
    assert got == COUNTERS
