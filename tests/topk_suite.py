"""Top-k recommender scenarios (smatrix_cf_topk_batch), shared by the simulator builds and the GPU tests of
tests/test_cf_topk.py.

The oracle for every item is the CPU checker's getrow + get(b, 0) with the arithmetic of
parity_suite.scenario_cf_read_side, ranked by score descending, then id ascending
(np.lexsort((ids, -scores))); the library's answer must be equal bit for bit: ids, the doubles' bits, order.
"""
from __future__ import annotations

import numpy as np

from parity_suite import checker

U32 = np.uint32
NONE = np.uint32(0xFFFFFFFF)


# ------------------------------------------------------------------ the oracle
def scores_of(ref, items):
    """(offsets[n+1], neighbour ids, scores) exactly as smatrix_cf_neighbors_batch defines them."""
    items = np.ascontiguousarray(items, dtype=U32)
    off, pairs = ref.getrow_many(items)
    off = off.astype(np.int64)
    seg = np.repeat(np.arange(len(items)), np.diff(off))
    a_tot = ref.get_many(items, np.zeros(len(items), U32)).astype(np.float64)
    b = pairs[:, 0].astype(U32)
    b_tot = ref.get_many(b, np.zeros(len(b), U32))
    b_tot = np.where(b_tot == 0, 1, b_tot).astype(np.float64)
    num = pairs[:, 1].astype(np.float64)
    den = np.sqrt(a_tot[seg]) * np.sqrt(b_tot)
    zero = (den == 0.0) | (num > den)
    sc = np.divide(num, den, out=np.zeros(len(num)), where=~zero)
    return off, b, sc


def rank(off, ids, sc, k):
    """Segmented ranking of CSR (off, ids, sc) -> the fixed-width answer (counts, ids[n,k], scores[n,k])."""
    off = np.asarray(off, dtype=np.int64)
    n = len(off) - 1
    seg = np.repeat(np.arange(n), np.diff(off))
    order = np.lexsort((ids, -sc, seg))
    pos = np.arange(len(order)) - off[seg[order]]
    keep = pos < k
    counts = np.minimum(np.diff(off), k).astype(U32)
    out_ids = np.full((n, k), NONE, U32)
    out_sc = np.full((n, k), -1.0)
    out_ids[seg[order][keep], pos[keep]] = ids[order][keep]
    out_sc[seg[order][keep], pos[keep]] = sc[order][keep]
    return counts, out_ids, out_sc


def oracle_topk(ref, items, k):
    return rank(*scores_of(ref, items), k)


def assert_same(got, want, what=""):
    gc, gi, gs = (np.asarray(a) for a in got)
    wc, wi, ws = want
    assert gc.shape == wc.shape and gi.shape == wi.shape and gs.shape == ws.shape, what
    bad = np.nonzero(gc.astype(U32) != wc)[0]
    assert not len(bad), f"{what}: counts differ at items {bad[:8]}: {gc[bad[:8]]} vs {wc[bad[:8]]}"
    bad = np.nonzero((gi.astype(U32) != wi).any(1))[0]
    assert not len(bad), f"{what}: ids differ for {len(bad)} items, first {bad[0]}: {gi[bad[0]][:12]} vs {wi[bad[0]][:12]}"
    bad = np.nonzero((gs.view(np.uint64) != ws.view(np.uint64)).any(1))[0]
    assert not len(bad), f"{what}: scores differ for {len(bad)} items, first {bad[0]}"


# ------------------------------------------------------------------ the table
ITEM0 = 1_000_000      # item rows are ITEM0 + i; neighbour ids are 1 .. pool (their totals sit at (b, 0))
ABSENT = np.array([7_777_777, 999_999_999], U32)


class Rows:
    """A table whose item rows have chosen lengths and score shapes, built with one set_batch (so a row's length
    is exact: its columns plus the column-0 pair)."""

    def __init__(self, seed: int, pool: int):
        self.rng = np.random.default_rng(seed)
        self.pool = pool
        self.tie_lo = pool + 1                                   # neighbours with one common total: equal scores
        self.ops = [(np.arange(1, pool + 1, dtype=U32), np.zeros(pool, U32),
                     self.rng.integers(1, 5000, pool).astype(U32))]
        self.ops.append((np.arange(self.tie_lo, self.tie_lo + pool, dtype=U32), np.zeros(pool, U32),
                         np.full(pool, 100, U32)))
        self.items: list[int] = []
        self.kinds: dict[str, list[int]] = {}

    def add(self, length: int, kind: str = "mixed"):
        """kind: mixed (varied scores with ties), zeros (most scores 0: num > den), tie (every neighbour the same
        score), straddle (a few high scores, then a tie group of length // 2, then low ones)."""
        a = ITEM0 + len(self.items)
        self.items.append(a)
        self.kinds.setdefault(kind, []).append(a)
        if length == 0:                                          # absent item
            return a
        m = length - 1
        rng = self.rng
        if kind == "tie":
            cols = self.tie_lo + rng.choice(self.pool, m, replace=False).astype(U32)
            vals = np.full(m, 7, U32)
            a_tot = 400
        elif kind == "straddle":
            cols = self.tie_lo + rng.choice(self.pool, m, replace=False).astype(U32)
            g = length // 2
            vals = np.concatenate([np.full(5, 50), np.full(g, 7), np.ones(m - 5 - g)]).astype(U32)
            a_tot = 400
        else:
            cols = 1 + rng.choice(self.pool, m, replace=False).astype(U32)
            vals = rng.integers(1, 60, m).astype(U32)
            a_tot = 4 if kind == "zeros" else int(rng.integers(1, 5000))
        self.ops.append((np.full(m + 1, a, U32), np.concatenate([[0], cols]).astype(U32),
                         np.concatenate([[a_tot], vals]).astype(U32)))
        return a

    def apply(self, ms, ref):
        xs, ys, vs = (np.concatenate([o[i] for o in self.ops]).astype(U32) for i in range(3))
        for m in ms:
            m.set_batch(xs, ys, vs)
        ref.apply("set", xs, ys, vs)


def boundary_rows(warp_max: int, block_max: int, ks=(1, 7, 32, 1024), big_times: int = 3):
    """Row sizes around every k and every class boundary, and several times the big threshold."""
    sizes = {0, 1, 2}
    for k in ks:
        sizes |= {k - 1, k, k + 1}
    for t in (warp_max, block_max):
        sizes |= {t - 1, t, t + 1}
    sizes.add(big_times * block_max + 5)
    return sorted(s for s in sizes if s >= 0)


def build(make, warp_max, block_max, ks=(1, 7, 32, 1024), big_times=3, make_more=()):
    """-> (matrices, checker, Rows): the boundary sizes (mixed scores), zero-tailed rows, an all-tie big row, and a
    tie group larger than the block class that straddles every k."""
    sizes = boundary_rows(warp_max, block_max, ks, big_times)
    rows = Rows(seed=len(sizes), pool=max(sizes) + block_max + 16)
    for s in sizes:
        rows.add(s)
    rows.add(min(block_max // 2, 300), "zeros")
    rows.add(block_max + 300, "zeros")
    rows.add(2 * block_max + 100, "tie")
    rows.add(3 * block_max, "straddle")
    ms = [make()] + [f() for f in make_more]
    ref = checker()
    rows.apply(ms, ref)
    return ms, ref, rows


def query_items(rows: Rows, rng) -> np.ndarray:
    """Every item, shuffled, with duplicates and absent ids."""
    items = np.array(rows.items, U32)
    q = np.concatenate([items, items[rng.integers(0, len(items), 9)], ABSENT, items[:3]])
    rng.shuffle(q)
    return q.astype(U32)


def scenario_boundaries(make, warp_max, block_max, ks=(1, 7, 32, 1024), big_times=3, make_pieces=None):
    """Bit-exact answers for every k over the boundary rows; with make_pieces, a table whose calls are cut into
    many pieces ($SMATRIX_TOPK_PAIRS small) answers identically.  Returns the stats the tests assert on."""
    ms, ref, rows = build(make, warp_max, block_max, ks, big_times, [make_pieces] if make_pieces else [])
    m = ms[0]
    rng = np.random.default_rng(3)
    q = query_items(rows, rng)
    st = {}
    for k in ks:
        got = m.cf_topk_batch(q, k)
        assert_same(got, oracle_topk(ref, q, k), f"k={k}")
        for dup in np.unique(q):                                 # duplicate items: identical answers
            w = np.nonzero(q == dup)[0]
            if len(w) > 1:
                assert (got[1][w] == got[1][w[0]]).all() and (got[2][w].view(np.uint64) == got[2][w[0]].view(np.uint64)).all()
        if make_pieces:
            assert_same(ms[1].cf_topk_batch(q, k), got, f"k={k}, many pieces")
    # the select's own paths: the all-tie row needs the id digits (more than 8 passes of 8 bits)
    for kind in ("tie", "straddle"):
        b0, p0 = m.stat("topk_big"), m.stat("topk_passes")
        items = np.array(rows.kinds[kind], U32)
        for k in ks:
            assert_same(m.cf_topk_batch(items, k), oracle_topk(ref, items, k), f"{kind}, k={k}")
        st[kind + "_big"] = m.stat("topk_big") - b0
        st[kind + "_passes"] = m.stat("topk_passes") - p0
    small = np.array([a for a in rows.items if len(ref.getrow_many([a])[1]) <= block_max], U32)
    b0, p0 = m.stat("topk_big"), m.stat("topk_passes")
    assert_same(m.cf_topk_batch(small, 32), oracle_topk(ref, small, 32), "small rows")
    st["small_big"], st["small_passes"] = m.stat("topk_big") - b0, m.stat("topk_passes") - p0
    a0 = m.stat("allocs")
    m.cf_topk_batch(q, 1024)                                     # the largest call again: scratch is reused
    st["allocs_again"] = m.stat("allocs") - a0
    for x in ms:
        x.close()
    ref.close()
    return st


def scenario_d2h(make, k=10):
    """Host outputs: the answers and a few control words come down, never the neighbour lists."""
    ms, ref, rows = build(make, 256, 4096, ks=(k,), big_times=2)
    m = ms[0]
    q = np.array(rows.items, U32)
    d0 = m.stat("d2h_bytes")
    assert_same(m.cf_topk_batch(q, k), oracle_topk(ref, q, k), "host outputs")
    d = m.stat("d2h_bytes") - d0
    pairs = len(ref.getrow_many(q)[1])
    assert len(q) * (12 * k + 4) <= d < len(q) * (12 * k + 4) + 4096, (d, len(q), pairs)
    m.close(); ref.close()
