"""Basket recommendation scenarios (smatrix_cf_recommend_batch), shared by the simulator builds and the GPU tests of
tests/test_cf_recommend.py.

The oracle takes every position's neighbour list from topk_suite.scores_of (the CPU checker's getrow + totals, the
lists smatrix_cf_neighbors_batch returns), sums each basket's pairs per id sequentially in position order (np.add.at
on position-ordered input is unbuffered and applies the additions in order, starting from 0.0), drops id 0 and the
basket's items, and ranks with topk_suite.rank.  The library's answer must be equal bit for bit.
"""
from __future__ import annotations

import numpy as np

import topk_suite as ts
from parity_suite import checker

U32 = np.uint32
ABSENT = ts.ABSENT


# ------------------------------------------------------------------ the oracle
def recommend_from_lists(boff, items, off, ids, sc, k):
    """Aggregate and rank per-position lists (off[n_items + 1], ids, sc) for the baskets boff over items."""
    boff = np.asarray(boff, dtype=np.int64)
    items = np.asarray(items, dtype=U32)
    off = np.asarray(off, dtype=np.int64)
    ids = np.asarray(ids, dtype=U32)
    sc = np.asarray(sc, dtype=np.float64)
    r_off, r_ids, r_sc = [0], [np.zeros(0, U32)], [np.zeros(0)]
    for i in range(len(boff) - 1):
        lo, hi = off[boff[i]], off[boff[i + 1]]
        u, inv = np.unique(ids[lo:hi], return_inverse=True)
        tot = np.zeros(len(u))
        np.add.at(tot, inv.reshape(-1), sc[lo:hi])
        keep = (u != 0) & ~np.isin(u, items[boff[i]:boff[i + 1]])
        r_ids.append(u[keep].astype(U32))
        r_sc.append(tot[keep])
        r_off.append(r_off[-1] + int(keep.sum()))
    return ts.rank(np.array(r_off, dtype=np.int64), np.concatenate(r_ids), np.concatenate(r_sc), k)


def oracle(ref, boff, items, k):
    return recommend_from_lists(boff, items, *ts.scores_of(ref, items), k)


def flatten(baskets):
    """list of item lists -> (offsets[n + 1] uint64, items uint32)"""
    lens = [len(b) for b in baskets]
    off = np.concatenate([[0], np.cumsum(lens)]).astype(np.uint64)
    items = np.concatenate([np.asarray(b, dtype=U32) for b in baskets] + [np.zeros(0, U32)]).astype(U32)
    return off, items


# ------------------------------------------------------------------ the table
class Table:
    """Pool ids 1..pool, each with a total at (b, 0); some of them (the items) get rows of exact lengths (column 0
    plus length - 1 columns drawn from the pool), so that items are candidates of each other and a basket's pairs
    are the sum of its items' row lengths.  Every row with hub=True holds column HUB = pool."""

    def __init__(self, seed: int, pool: int):
        self.rng = np.random.default_rng(seed)
        self.pool = pool
        self.hub = pool
        self.tot = self.rng.integers(1, 5000, pool + 1).astype(U32)
        self.rows: dict[int, tuple[np.ndarray, np.ndarray]] = {}
        self.next_item = 1
        self.by_len: dict[int, list[int]] = {}

    def length(self, a) -> int:
        return 1 + len(self.rows[a][0]) if a in self.rows else (1 if 1 <= a <= self.pool else 0)

    def row(self, length: int, hub: bool = True, self_loop: bool = False, cols=None, vals=None) -> int:
        a = self.next_item
        self.next_item += 1
        assert a < self.hub
        if cols is None:
            m = length - 1
            fixed = ([self.hub] if hub and m > 0 else []) + ([a] if self_loop and m > 1 else [])
            others = np.setdiff1d(np.arange(1, self.pool + 1), [a, self.hub])
            cols = np.concatenate([fixed, self.rng.choice(others, m - len(fixed), replace=False)]).astype(U32)
            vals = self.rng.integers(1, 60, m).astype(U32)
        self.rows[a] = (np.asarray(cols, U32), np.asarray(vals, U32))
        self.by_len.setdefault(self.length(a), []).append(a)
        return a

    def of_len(self, length: int) -> int:
        """an item whose row has exactly `length` pairs (a new one if there is none yet)"""
        return self.by_len[length][0] if self.by_len.get(length) else self.row(length)

    def ops(self):
        xs = [np.arange(1, self.pool + 1, dtype=U32)]
        ys = [np.zeros(self.pool, U32)]
        vs = [self.tot[1:]]
        for a, (c, v) in self.rows.items():
            xs.append(np.full(len(c), a, U32))
            ys.append(c)
            vs.append(v)
        return tuple(np.concatenate(z).astype(U32) for z in (xs, ys, vs))

    def apply(self, ms, ref):
        xs, ys, vs = self.ops()
        for m in ms:
            m.set_batch(xs, ys, vs)
        ref.apply("set", xs, ys, vs)

    def pairs(self, basket) -> int:
        return sum(self.length(int(a)) for a in basket)


def build_baskets(t: Table, warp_max: int, block_max: int):
    """-> (baskets, named): every basket shape of the contract, with their sizes around both class thresholds and
    over the big one.  `named` maps a shape to the indices of its baskets."""
    B: list[list[int]] = []
    named: dict[str, list[int]] = {}

    def add(kind, basket):
        named.setdefault(kind, []).append(len(B))
        B.append([int(a) for a in basket])

    singles = [t.row(L) for L in (2, 3, 9, 40)] + [t.row(12, self_loop=True), t.row(30, hub=False, self_loop=True)]
    add("empty", [])
    add("absent", list(ABSENT))
    for a in singles:
        add("single", [a])
    add("single", [t.hub])                                           # a row of column 0 only: nothing to offer
    add("repeated", [singles[0], singles[1], singles[0], singles[0], ABSENT[0], singles[1]])
    add("overlap", singles[:5])                                      # HUB at every position
    add("overlap", [t.hub] + singles[:4])                            # ... and excluded: it is in the basket
    x = t.row(0, cols=[t.next_item + 1], vals=[3])                   # x <-> y only: every candidate is excluded
    y = t.row(0, cols=[x], vals=[5])
    add("excluded", [x, y])
    add("excluded", [x, y, ABSENT[1], y])
    for thr in (warp_max, block_max):
        for d in (-1, 0, 1):
            L1 = thr // 2
            add("threshold", [t.of_len(L1), t.of_len(thr + d - L1)])
            add("threshold", [t.of_len(thr + d)])
    big = t.of_len(3 * block_max + 5)
    add("big", [big])
    add("big", [big, singles[0], big, ABSENT[0]])
    mid = [t.row(block_max // 3 + 50) for _ in range(4)]
    add("big", mid)
    add("big", mid[:2] + [t.hub, mid[0]])
    add("big", [t.of_len(L) for L in (100, 101, 102, 103)] * ((block_max // 400) + 2))
    return B, named


def sum_order_basket(t: Table, positions: int = 12, common: int = 24):
    """A basket whose items share `common` neighbours with scores of very different sizes (totals from 1 to 10^6),
    so that the sums depend on the order of the additions."""
    cands = np.arange(t.pool - common, t.pool, dtype=U32)
    t.tot[cands] = t.rng.choice(np.array([1, 2, 3, 7, 999_983, 1_000_000]), common).astype(U32)
    basket = []
    for j in range(positions):
        vals = t.rng.integers(1, 60, common).astype(U32)
        if j % 3 == 0:
            vals = t.rng.integers(1, 3, common).astype(U32)
        basket.append(t.row(0, cols=cands, vals=vals))
    return basket


def setup(make, warp_max, block_max, make_more=(), seed=5):
    """-> (matrices, checker, table, baskets, named)"""
    pool = 3 * block_max + 5 + block_max + 64
    t = Table(seed, pool)
    baskets, named = build_baskets(t, warp_max, block_max)
    order = sum_order_basket(t)
    named["order"] = [len(baskets)]
    baskets.append(order)
    for a in list(t.rows)[:3]:                                        # raise some totals: more varied scores
        t.tot[a] = 17
    ms = [make()] + [f() for f in make_more]
    ref = checker()
    t.apply(ms, ref)
    return ms, ref, t, baskets, named


def check_sum_order(ref, basket):
    """The basket's sums in position order differ from those in reverse order for some candidate (so equality with
    the oracle pins the order, not a tolerance); returns the forward sums by id."""
    off, ids, sc = ts.scores_of(ref, basket)
    fwd: dict[int, float] = {}
    rev: dict[int, float] = {}
    for j in range(len(basket)):
        for p in range(off[j], off[j + 1]):
            fwd[int(ids[p])] = fwd.get(int(ids[p]), 0.0) + float(sc[p])
    for j in reversed(range(len(basket))):
        for p in range(off[j], off[j + 1]):
            rev[int(ids[p])] = rev.get(int(ids[p]), 0.0) + float(sc[p])
    differ = [b for b in fwd if b != 0 and fwd[b] != rev[b]]
    assert differ, "the order basket does not tell the summation orders apart"
    return fwd


def scenario_baskets(make, warp_max, block_max, ks=(1, 7, 32, 1024), make_pieces=None):
    """Bit-exact answers for every k and basket shape; with make_pieces a table whose calls are cut into many pieces
    answers identically.  Returns the stats the tests assert on."""
    ms, ref, t, baskets, named = setup(make, warp_max, block_max, [make_pieces] if make_pieces else [])
    m = ms[0]
    off, items = flatten(baskets)
    is_big = [t.pairs(b) > block_max for b in baskets]
    assert all(is_big[i] for i in named["big"])
    st = {"n_big": sum(is_big)}
    for k in ks:
        want = oracle(ref, off, items, k)
        b0 = m.stat("rec_big")
        got = m.cf_recommend_batch(off, items, k)
        st.setdefault("rec_big", []).append(m.stat("rec_big") - b0)
        ts.assert_same(got, want, f"k={k}")
        for kind, idx in named.items():                              # each shape on its own, too
            sub = [baskets[i] for i in idx]
            so, si = flatten(sub)
            b0 = m.stat("rec_big")
            ts.assert_same(m.cf_recommend_batch(so, si, k), tuple(a[idx] for a in want), f"{kind}, k={k}")
            assert m.stat("rec_big") - b0 == sum(is_big[i] for i in idx), f"{kind}: the global sort ran where intended"
        if make_pieces:
            p = ms[1]
            b0 = p.stat("rec_big")
            ts.assert_same(p.cf_recommend_batch(off, items, k), got, f"k={k}, many pieces")
            st.setdefault("rec_big_pieces", []).append(p.stat("rec_big") - b0)
    for kind in ("empty", "absent", "excluded"):
        for i in named[kind]:
            assert got[0][i] == 0, kind
    fwd = check_sum_order(ref, baskets[named["order"][0]])
    i = named["order"][0]
    c = int(got[0][i])
    assert c == min(ks[-1], len([b for b in fwd if b != 0 and b not in baskets[i]]))
    for r in range(c):                                               # the forward sums themselves, bit for bit
        assert np.float64(fwd[int(got[1][i][r])]).view(np.uint64) == np.float64(got[2][i][r]).view(np.uint64)
    small = [b for b in baskets if t.pairs(b) <= block_max]
    so, si = flatten(small)
    b0 = m.stat("rec_big")
    ts.assert_same(m.cf_recommend_batch(so, si, 32), oracle(ref, so, si, 32), "small baskets")
    st["small_big"] = m.stat("rec_big") - b0
    a0 = m.stat("allocs")
    m.cf_recommend_batch(off, items, 1024)                            # the largest call again: scratch is reused
    st["allocs_again"] = m.stat("allocs") - a0
    for x in ms:
        x.close()
    ref.close()
    return st


def scenario_single_vs_topk(make, warp_max, block_max, ks=(1, 7, 32, 1024)):
    """A one-item basket [a] is cf_topk_batch([a], k + 2) without a and id 0, cut to k."""
    ms, ref, t, baskets, named = setup(make, warp_max, block_max)
    m = ms[0]
    items = np.array(sorted(t.rows)[:40] + [t.hub, int(ABSENT[0])], U32)
    off = np.arange(len(items) + 1, dtype=np.uint64)
    for k in ks:
        got = m.cf_recommend_batch(off, items, k)
        kk = min(k + 2, 1024)
        tc, ti, tsc = m.cf_topk_batch(items, kk)
        for j, a in enumerate(items):
            keep = [(b, s) for b, s in zip(ti[j][:tc[j]], tsc[j][:tc[j]]) if b != a and b != 0][:k]
            c = len(keep)
            if tc[j] < kk or c == k:                                 # the top-k list held every candidate needed
                assert got[0][j] == c, (a, k)
            assert [int(b) for b, _ in keep] == [int(b) for b in got[1][j][:c]], (a, k)
            assert np.array([s for _, s in keep], dtype=np.float64).view(np.uint64).tolist() == \
                got[2][j][:c].view(np.uint64).tolist(), (a, k)
    m.close()
    ref.close()


def scenario_d2h(make, k=10):
    """Host outputs: the answers and a few control words come down, never the neighbour lists."""
    ms, ref, t, baskets, named = setup(make, 256, 4096)
    m = ms[0]
    off, items = flatten(baskets)
    want = oracle(ref, off, items, k)
    d0 = m.stat("d2h_bytes")
    ts.assert_same(m.cf_recommend_batch(off, items, k), want, "host outputs")
    d = m.stat("d2h_bytes") - d0
    n = len(baskets)
    assert n * (12 * k + 4) <= d < n * (12 * k + 4) + 4096, (d, n)
    a0 = m.stat("allocs")
    ts.assert_same(m.cf_recommend_batch(off, items, k), want, "again")
    assert m.stat("allocs") == a0
    m.close()
    ref.close()
