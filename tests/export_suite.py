"""Enumeration scenarios (smatrix_list_rows, smatrix_getrow_sorted_batch, smatrix_b200_sort_rows), shared by the
simulator builds and the GPU tests of tests/test_export.py.

The oracle shares no code with the library:
  row set   the directory of the C checker's own .smx file: CpuMatrix("port") is fed the same stream, saves itself,
            and tests/smx_file.py (numpy only) reads the row keys back;
  pairs     sorted(ref.getrow(x)) of the checker, compared in order with the library's output, which is never
            sorted here (a build that skipped the device sort fails).
"""
from __future__ import annotations

import os
import tempfile

import numpy as np

import smx_file
from oracle import cpu

U32 = np.uint32
TOP = 0xFFFFFFFF


def port() -> cpu.CpuMatrix:
    return cpu.CpuMatrix("port")


def oracle_rows(ref: cpu.CpuMatrix) -> np.ndarray:
    """the checker's row keys, from its own file"""
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, "ref.smx")
        ref.save(path)
        return np.array(sorted(smx_file.read(path)), dtype=U32)


def want_pairs(ref, x) -> np.ndarray:
    return np.array(sorted(ref.getrow(int(x))), dtype=U32).reshape(-1, 2)


def assert_rows_equal(offsets, pairs, ref, keys, what=""):
    offsets = np.asarray(offsets, dtype=np.int64)
    pairs = np.asarray(pairs).view(U32).reshape(-1, 2)
    assert len(offsets) == len(keys) + 1 and offsets[0] == 0, what
    for i, x in enumerate(np.asarray(keys).astype(np.int64) & 0xFFFFFFFF):   # int32 keys of a tensor too
        got = pairs[offsets[i]:offsets[i + 1]]
        want = want_pairs(ref, x)
        assert got.shape == want.shape and (got == want).all(), f"{what}: row {int(x)}: {got[:6]} vs {want[:6]}"


class Stream:
    """A stream of batches applied to every handle and to the checker alike."""

    def __init__(self, ms, ref, seed=7):
        self.ms, self.ref = ms, ref
        self.rng = np.random.default_rng(seed)

    def op(self, op, xs, ys, vs):
        xs, ys, vs = (np.asarray(a, dtype=np.uint64).astype(U32) for a in (xs, ys, vs))
        for m in self.ms:
            getattr(m, op + "_batch")(xs, ys, vs)
        self.ref.apply(op, xs, ys, vs)

    def row(self, x, length, col0=False, extra=()):
        """row x with `length` pairs: column 0 (when col0) plus distinct columns != 0, `extra` among them"""
        m = length - (1 if col0 else 0)
        fixed = [c for c in extra if c][:m]
        cols = np.concatenate([np.array(fixed, dtype=np.uint64),
                               self.rng.choice(np.arange(1, 8 * length + 64, dtype=np.uint64) + 1000, m - len(fixed),
                                               replace=False)])
        vals = self.rng.integers(1, 1 << 32, m, dtype=np.uint64)
        if col0:
            cols, vals = np.concatenate([[0], cols]), np.concatenate([[self.rng.integers(1, 1000)], vals])
        self.op("set", np.full(len(cols), x), cols, vals)


def build_shapes(st: Stream, warp_max: int, block_max: int, big: int) -> dict[str, list[int]]:
    """Every row shape of the contract; -> {shape: row keys}."""
    named: dict[str, list[int]] = {}
    add = lambda kind, x: named.setdefault(kind, []).append(x)
    for x in (0, 1, 1 << 31, TOP):                              # the extreme keys, with the extreme columns
        st.row(x, 9, col0=True, extra=(TOP, 1 << 31, (1 << 31) - 1, 1))
        add("keys", x)
    st.op("incr", [11, 12], [0, 0], [5, 7])                      # column 0 only
    add("col0", 11); add("col0", 12)
    st.op("incr", [13, 13], [0, 0], [5, 0])
    st.op("decr", [13], [0], [5])                                # column 0 back to 0: no pairs
    st.op("set", [14], [0], [0])                                 # created by set 0: no pairs
    add("empty", 13); add("empty", 14)
    st.op("set", [15, 15, 15], [3, TOP, 9], [0, 0, 4])           # zero-valued cells on columns != 0 stay live
    add("zeros", 15)
    x = 100
    for L in (1, 2, 3, 4, 5):                                    # inline rows and 5-cell rows
        st.row(x, L); add("inline", x); x += 1
        st.row(x, L + 1, col0=True); add("inline", x); x += 1
    for L in (20, 100, 200, 400, 1500, 5000):                    # buckets of 32 .. 8192 cells (fill and chunks)
        st.row(x, L); add("bucket", x); x += 1
    for thr in (warp_max, block_max):
        for d in (-1, 0, 1):
            st.row(x, thr + d); add("threshold", x); x += 1
            st.row(x, thr + d, col0=True); add("threshold", x); x += 1
    st.row(x, big, col0=True, extra=(TOP, 1 << 31)); add("big", x); x += 1
    for k in range(5):                                           # several big rows: groups of them
        st.row(x, block_max + 1 + 37 * k, col0=k % 2 == 0); add("big", x); x += 1
    return named


def check_listing(m, ref, what=""):
    """rows() against the checker's file, and paging through it"""
    want = oracle_rows(ref)
    got = m.rows()
    assert got.dtype == U32 and (got == want).all(), f"{what}: {len(got)} rows vs {len(want)}"
    for per in (1, 7, 1000):
        pages, start = [], 0
        while True:
            p = m.rows(start, per)
            pages.append(p)
            if len(p) < per or p[-1] == TOP:
                break
            start = int(p[-1]) + 1
        assert (np.concatenate(pages) == want).all(), f"{what}: pages of {per}"
    return want


def scenario_shapes(make, warp_max, block_max, big, make_pieces=None):
    """Every shape and class, listed and read back sorted; with make_pieces a handle whose big segments are cut into
    many groups answers the same.  -> stats"""
    ms = [make()] + ([make_pieces()] if make_pieces else [])
    m, ref = ms[0], port()
    assert m.rows().shape == (0,) and m._lib.smatrix_list_rows(m._handle(), 0, None, 0) == 0
    sentinel = np.full(4, 77, U32)
    assert m._lib.smatrix_list_rows(m._handle(), 0, sentinel.ctypes.data, 4) == 0 and (sentinel == 77).all()
    st = Stream(ms, ref)
    named = build_shapes(st, warp_max, block_max, big)
    keys = check_listing(m, ref, "shapes")
    assert set(x for v in named.values() for x in v) == set(keys.tolist())
    assert len(keys) == m.stat("rows")
    lens = np.array([len(ref.getrow(int(x))) for x in keys])
    n_big = int((lens > block_max).sum())
    b0 = m.stat("sort_big")
    off, pairs = m.getrow_sorted_batch(keys)
    assert m.stat("sort_big") - b0 == n_big
    assert_rows_equal(off, pairs, ref, keys, "all rows")
    for kind, xs in named.items():
        o, p = m.getrow_sorted_batch(np.array(xs, U32))
        assert_rows_equal(o, p, ref, xs, kind)
    for kind in ("empty",):
        o, _ = m.getrow_sorted_batch(np.array(named[kind], U32))
        assert (o == 0).all(), kind
    small = keys[lens <= block_max]
    b0 = m.stat("sort_big")
    assert_rows_equal(*m.getrow_sorted_batch(small), ref, small, "small rows")
    assert m.stat("sort_big") == b0
    stats = {"n_big": n_big}
    if make_pieces:
        p = ms[1]
        b0 = p.stat("sort_big")
        o2, p2 = p.getrow_sorted_batch(keys)
        assert (o2 == off).all() and (p2 == pairs).all(), "many groups"
        stats["sort_big_pieces"] = p.stat("sort_big") - b0
    # paging edges and iter_rows
    assert (m.rows(TOP) == [TOP]).all() and (m.rows(TOP, 5) == [TOP]).all()
    assert (m.rows(0, 3) == keys[:3]).all() and (m.rows(2, 2) == keys[(keys >= 2)][:2]).all()
    assert m._lib.smatrix_list_rows(m._handle(), 2, None, 0) == int((keys >= 2).sum())
    seen = []
    for per in (1, 7, 1000):
        seen = []
        for k, o, p in m.iter_rows(0, per):
            assert len(k) <= per
            assert_rows_equal(o, p, ref, k, f"iter_rows({per})")
            seen.append(k)
        assert (np.concatenate(seen) == keys).all(), f"iter_rows({per})"
    assert (np.concatenate([k for k, _, _ in m.iter_rows(1 << 31, 2)]) == keys[keys >= 1 << 31]).all()
    # a repeated call allocates nothing; host outputs bring down the answer and a few control words
    m.rows(); m.getrow_sorted_batch(keys)
    a0, d0 = m.stat("allocs"), m.stat("d2h_bytes")
    got = m.rows()
    d1 = m.stat("d2h_bytes")
    assert 4 * len(keys) <= d1 - d0 < 4 * len(keys) + 4096
    off, pairs = m.getrow_sorted_batch(keys)
    d2 = m.stat("d2h_bytes")
    assert 8 * (len(keys) + 1) + 8 * len(pairs) <= d2 - d1 < 8 * (len(keys) + 1) + 8 * len(pairs) + 4096
    assert m.stat("allocs") == a0, "a repeated call allocated"
    for x in ms:
        x.close()
    ref.close()
    return stats


def scenario_follows_writes(make, tmp_path, big=2000):
    """New rows, a directory rehash and row growth show in the next listing; a snapshot reloads to the same rows."""
    path = os.path.join(str(tmp_path), "export.smx")
    m, ref = make(path), port()
    st = Stream([m], ref, seed=11)
    st.op("incr", [5, 6, 7], [1, 0, 2], [1, 1, 1])
    check_listing(m, ref, "first")
    g0, d0 = m.stat("row_grows"), m.stat("dir_grows")
    xs = st.rng.choice(np.arange(1, 1 << 32, 9973, dtype=np.uint64), 3000, replace=False)
    st.op("incr", xs, np.full(len(xs), 3), np.ones(len(xs)))               # many new rows: the directory grows
    st.row(6, big, extra=(TOP,))                                          # and a row grows
    assert m.stat("dir_grows") > d0 and m.stat("row_grows") > g0
    keys = check_listing(m, ref, "after writes")
    assert_rows_equal(*m.getrow_sorted_batch(keys), ref, keys, "after writes")
    m.close()
    m2 = make(path)
    got = m2.rows()
    assert (got == keys).all(), "after the reload"
    assert_rows_equal(*m2.getrow_sorted_batch(got), ref, got, "after the reload")
    m2.close()
    ref.close()


def foreign_csr(rng, lens):
    """a CSR of (column, value) pairs with unique random columns per segment (half of them >= 2^31)"""
    off = np.concatenate([[0], np.cumsum(lens)]).astype(np.uint64)
    cols = np.concatenate([rng.choice(1 << 32, L, replace=False) for L in lens] + [np.zeros(0, np.int64)])
    pairs = np.stack([cols, rng.integers(0, 1 << 32, len(cols))], axis=1).astype(U32)
    return off, pairs


def sorted_csr(off, pairs):
    out = pairs.copy()
    for i in range(len(off) - 1):
        seg = pairs[off[i]:off[i + 1]]
        out[off[i]:off[i + 1]] = seg[np.argsort(seg[:, 0], kind="stable")]
    return out


def scenario_sort_rows(m, warp_max, block_max, dev, down):
    """smatrix_b200_sort_rows on CSRs that no table made: every class, empty segments, columns >= 2^31."""
    rng = np.random.default_rng(3)
    lens = [0, 1, 2, 3, 0, warp_max - 1, warp_max, warp_max + 1, 0, block_max - 1, block_max, block_max + 1,
            3 * block_max + 5, 0, 2, block_max + 300, 17]
    off, pairs = foreign_csr(rng, lens)
    b0 = m.stat("sort_big")
    d_off, d_pairs = dev(m, off), dev(m, pairs)
    m._lib.smatrix_b200_sort_rows(m._handle(), len(lens), d_off, d_pairs)
    got = down(m, d_pairs, pairs)
    assert (got == sorted_csr(off, pairs)).all()
    assert m.stat("sort_big") - b0 == sum(L > block_max for L in lens)
    assert (got[:, 0] >= 1 << 31).any()
    m.dev_free(d_off); m.dev_free(d_pairs)
