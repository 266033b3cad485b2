"""Adversarial-key scenarios shared by the CPU tests (simulator builds) and the GPU tests, both in
tests/test_collisions.py.  The parity suite feeds the table well-mixed keys, which give short probe runs;
here the keys are chosen through the inverses of the kernels' own hash functions so that

  - many rows share the low bits of smx_mix_row: one directory home (the LAST entry of a directory of up to
    2^low_bits entries), one long probe chain that wraps to entry 0 and from the last directory slice to
    slice 0;
  - many columns of a row share the low bits of smx_mix_col, all ones: in a bucket of up to 2^tile_log
    sectors every column sits in one run that wraps at the bucket's end, and in a bigger bucket every run
    starts at the last sector of a re-placement tile (k_migrate_tiles), so it spills;
  - host-array batches are cut into many staged pieces (SMATRIX_STAGE=1024), so that every staging slot
    of the double-buffered upload and of the four-stream point read is reused.

Everything is compared, bit-exact, with parity_suite.checker() through parity_suite.compare.
"""
from __future__ import annotations

import numpy as np

from conftest import safe_stream
from parity_suite import U32, apply_both, checker, compare

ROW_MUL = (0x85EBCA6B, 0xC2B2AE35)   # smx_mix_row: x ^= x >> 16; x *= a; x ^= x >> 13; x *= b; x ^= x >> 16
ROW_SHIFT = (16, 13, 16)
COL_MUL = (0x7FEB352D, 0x846CA68B)   # smx_mix_col: the same shape with shifts 16, 15, 16
COL_SHIFT = (16, 15, 16)
DIR_CREATE_STEPS = 256               # dir_find creates a row at most this many probe steps - 1 from its home


# ------------------------------------------------------------------ the kernels' hash functions and their inverses
def _mix(v, mul, shift):
    x = np.array(v, dtype=U32)
    with np.errstate(over="ignore"):
        x ^= x >> U32(shift[0]); x *= U32(mul[0])
        x ^= x >> U32(shift[1]); x *= U32(mul[1])
        x ^= x >> U32(shift[2])
    return x


def _unshift(h, s):
    """inverse of x ^= x >> s: every pass fixes s more of the top bits"""
    x = h.copy()
    for _ in range(32 // s + 1):
        x = h ^ (x >> U32(s))
    return x


def _unmix(h, mul, shift):
    x = np.array(h, dtype=U32)
    with np.errstate(over="ignore"):
        x = _unshift(x, shift[2]) * U32(pow(mul[1], -1, 2**32))
        x = _unshift(x, shift[1]) * U32(pow(mul[0], -1, 2**32))
        return _unshift(x, shift[0])


def mix_row(x):
    return _mix(x, ROW_MUL, ROW_SHIFT)


def mix_col(y):
    return _mix(y, COL_MUL, COL_SHIFT)


def unmix_row(h):
    return _unmix(h, ROW_MUL, ROW_SHIFT)


def unmix_col(h):
    return _unmix(h, COL_MUL, COL_SHIFT)


def check_mixers():
    # known answers of the C functions (smx_kernels.cu); smx_mix_row is murmur3's fmix32
    assert list(mix_row([1, 0x12345678, 0xFFFFFFFF, 2654435761])) == [0x514E28B7, 0xE37CD1BC, 0x81F16F39, 0x11FD02EB]
    assert list(mix_col([1, 0x12345678, 0xFFFFFFFF, 2654435761])) == [0x688990C0, 0xF5E71C96, 0x6768824A, 0x6D523710]
    edges = np.array([0, 1, 2, 3, 0x7FFF, 0x8000, 0xFFFF, 0x10000, 0x7FFFFFFF, 0x80000000, 0x80000001,
                      0xFFFFFFFE, 0xFFFFFFFF, 0xAAAAAAAA, 0x55555555], U32)
    rng = np.random.default_rng(1)
    vals = np.concatenate([edges, rng.integers(0, 2**32, 100000, dtype=np.uint64).astype(U32)])
    for mix, unmix in ((mix_row, unmix_row), (mix_col, unmix_col)):
        assert (mix(unmix(vals)) == vals).all() and (unmix(mix(vals)) == vals).all()
    assert mix_row([0])[0] == 0 and mix_col([0])[0] == 0    # so an all-ones low part never yields column 0


def colliding(n: int, low_bits: int, unmix, first: int = 0, rng=None):
    """n distinct keys whose hash has all of its low `low_bits` bits set; the high bits are first, first + 1, ...
    or, with rng, drawn without replacement"""
    space = 1 << (32 - low_bits)
    hi = (rng.choice(space, size=n, replace=False) if rng is not None
          else np.arange(first, first + n)).astype(np.uint64)
    assert n <= space and (rng is not None or first + n <= space)
    return unmix(((hi << np.uint64(low_bits)) | np.uint64((1 << low_bits) - 1)).astype(U32))


def chain_rows(n: int, low_bits: int, first: int = 0):
    return colliding(n, low_bits, unmix_row, first)


def _interleave(rng, xs, ys, vs):
    """Shuffle a batch given row by row (each row's ops in its own order) while keeping every row's own order."""
    grp = np.cumsum(np.r_[0, xs[1:] != xs[:-1]])
    t = rng.random(len(xs))
    t = t[np.lexsort((t, grp))]          # ascending inside each row's run
    order = np.argsort(t, kind="stable")
    return xs[order], ys[order], vs[order]


def _dev(m, a):
    from libsmatrix_b200.matrix import DevPtr
    a = np.ascontiguousarray(a, U32)
    p = m.dev_alloc(max(a.nbytes, 8))
    if a.nbytes:
        m.memcpy(p, a.ctypes.data, a.nbytes)
    return DevPtr(p, len(a))


def _device_get(m, qx, qy):
    dx, dy, do = _dev(m, qx), _dev(m, qy), _dev(m, np.zeros(len(qx), U32))
    m.get_batch(dx, dy, do)
    got = np.empty(len(qx), U32)
    m.memcpy(got.ctypes.data, do.ptr, got.nbytes)
    for d in (dx, dy, do):
        m.dev_free(d.ptr)
    return got


STATS = ("dir_grows", "dir_cap", "rows", "spilled", "recycled", "sliced_gets", "row_grows")


def _stats(m):
    return {k: m.stat(k) for k in STATS}


# ------------------------------------------------------------------ row chains
def _chain_batch(rng, rows, cols_per_row: int, col0_every: int):
    """cols_per_row new columns per row; for every col0_every-th row an incr on column 0 goes between its columns
    (column 0 turns non-zero mid-batch: k_sync_rowlen and k_finalize_t0 find these rows with dir_find)"""
    xs, ys, vs = [], [], []
    for k, r in enumerate(rows):
        cols = list(rng.integers(1, 2**32, cols_per_row, dtype=np.uint64).astype(U32))
        cols += cols[:2]                                      # the same columns again: existing cells
        if k % col0_every == 0:
            cols.insert(int(rng.integers(0, len(cols) + 1)), U32(0))
        xs += [r] * len(cols); ys += cols
    xs, ys = np.array(xs, U32), np.array(ys, U32)
    vs = np.where(ys == 0, rng.integers(1, 6, len(ys)), rng.integers(0, 2**32, len(ys), dtype=np.uint64)).astype(U32)
    return _interleave(rng, xs, ys, vs)


def scenario_row_chains(make, n_rows: int = 700, low_bits: int = 22, singles: int = 6, seed: int = 41):
    """n_rows rows with one directory home: written in batches of several hundred rows, then as a set batch with
    duplicate keys, then in batches of ONE new row each; read back with gets, rowlen and getrow — plus reads of
    never-written rows with the same home (each such miss walks the whole chain), in input order and, on device
    arrays, in directory-slice order.  Returns the table's counters."""
    rng = np.random.default_rng(seed)
    ids = chain_rows(n_rows + singles + 100, low_bits)
    chain, late, absent = ids[:n_rows], ids[n_rows:n_rows + singles], ids[n_rows + singles:]
    mixed = np.arange(1, 201, dtype=U32) * U32(2654435761)    # ordinary rows in the same batches
    m, ref = make(), checker()
    for part in np.array_split(chain, [n_rows * 2 // 5]):
        xs, ys, vs = _chain_batch(rng, np.concatenate([part, mixed[:100]]), 5, 2)
        apply_both(m, ref, "incr", xs, ys, vs)
    # set, several writes per key (last writer wins), column 0 of the rows that did not have it yet included
    n = 8 * n_rows
    xs = rng.choice(np.concatenate([chain, mixed]), n)
    ys = np.where(rng.random(n) < 0.15, 0, rng.integers(1, 12, n)).astype(U32)
    vs = rng.integers(1, 2**32, n, dtype=np.uint64).astype(U32)
    apply_both(m, ref, "set", xs, ys, vs)
    for r in late:                                            # one new row on the chain per batch
        xs, ys, vs = _chain_batch(rng, np.concatenate([[r], rng.choice(chain, 20)]).astype(U32), 3, 3)
        apply_both(m, ref, "incr", xs, ys, vs)
    rows = np.concatenate([chain, late, absent, mixed])
    hit = rng.integers(0, len(xs), 2000)
    qx = np.concatenate([rng.choice(chain, 4000), absent, rng.choice(absent, 1000), xs[hit]]).astype(U32)
    qy = np.concatenate([rng.integers(0, 12, 5000 + len(absent)), ys[hit]]).astype(U32)
    compare(m, ref, rows, qx, qy)
    want = ref.get_many(qx, qy)
    for mode in (0, 2):                                       # input order / always by directory slice
        m.set_get_slices(mode)
        got = _device_get(m, qx, qy)
        assert (got == want).all(), f"device get, mode {mode}: {int((got != want).sum())} mismatches"
    m.set_get_slices(1)
    stats = _stats(m)
    m.close(); ref.close()
    return stats


def scenario_chain_resizes(make, n_rows: int = 300, low_bits: int = 22, singles: int = 3):
    """Once a chain is longer than dir_find's create limit, the directory has been grown until the chain's rows
    fit.  A later batch that adds ONE row to that chain must not resize the directory more than once: a shrink
    after the chunk that brought the chain back beyond the limit would make every such batch grow the directory
    all the way up again and shrink it back (gigabytes of memset per call on the full-size table)."""
    assert n_rows > DIR_CREATE_STEPS
    ids = chain_rows(n_rows + singles + 50, low_bits)
    m, ref = make(), checker()
    ones = np.ones(n_rows, U32)
    apply_both(m, ref, "incr", ids[:n_rows], ones, ones)
    for k, r in enumerate(ids[n_rows:n_rows + singles]):
        before = m.stat("dir_grows")
        apply_both(m, ref, "incr", np.array([r, ids[k]], U32), np.array([2, 2], U32), np.array([5, 7], U32))
        resized = m.stat("dir_grows") - before
        assert resized <= 1, f"one new row on a chain of {n_rows + k} rows resized the directory {resized} times"
    rows = ids
    compare(m, ref, rows, np.repeat(rows, 3), np.tile(np.array([0, 1, 2], U32), len(rows)))
    m.close(); ref.close()


# ------------------------------------------------------------------ column runs
def scenario_column_runs(make, n_cols=(20000, 30000, 40000), tile_log: int = 10, rounds: int = 4, seed: int = 43):
    """Rows whose columns all have their bucket home at sector 2^tile_log - 1 modulo 2^tile_log (tile_log = the
    re-placement tile, MIG_TILE_LOG): runs that wrap at the bucket end while the bucket is at most one tile, runs
    that start at a tile's last sector (and spill) once it is bigger.  The rows grow in the same rounds (several
    big rows per k_migrate_tiles launch, one spill list), next to ordinary rows.  incr / decr / set, then
    incr_batch_out (k_find_addr walks the runs), gets with misses on colliding columns, getrow.  Returns the
    table's counters."""
    rng = np.random.default_rng(seed)
    big = np.array([7, 8, 9], U32) * U32(2654435761)
    held = 2000                                               # colliding columns never written: misses
    allc = colliding(sum(n_cols) + held * len(big), tile_log, unmix_col, rng=rng)
    cols, at = [], 0
    for n in n_cols:
        cols.append(allc[at:at + n + held]); at += n + held
    m, ref = make(), checker()
    for r in range(rounds):
        op = ("incr", "decr", "set", "incr", "incr")[r % 5]
        xs, ys = [], []
        for row, c, n in zip(big, cols, n_cols):
            new = c[n * r // rounds:n * (r + 1) // rounds]
            old = rng.choice(c[:max(1, n * r // rounds)], len(new) // 4)   # cells written in earlier rounds
            xs.append(np.full(len(new) + len(old), row, U32)); ys += [new, old]
        xs.append(rng.integers(100, 400, 6000).astype(U32))
        ys.append(rng.integers(1, 60, 6000).astype(U32))
        xs, ys = np.concatenate(xs), np.concatenate(ys)
        vs = rng.integers(1, 2**32, len(xs), dtype=np.uint64).astype(U32)
        perm = rng.permutation(len(xs))
        apply_both(m, ref, op, xs[perm], ys[perm], vs[perm])
    # per-op return values: every op's cell is found again by walking its run
    pick = rng.integers(0, len(big), 30000)
    xs = big[pick]
    ys = np.array([cols[p][int(rng.integers(0, n_cols[p] + 200))] for p in pick], U32)   # a few new columns too
    vs = rng.integers(1, 2**32, len(xs), dtype=np.uint64).astype(U32)
    got = np.asarray(m.incr_batch_out(xs, ys, vs))
    want = ref.apply("incr", xs, ys, vs, want_out=True)
    assert (got == want).all(), f"incr_batch_out: {int((got != want).sum())} return values differ"
    qx = np.concatenate([np.full(3000 + held, row, U32) for row in big] + [rng.integers(100, 400, 2000).astype(U32)])
    qy = np.concatenate([np.concatenate([rng.choice(c[:n], 3000), c[n:]]) for c, n in zip(cols, n_cols)]
                        + [rng.integers(1, 80, 2000).astype(U32)])
    compare(m, ref, np.concatenate([big, np.arange(100, 402, dtype=U32)]), qx, qy)
    stats = _stats(m)
    m.close(); ref.close()
    return stats


# ------------------------------------------------------------------ staged host batches
def scenario_staged_host_batches(make, pieces: int = 13, seed: int = 47):
    """Host-array batches of pieces * 1024 + 1 ops on a table opened with SMATRIX_STAGE=1024: writes go up in 1024-op
    pieces through two staging buffers, point reads in 1024-query pieces over four streams.  Set with the last
    writer in a later piece, column 0 turning non-zero in a later piece than the row's first columns, incr / set
    batches with per-op return values — against the checker, and against a second table that got the same ops
    as device arrays (no staging)."""
    rng = np.random.default_rng(seed)
    n = pieces * 1024 + 1
    m, md, ref = make(), make(), checker()

    def both(op, xs, ys, vs):
        apply_both(m, ref, op, xs, ys, vs)
        dx, dy, dv = _dev(md, xs), _dev(md, ys), _dev(md, vs)
        getattr(md, op + "_batch")(dx, dy, dv)
        for d in (dx, dy, dv):
            md.dev_free(d.ptr)

    # set: ~10 writes per key spread over all pieces, column 0 included (non-zero values)
    rows = np.arange(30, dtype=U32) * U32(2654435761)
    xs, ys = rows[rng.integers(0, 30, n)], rng.integers(0, 40, n).astype(U32)
    both("set", xs, ys, rng.integers(1, 2**32, n, dtype=np.uint64).astype(U32))
    # incr: 100 rows get 12 columns in the first two pieces, column 0 in piece 6, 12 more columns in the last pieces
    late = np.arange(1000, 1100, dtype=U32)
    early = np.repeat(late, 12), rng.integers(1, 500, 1200).astype(U32)
    after = np.repeat(late, 12), rng.integers(500, 1000, 1200).astype(U32)
    fill = rng.integers(2000, 2300, n).astype(U32), rng.integers(1, 50, n).astype(U32)
    head, mid = 6 * 1024 - 1200, n - 6 * 1024 - 100 - 1200
    xs = np.concatenate([early[0], fill[0][:head], late, fill[0][head:head + mid], after[0]])
    ys = np.concatenate([early[1], fill[1][:head], np.zeros(100, U32), fill[1][head:head + mid], after[1]])
    assert len(xs) == n
    both("incr", xs, ys, np.where(ys == 0, 3, 1).astype(U32))
    rowlist = np.concatenate([rows, late, np.arange(2000, 2301, dtype=U32)])
    # per-op return values over many pieces
    for op in ("incr", "set"):
        xs, ys, vs = safe_stream(rng, n, 400, 60, op, col0_rate=0.05)
        xs = xs + U32(5000)
        got = np.asarray(getattr(m, op + "_batch_out")(xs, ys, vs))
        want = ref.apply(op, xs, ys, vs, want_out=True)
        assert (got == want).all(), f"{op}_batch_out: {int((got != want).sum())} return values differ"
        dx, dy, dv = _dev(md, xs), _dev(md, ys), _dev(md, vs)
        getattr(md, op + "_batch")(dx, dy, dv)
        for d in (dx, dy, dv):
            md.dev_free(d.ptr)
    rowlist = np.concatenate([rowlist, np.arange(5000, 5401, dtype=U32)])
    # reads: n queries = pieces + 1 staged pieces, the last one ragged
    qx = rng.choice(rowlist, n).astype(U32)
    qy = rng.integers(0, 1000, n).astype(U32)
    compare(m, ref, rowlist, qx, qy)
    compare(md, ref, rowlist, qx, qy)
    assert (_device_get(md, qx, qy) == np.asarray(m.get_batch(qx, qy))).all()
    m.close(); md.close(); ref.close()
