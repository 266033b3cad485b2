"""Incremental checkpoints of the file mode (smatrix_b200_checkpoint / smatrix_b200_shard_checkpoint): only the
row blocks of the rows written since the file last matched the table are appended, then a new directory, then the
header's pointer is switched.  Shared by the simulator tests (tests/test_checkpoint.py) and the B200 tests.

Every check compares a checkpointed file with a FULL snapshot of the same table, taken by a twin handle that
applied the same ops: both must load to the same gets, rowlens, column-sorted getrows and totals, in our loader,
in the C checker's positional load and, where it is built, in the reference."""
from __future__ import annotations

import os
import shutil

import numpy as np

from oracle import cpu
from conftest import safe_stream
import smx_file
import snapshot_suite as ss

U32 = np.uint32
BLOCK = 16 + 4194304 * 12          # one directory block of 2^22 entries


def head_ptr(path: str) -> int:
    with open(path, "rb") as f:
        f.seek(8)
        return int.from_bytes(f.read(8), "little")


def set_head_ptr(path: str, at: int) -> None:
    with open(path, "r+b") as f:
        f.seek(8)
        f.write(int(at).to_bytes(8, "little"))


def same_file(a: str, b: str, exact: bool) -> None:
    """Two full snapshots of the same table: byte for byte where the listing order is deterministic (the
    simulator); on a GPU the rows are listed and cells placed in whatever order the threads got there, so the
    same header, size and rows, each at the same size with the same cells."""
    if exact:
        assert open(a, "rb").read() == open(b, "rb").read()
        return
    assert head_ptr(a) == head_ptr(b) == 512 and os.path.getsize(a) == os.path.getsize(b)
    fa, fb = smx_file.read(a), smx_file.read(b)
    assert fa.keys() == fb.keys()
    for row, (size, cells) in fa.items():
        assert size == fb[row][0] and smx_file.live(cells) == smx_file.live(fb[row][1]), f"row {row}"


def copy(src: str, dst: str) -> str:
    shutil.copy(src, dst)
    return dst


def view(m, rows, qx, qy):
    """What a table answers: gets, rowlens, column-sorted getrows and the totals."""
    o, p = m.getrow_batch(rows)
    return (np.asarray(m.get_batch(qx, qy)).copy(), np.asarray(m.rowlen_batch(rows)).copy(), o.copy(),
            cpu.sort_rows(o, p), [m.stat(k) for k in ("rows", "nnz", "value_sum")])


def checker_view(kind, path, rows, qx, qy):
    """The same through the C checker ("port") or the reference: no stats, the rest identical."""
    c = cpu.CpuMatrix(kind, path)
    try:
        o, p = c.getrow_many(rows)
        return (c.get_many(qx, qy), c.rowlen_many(rows), o, cpu.sort_rows(o, p))
    finally:
        c.close()


def same(a, b, what):
    for k, (x, y) in enumerate(zip(a, b)):
        assert np.array_equal(np.asarray(x), np.asarray(y)), f"{what}: part {k} differs"


def loaded(make, path, tmp, rows, qx, qy, tag):
    """Our loader's view of a file (on a copy: closing a file-backed handle writes it)."""
    m = make(copy(path, os.path.join(tmp, f"load_{tag}.smx")))
    try:
        return view(m, rows, qx, qy)
    finally:
        m.close()


def check_readers(make, path, want_path, tmp, rows, qx, qy, tag):
    """path (checkpointed) loads like want_path (a full snapshot of the same table) in every reader, and every row
    of it passes the independent reader's structure and reachability checks."""
    same(loaded(make, path, tmp, rows, qx, qy, tag + "_ck"), loaded(make, want_path, tmp, rows, qx, qy, tag + "_full"),
         f"{tag}: our loader")
    kinds = ["port"] + (["reference"] if cpu.have_reference() else [])
    for kind in kinds:
        same(checker_view(kind, copy(path, os.path.join(tmp, f"{kind}_{tag}_ck.smx")), rows, qx, qy),
             checker_view(kind, copy(want_path, os.path.join(tmp, f"{kind}_{tag}_full.smx")), rows, qx, qy),
             f"{tag}: {kind}")
    for row, (size, cells) in smx_file.read(path).items():
        smx_file.check_row(row, size, cells)


def updates(seed, rows_touched, new_rows=()):
    """An op batch list touching exactly `rows_touched` (existing rows) and `new_rows`: incr with column-0
    traffic, a `set 0` cell, a zero-valued incr that wraps, and columns of the 3000-column row 5000 if listed."""
    rng = np.random.default_rng(seed)
    keys = np.asarray(sorted(set(int(r) for r in rows_touched) | set(int(r) for r in new_rows)), U32)
    ops = []
    xs = np.repeat(keys, 6)
    ys = rng.integers(1, 200, len(xs)).astype(U32)
    ys[::5] = 0                                                   # column 0 of these rows
    vs = rng.integers(1, 500, len(xs)).astype(U32)
    ops.append(("incr", xs, ys, vs))
    ops.append(("set", keys[:1], np.array([7], U32), np.array([0], U32)))           # set 0: a zero-valued cell
    ops.append(("incr", keys[-1:], np.array([9], U32), np.array([0], U32)))         # an incr by 0
    if 5000 in keys:
        ly = np.arange(1, 3001, dtype=U32) * U32(2654435761)
        ops.append(("incr", np.full(3000, 5000, U32), ly, np.ones(3000, U32)))
    return ops, keys


def apply(m, ops, how="batch"):
    for op, x, y, v in ops:
        if how == "out":
            getattr(m, op + "_batch_out")(x, y, v)
        else:
            getattr(m, op + "_batch")(x, y, v)


def queries(rows, extra_rows=()):
    r = np.unique(np.concatenate([np.asarray(rows, U32), np.asarray(extra_rows, U32)]))
    qx = np.repeat(r, 8)
    qy = np.tile(np.array([0, 1, 7, 9, 50, 150, 199, 2654435761], U32), len(r))
    return r, qx, qy


# ------------------------------------------------------------------ one handle
def scenario_equivalence(make, tmp_path, exact=True):
    """Build and persist, touch a known subset, checkpoint: the file loads like a full snapshot in every reader;
    only the dirty rows were appended, nothing before the old end but the header pointer changed; the crash
    states (old pointer, appended region cut anywhere) load to the previous state; a no-op leaves it alone."""
    tmp = str(tmp_path)
    f, g = os.path.join(tmp, "ck.smx"), os.path.join(tmp, "full.smx")
    m, t = make(f), make(g)                                      # t: the twin that takes full snapshots
    rows, qx, qy = ss._build(lambda op, x, y, v: (getattr(m, op + "_batch")(x, y, v),
                                                  getattr(t, op + "_batch")(x, y, v)), np.random.default_rng(41))
    assert m.stat("dirty_rows") == m.stat("rows")                # written since open, no file yet
    assert m.snapshot() == 0 and t.snapshot() == 0
    assert m.stat("dirty_rows") == 0
    same_file(f, g, exact)
    old = open(f, "rb").read()
    touched = [0, 3, 17, 40, 151, 4000, 5000]
    ops, keys = updates(5, touched, new_rows=[90001, 90002])
    apply(m, ops); apply(t, ops)
    assert m.stat("dirty_rows") == len(keys)
    rows, qx, qy = queries(rows, keys)
    before = loaded(make, f, tmp, rows, qx, qy, "before")
    assert m.checkpoint() == 0
    assert m.stat("dirty_rows") == 0
    assert t.snapshot() == 0
    new = open(f, "rb").read()
    E = (len(old) + 7) & ~7
    D = head_ptr(f)
    parsed = smx_file.read(f)
    dirty_bytes = sum(16 + 8 * parsed[int(k)][0] for k in keys)
    assert D == E + dirty_bytes, "the dirty rows' blocks, then the directory"
    assert len(new) == D + BLOCK, "file = old end (aligned) + dirty blocks + one directory block"
    assert new[:8] == old[:8] and new[16:len(old)] == old[16:], "nothing before the old end but the pointer"
    for k in keys:                                               # the dirty rows' blocks are the new ones
        assert _entry_offset(new, D, int(k)) >= E
    clean = [int(r) for r in parsed if r not in set(int(k) for k in keys)]
    for r in clean[:50]:                                         # the clean rows keep their old blocks
        assert _entry_offset(new, D, r) < len(old)
    check_readers(make, f, g, tmp, rows, qx, qy, "gen1")
    # the intermediate states of the write: header not switched yet, appended region cut anywhere
    crash = copy(f, os.path.join(tmp, "crash.smx"))
    set_head_ptr(crash, 512)
    same(loaded(make, crash, tmp, rows, qx, qy, "crash"), before, "old pointer")
    for cut in (len(old), E, E + 1, (E + D) // 2, D, D + 16, D + BLOCK // 2):
        c = copy(crash, os.path.join(tmp, f"cut{cut}.smx"))
        os.truncate(c, cut)
        same(loaded(make, c, tmp, rows, qx, qy, f"cut{cut}"), before, f"old pointer, cut at {cut}")
    # nothing written since: nothing changes, the file is not even opened for writing
    st = os.stat(f)
    assert m.checkpoint() == 0
    assert open(f, "rb").read() == new and os.stat(f).st_mtime_ns == st.st_mtime_ns
    m.close(); t.close()
    same_file(f, g, exact)                                        # close still writes the full snapshot


def _entry_offset(data: bytes, dir_at: int, row: int) -> int:
    ents = np.frombuffer(data, smx_file.ENTRY, 4194304, dir_at + 16)
    k = np.flatnonzero((ents["row"] == row) & (ents["off"] != 0))
    assert len(k) == 1, f"row {row} listed {len(k)} times"
    return int(ents["off"][k[0]])


def scenario_generations(make, tmp_path, n_gen=4, exact=True):
    """Checkpoints in a row, each compared with its moment; whether one appends or falls back to a snapshot (the
    file would pass twice a full snapshot) is decided from sizes alone, and every fall-back puts the header back
    at 512.  The file never exceeds twice the full snapshot's size."""
    tmp = str(tmp_path)
    f, g = os.path.join(tmp, "gen.smx"), os.path.join(tmp, "gen_full.smx")
    m, t = make(f), make(g)
    rows, qx, qy = ss._build(lambda op, x, y, v: (getattr(m, op + "_batch")(x, y, v),
                                                  getattr(t, op + "_batch")(x, y, v)), np.random.default_rng(41))
    assert m.checkpoint() == 0, "no base yet: a full snapshot"
    assert t.snapshot() == 0
    same_file(f, g, exact)                                        # the first checkpoint on a new path: the snapshot
    seen = set()
    for gen in range(n_gen):
        touched = np.arange(gen * 30, gen * 30 + 60) % 152
        if gen == n_gen - 1:
            touched = np.arange(152)                              # every row
        ops, keys = updates(100 + gen, touched, new_rows=[91000 + gen])
        apply(m, ops); apply(t, ops)
        rows, qx, qy = queries(rows, keys)
        size0 = os.path.getsize(f)
        assert m.checkpoint() == 0 and t.snapshot() == 0
        full = os.path.getsize(g)
        assert os.path.getsize(f) <= 2 * full
        appended = head_ptr(f) != 512
        seen.add(appended)
        if appended:
            assert os.path.getsize(f) > size0
        check_readers(make, f, g, tmp, rows, qx, qy, f"gen{gen}")
    assert seen == {True, False}, "both an appending checkpoint and a fall-back"
    m.close(); t.close()


def scenario_dirty_counts(make, tmp_path):
    """stat("dirty_rows") = the distinct rows each write API touched since the last save."""
    tmp = str(tmp_path)
    f = os.path.join(tmp, "cnt.smx")
    m = make(f)
    rows, qx, qy = ss._build(lambda op, x, y, v: getattr(m, op + "_batch")(x, y, v), np.random.default_rng(41))
    assert m.snapshot() == 0
    rng = np.random.default_rng(3)
    for api in ("incr", "decr", "set", "incr_out", "decr_out", "set_out", "single"):
        keys = np.unique(rng.integers(0, 160, 25).astype(U32))
        ys = rng.integers(0, 60, len(keys)).astype(U32)
        vs = np.ones(len(keys), U32)
        if api == "single":
            for x, y in zip(keys.tolist(), ys.tolist()):
                m.incr(x, y, 1)
        elif api.endswith("_out"):
            getattr(m, api[:-4] + "_batch_out")(keys, ys, vs)
        else:
            getattr(m, api + "_batch")(keys, ys, vs)
        assert m.stat("dirty_rows") == len(keys), api
        assert m.checkpoint() == 0
        assert m.stat("dirty_rows") == 0
    # a read marks nothing
    m.get_batch(qx, qy); m.rowlen_batch(rows); m.getrow_batch(rows)
    assert m.stat("dirty_rows") == 0
    m.close()


def scenario_fallbacks(make, tmp_path):
    """A file replaced behind the handle by one with another row set is rewritten whole; a checkpoint that
    cannot write (the path is a directory) returns -1 and keeps the rows dirty, and the next one writes them."""
    tmp = str(tmp_path)
    f, g, other = (os.path.join(tmp, n) for n in ("fb.smx", "fb_full.smx", "other.smx"))
    m, t = make(f), make(g)
    rows, qx, qy = ss._build(lambda op, x, y, v: (getattr(m, op + "_batch")(x, y, v),
                                                  getattr(t, op + "_batch")(x, y, v)), np.random.default_rng(41))
    assert m.snapshot() == 0
    o = make(other)                                               # same rows but one: another row set
    ss._build(lambda op, x, y, v: getattr(o, op + "_batch")(x, y, v), np.random.default_rng(41))
    o.incr(123456, 1, 1)
    o.close()
    shutil.copy(other, f)
    ops, keys = updates(7, [1, 2, 3])
    apply(m, ops); apply(t, ops)
    rows, qx, qy = queries(rows, keys)
    assert m.checkpoint() == 0 and t.snapshot() == 0
    assert head_ptr(f) == 512, "rewritten whole"
    check_readers(make, f, g, tmp, rows, qx, qy, "replaced")
    # failure: the path is a directory now
    ops, keys = updates(8, [10, 11, 12, 13])
    apply(m, ops); apply(t, ops)
    rows, qx, qy = queries(rows, keys)
    os.rename(f, f + ".away")
    os.mkdir(f)
    assert m.checkpoint() == -1
    assert m.stat("dirty_rows") == len(keys)
    os.rmdir(f)
    os.rename(f + ".away", f)
    assert m.checkpoint() == 0 and t.snapshot() == 0
    assert m.stat("dirty_rows") == 0
    assert head_ptr(f) != 512, "appended"
    check_readers(make, f, g, tmp, rows, qx, qy, "after_failure")
    m.close(); t.close()
    # a file that is gone: the next checkpoint writes it whole
    m = make(f)
    os.unlink(f)
    m.incr(1, 1, 1)
    assert m.checkpoint() == 0 and head_ptr(f) == 512
    m.close()


def scenario_foreign(make, tmp_path):
    """Files written by the C checker in an append-only writer's layouts: ours opens one, updates, checkpoints,
    and our loader and the checker read the result alike (and the reference, where it is built: it then reopens
    the checkpointed file, applies more ops and closes, and ours reads what it wrote)."""
    tmp = str(tmp_path)
    xs, ys, vs = safe_stream(np.random.default_rng(11), 8000, 140, 80, "incr", col0_rate=0.05)
    ck = cpu.CpuMatrix("port")
    ck.apply("incr", xs, ys, vs)
    rows = np.unique(xs)
    layouts = {"plain": {}, "shuffled": dict(shuffled=True), "dead": dict(dead=True),
               "unaligned": dict(unaligned=True), "small_dir": dict(small_dir=True),
               "all": dict(shuffled=True, dead=True, unaligned=True, small_dir=True)}
    files = {}
    for name, kw in layouts.items():
        files[name] = os.path.join(tmp, f"foreign_{name}.smx")
        ck.save(files[name], **kw)
    if cpu.have_reference():
        r = cpu.CpuMatrix("reference", os.path.join(tmp, "foreign_ref.smx"))
        r.apply("incr", xs, ys, vs)
        r.close()
        files["reference"] = os.path.join(tmp, "foreign_ref.smx")
    ck.close()
    ops, keys = updates(9, rows[::9], new_rows=[95000])
    allrows, qx, qy = queries(rows, keys)
    for name, path in files.items():
        work = copy(path, os.path.join(tmp, f"work_{name}.smx"))
        twin = copy(path, os.path.join(tmp, f"twin_{name}.smx"))
        m, t = make(work), make(twin)
        apply(m, ops); apply(t, ops)
        assert m.stat("dirty_rows") == len(keys)
        assert m.checkpoint() == 0 and t.snapshot() == 0
        assert head_ptr(work) != 512, f"{name}: appended to the foreign file"
        ck_file = copy(work, os.path.join(tmp, f"ck_{name}.smx"))
        m.close(); t.close()                                      # (close rewrites `work` whole)
        check_readers(make, ck_file, twin, tmp, allrows, qx, qy, f"foreign_{name}")
        if cpu.have_reference():
            more = safe_stream(np.random.default_rng(12), 3000, 150, 90, "incr", col0_rate=0.05)
            r = cpu.CpuMatrix("reference", copy(ck_file, os.path.join(tmp, f"ref_{name}.smx")))
            r.apply("incr", *more)
            want = (r.get_many(qx, qy), r.rowlen_many(allrows))
            r.close()
            m = make(copy(os.path.join(tmp, f"ref_{name}.smx"), os.path.join(tmp, f"ours_of_ref_{name}.smx")))
            got = (np.asarray(m.get_batch(qx, qy)), np.asarray(m.rowlen_batch(allrows)))
            m.close()
            same(got, want, f"{name}: the reference's file after our checkpoint")


# ------------------------------------------------------------------ sharded
def scenario_sharded(make, open_sharded, tmp_path, world, other):
    """A checkpoint at world W: the rows each rank routed count as dirty on their owners, the file loads answer for
    answer like the single-GPU checkpoint of the same stream and like a full snapshot, at another world too, and
    in the checker.  Writes go through ordered, unordered and *_batch_out routes."""
    tmp = str(tmp_path)
    state = os.path.join(tmp, "base.smx")
    m = make(state)
    rows, qx, qy = ss._build(lambda op, x, y, v: getattr(m, op + "_batch")(x, y, v), np.random.default_rng(41))
    m.close()
    gens = [updates(20, np.arange(0, 150, 7), new_rows=[96000, 96001]),
            updates(21, np.arange(3, 152, 11), new_rows=[97000]),
            updates(22, [5000, 4000, 1])]
    for k, (ops, keys) in enumerate(gens):
        rows, qx, qy = queries(rows, keys)
        single, single_ck, full, shard, shard_ck = (os.path.join(tmp, f"{n}{k}.smx") for n in
                                                    ("single", "single_ck", "full", "shard", "shard_ck"))
        m = make(copy(state, single))
        apply(m, ops)
        assert m.checkpoint() == 0 and head_ptr(single) != 512
        copy(single, single_ck)                                  # (close rewrites it whole)
        m.close()
        t = make(copy(state, full))
        apply(t, ops)
        t.close()                                                 # the full snapshot of the same table

        def fn(s, r, ops=ops, k=k):
            sl = lambda a: a[r * len(a) // world:(r + 1) * len(a) // world]
            for op, x, y, v in ops:
                if k == 2:
                    getattr(s, op + "_batch_out")(sl(x), sl(y), sl(v))
                elif op == "set":
                    s.set_batch(sl(x), sl(y), sl(v))
                else:
                    getattr(s, op + "_batch")(sl(x), sl(y), sl(v), ordered=(k == 0))
            dirty = s.sum(s.stat("dirty_rows"))
            rc = s.checkpoint()
            after = s.sum(s.stat("dirty_rows"))
            s.barrier()
            if r == 0:
                copy(shard, shard_ck)
            s.barrier()
            return rc, dirty, after
        out = open_sharded(world, copy(state, shard), fn)
        for r in range(world):
            assert out[r] == (0, len(keys), 0), f"gen {k}, rank {r}: {out[r]}"
        assert head_ptr(shard_ck) != 512, "appended"
        check_readers(make, shard_ck, full, tmp, rows, qx, qy, f"sharded{k}")
        check_readers(make, single_ck, full, tmp, rows, qx, qy, f"single{k}")
        got = open_sharded(other, copy(shard_ck, shard_ck + ".o"), lambda s, r: _sharded_view(s, rows, qx, qy))
        want = loaded(make, full, tmp, rows, qx, qy, f"sh_full{k}")
        for r in range(other):
            same(got[r], want, f"gen {k}: world {world} checkpoint reloaded at world {other}, rank {r}")
        state = full


def scenario_sharded_fallbacks(make, open_sharded, tmp_path, world):
    """Collective fall-backs and failure: no base (a new path) -> the full snapshot on every rank; a second
    checkpoint that would pass twice a full snapshot -> the snapshot; a directory at the path -> -1 on every rank
    with the rows still dirty, and the next checkpoint writes them."""
    tmp = str(tmp_path)
    f = os.path.join(tmp, "shfb.smx")
    xs, ys, vs = safe_stream(np.random.default_rng(5), 6000, 150, 90, "incr", col0_rate=0.05)

    def fn(s, r):
        sl = lambda a: a[r * len(a) // world:(r + 1) * len(a) // world]
        s.incr_batch(sl(xs), sl(ys), sl(vs))
        res = [s.checkpoint(), head_ptr(f)]                       # no base: the snapshot
        s.incr_batch(sl(xs[:100]), sl(ys[:100]), sl(vs[:100]))
        res += [s.checkpoint(), head_ptr(f)]                      # appended
        s.incr_batch(sl(xs[:300]), sl(ys[:300]), sl(vs[:300]))
        res += [s.checkpoint(), head_ptr(f)]                      # past twice a snapshot: rewritten
        s.incr_batch(sl(xs[:50]), sl(ys[:50]), sl(vs[:50]))
        dirty = s.sum(s.stat("dirty_rows"))
        s.barrier()
        if r == 0:
            os.rename(f, f + ".away"); os.mkdir(f)
        s.barrier()
        res += [s.checkpoint(), s.sum(s.stat("dirty_rows")) == dirty and dirty > 0]
        s.barrier()
        if r == 0:
            os.rmdir(f); os.rename(f + ".away", f)
        s.barrier()
        res += [s.checkpoint(), s.sum(s.stat("dirty_rows"))]
        return res
    out = open_sharded(world, f, fn)
    for r in range(world):
        rc1, p1, rc2, p2, rc3, p3, rc4, kept_dirty, rc5, left = out[r]
        assert (rc1, p1, rc2, rc3, p3, rc4, kept_dirty, rc5, left) == (0, 512, 0, 0, 512, -1, True, 0, 0), out[r]
        assert p2 != 512
    m = make(copy(f, f + ".single"))                              # the close wrote it whole: it loads
    assert m.stat("rows") == len(np.unique(xs))
    m.close()


def _sharded_view(s, rows, qx, qy):
    o, p = s.getrow_batch(rows)
    return (np.asarray(s.get_batch(qx, qy)).copy(), np.asarray(s.rowlen_batch(rows)).copy(), o.copy(),
            cpu.sort_rows(o, p), [s.sum(s.stat(k)) % 2**64 for k in ("rows", "nnz", "value_sum")])
