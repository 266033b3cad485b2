""".smx snapshots and loads against the CPU checker's file mode (oracle/smatrix_oracle.c) and an independent
reader (tests/smx_file.py).  Shared by the simulator tests and the B200 tests (tests/test_snapshot_oracle.py).

The promise under test (DESIGN.md 8): a file written by the library is what the reference writes — every row
block at the reference's row size S, holding the row's cells where the reference's `column % size` probe finds
them, before and after its loader clears the zero-valued slots — and a reload restores the reference's state:
S = the file's row size, `used` recounted.  Everything here is compared with the checker, never with ourselves.

Histories stay inside the reference's safe domain (SURVEY.md Q3).  Column 0 returns to 0 only in rows whose
columns are 1 .. k, so its slot (slot 0) is never inside another cell's probe run, and such a row does not grow
until column 0 is non-zero again: the library's rowlen state, like Q3, takes column 0 as non-zero from the
moment it is first set (a reload starts that afresh).
"""
from __future__ import annotations

import shutil

import numpy as np

from oracle import cpu
import parity_suite as ps
import smx_file

U32 = np.uint32
M16 = 65536            # columns c + i * M16 share their home slot c % S for every S <= 2^16


class History:
    """Op batches for the library and the checker.  Ops are kept per (stage, op) in the order they were
    added; stages run in order, so 'column 0 after the columns' is a later stage."""

    def __init__(self):
        self.parts: dict[tuple[int, str], list] = {}
        self.cells: dict[int, set] = {}         # row -> columns touched (queries)

    def add(self, stage, op, x, ys, vs):
        ys = np.asarray(ys, dtype=np.uint64).astype(U32)
        vs = np.broadcast_to(np.asarray(vs, dtype=np.uint64).astype(U32), ys.shape)
        self.parts.setdefault((stage, op), []).append((np.full(len(ys), x, U32), ys, vs))
        self.cells.setdefault(int(x), set()).update(int(y) for y in ys)

    def batches(self):
        for (stage, op) in sorted(self.parts, key=lambda k: k[0]):
            xs, ys, vs = (np.concatenate(a) for a in zip(*self.parts[stage, op]))
            yield op, xs, ys, vs

    def apply(self, *targets, after=None):
        """every batch to every target; after(): a check run after each batch"""
        for op, xs, ys, vs in self.batches():
            for t in targets:
                if isinstance(t, cpu.CpuMatrix):
                    t.apply(op, xs, ys, vs)
                else:
                    getattr(t, op + "_batch")(xs, ys, vs)
            if after:
                after()

    def queries(self):
        """rows, and (row, column) queries: every touched cell, column 0 and one missing column per row."""
        rows = np.array(sorted(self.cells), U32)
        qx, qy = [], []
        for x, cs in self.cells.items():
            cs = sorted(cs | {0, 0xFFFFFFF1})
            qx += [x] * len(cs)
            qy += cs
        return rows, np.array(qx, U32), np.array(qy, U32)


class _Rows:
    def __init__(self, seed):
        self.rng = np.random.default_rng(seed)
        self.n = 0

    def row(self):
        self.n += 1
        return (self.n * 2654435761 + 12345) % 2**32

    def cols(self, n):
        """n distinct random columns != 0 (random homes: ordinary collisions and runs)"""
        c = np.unique(self.rng.integers(1, 2**32, n + n // 4 + 8, dtype=np.uint64))[: n + n // 8 + 4]
        return self.rng.permutation(c)[:n]

    def vals(self, n):
        return self.rng.integers(1, 1000, n, dtype=np.uint64)


def edge_history(seed=1, sizes=(16, 32, 256, 4096), hiding=True, huge=()):
    """Rows at the edges where a row block is written at the wrong size or a cell is put where the reference's
    probe cannot find it.  hiding=False leaves out the rows whose *checker* layout has a zero-valued cell
    inside a probe run (the reference's own file hides cells behind it after a reload: DESIGN.md 8).
    `huge`: extra column counts for single rows with column 0 and zero-valued cells (the B200 runs)."""
    H, R = History(), _Rows(seed)
    follow = []                                              # rows that get the follow-up's growth
    for S in sizes:
        h = S // 2
        H.add(0, "incr", R.row(), R.cols(h), R.vals(h))                        # used = S/2
        r = R.row(); H.add(0, "incr", r, R.cols(h + 1), R.vals(h + 1))         # used = S/2 + 1
        follow.append((r, S))
        r = R.row(); H.add(0, "incr", r, R.cols(h + 1), R.vals(h + 1))         # S/2 + 2 cells: column 0
        H.add(1, "set", r, [0], [7])                                          # after the last growth (d=0, z=1)
        follow.append((r, S))
        L = 9 if S == 16 else h                                               # column 0 first: S=16 holds 10
        H.add(0, "incr", R.row(), np.r_[0, R.cols(L)], np.r_[3, R.vals(L)])   # cells, else used = S/2 + 1
        H.add(0, "incr", R.row(), R.cols(h + 2), R.vals(h + 2))                # the next S
    # column 0 non-zero, a growth (d = 1), then back to 0 (z = 0); then non-zero again and more growth
    b1 = R.row()
    H.add(0, "incr", b1, np.r_[0, 1:11], np.r_[5, R.vals(10)])
    H.add(3, "set", b1, [0], [0])
    b2 = R.row()
    H.add(0, "incr", b2, np.r_[0, 1:11], np.r_[5, R.vals(10)])
    H.add(3, "set", b2, [0], [0])
    H.add(4, "incr", b2, np.arange(11, 16), R.vals(5))                       # no growth while it is 0
    H.add(5, "set", b2, [0], [9])
    H.add(6, "incr", b2, np.arange(18, 41), R.vals(23))
    # many columns on one home; runs that wrap at the end of the block, with column 0 behind them
    H.add(0, "incr", R.row(), 7 + M16 * np.arange(1, 25), R.vals(24))
    r = R.row()
    H.add(0, "incr", r, M16 * np.arange(1, 21) - 1, R.vals(20))            # home S - 1 for every S
    H.add(1, "set", r, [0], [3])
    # column 0, then a zero-valued column homed at slot 0 and a zero-valued cell at the end of a run
    r = R.row()
    H.add(0, "incr", r, [0, 3, 4], [4, 1, 1])
    H.add(1, "set", r, [7 * M16, 4 + M16], [0, 0])
    # inline rows (<= 4 cells), 5 cells, with column 0 and a zero-valued cell
    for n in (1, 2, 3, 4, 5):
        H.add(0, "incr", R.row(), R.cols(n), R.vals(n))
    r = R.row(); H.add(0, "incr", r, np.r_[0, R.cols(3)], np.r_[2, R.vals(3)])
    r = R.row(); c = R.cols(4); H.add(0, "incr", r, c[:3], R.vals(3)); H.add(1, "set", r, c[3:], [0])
    # rows with no live cell: column 0 set to 0 only, and a row of zero-valued cells only
    H.add(1, "set", R.row(), [0], [0])
    r = R.row(); c = R.cols(40); H.add(1, "set", r, c, np.zeros(40))
    # a row the device keeps in a 2048-cell bucket at a reference size of 512
    r = R.row(); H.add(0, "incr", r, np.r_[0, R.cols(300)], np.r_[1, R.vals(300)])
    if hiding:
        # zero-valued cells (set 0, and incr wrapping to 0) in the middle of long probe runs
        r = R.row(); c = 5 + M16 * np.arange(1, 31); v = R.vals(30)
        H.add(0, "incr", r, c, v)
        H.add(1, "set", r, c[[9, 10, 19]], [0, 0, 0])
        H.add(2, "incr", r, c[14:15], [2**32 - int(v[14])])
        r = R.row(); c = M16 * np.arange(1, 21) - 1
        H.add(0, "incr", r, c, R.vals(20))
        H.add(1, "set", r, np.r_[0, c[[4, 11]]], [3, 0, 0])
        r = R.row(); c = R.cols(2500); v = R.vals(2500)                      # and in a big row
        H.add(0, "incr", r, np.r_[0, c], np.r_[6, v])
        H.add(1, "set", r, c[::97], 0)
        H.add(2, "incr", r, c[5::101], 2**32 - v[5::101].astype(np.int64))
    for n in huge:
        r = R.row(); c = R.cols(n); v = R.vals(n)
        H.add(0, "incr", r, np.r_[0, c], np.r_[1, v])
        if hiding:
            H.add(1, "set", r, c[::1009], 0)
    H.b_rows, H.follow = (b1, b2), follow
    return H


def follow_up(H, seed=2):
    """The same stream for both after a reload: column 0 turning non-zero (and back to 0 where that is
    safe), a new column in every row, `set 0` on an existing cell, growth past the next S."""
    F, rng = History(), np.random.default_rng(seed)
    for x, cs in H.cells.items():
        if x in H.b_rows:
            continue
        F.add(0, "set", x, [0], [11])
        F.add(1, "incr", x, rng.integers(1, 2**32, 1, dtype=np.uint64), [1])
        old = sorted(cs - {0})
        if old:
            F.add(2, "set", x, [old[len(old) // 2]], [0])
    for x in H.b_rows:
        top = max(H.cells[x]) + 1
        F.add(0, "set", x, [0], [11])
        F.add(1, "incr", x, np.arange(top, top + 3), [1])
        F.add(3, "set", x, [0], [0])
        F.add(4, "incr", x, np.arange(top + 3, top + 6), [2])                # no growth while it is 0
        F.add(5, "set", x, [0], [12])
        F.add(6, "incr", x, np.arange(top + 6, top + 60), [3])               # growth with column 0 non-zero
    for x, S in H.follow:
        F.add(4, "incr", x, rng.integers(1, 2**32, S // 2 + 2, dtype=np.uint64), [1])
    return F


def tile_history(seed=3):
    """Rows around the loader's tile (2^12 cells): 4095 / 4096 / 4097 live cells in 8192-cell blocks, a row of
    several tiles, rows with no live cell, and the edge rows."""
    H = edge_history(seed, sizes=(16, 256), hiding=False)
    R = _Rows(seed + 100)
    R.n = 10_000
    for n in (4095, 4096, 4097, 9000):
        H.add(0, "incr", R.row(), np.r_[0, R.cols(n)], np.r_[1, R.vals(n)])
    for n in (100, 5000):
        r = R.row(); c = R.cols(n); H.add(1, "set", r, c, np.zeros(n))
    return H


# ---------------------------------------------------------------------------------------- checks
def check_file(path, ck, rows):
    """The library's file against the checker's table: the same rows, each at the checker's row size, holding
    the checker's non-empty cells, every one found by the reference's probe before and after clearing."""
    f = smx_file.read(path)
    rows = np.asarray(rows, U32)
    sizes = np.array([ck.rowsize(int(x)) for x in rows])
    assert set(f) == set(rows[sizes > 0].tolist()), "the file's rows are not the checker's"
    bad = [(int(x), f[int(x)][0], int(s)) for x, s in zip(rows, sizes) if s and f[int(x)][0] != s]
    assert not bad, f"{len(bad)} rows at a size the checker does not have (row, ours, checker): {bad[:6]}"
    o, p = ck.getrow_many(rows)
    p = cpu.sort_rows(o, p)
    for i, x in enumerate(rows.tolist()):
        if x not in f:
            continue
        size, cells = f[x]
        got = np.array(smx_file.live(cells), U32).reshape(-1, 2)
        assert np.array_equal(got, p[o[i]:o[i + 1]]), f"row {x}: cells differ from the checker's"
        smx_file.check_row(x, size, cells)
    return f


def hidden(f):
    """(row, column) of the non-zero cells that the reference's positional load cannot find."""
    return {(x, int(c)) for x, (size, cells) in f.items()
            for c in smx_file.unreachable(size, smx_file.cleared(cells))}


def copy(path, to):
    return shutil.copy(path, to)


# ---------------------------------------------------------------------------------------- scenarios
def scenario_save_then_reload(make, tmp_path, huge=()):
    """Save side, then each library reloads the library's file and both continue."""
    H = edge_history(huge=huge)
    rows, qx, qy = H.queries()
    f = str(tmp_path / "ours.smx")
    m, ck = make(f), cpu.CpuMatrix("port")
    H.apply(m, ck)
    ps.compare(m, ck, rows, qx, qy)
    m.close()
    check_file(f, ck, rows)
    ck.close()
    ck2, m2 = cpu.CpuMatrix("port", copy(f, str(tmp_path / "for_checker.smx"))), make(copy(f, str(tmp_path / "r.smx")))
    ps.compare(m2, ck2, rows, qx, qy)                    # zero-valued cells are gone; rowlen is the recount
    F = follow_up(H)
    frows, fx, fy = F.queries()
    F.apply(m2, ck2, after=lambda: ps.compare(m2, ck2, rows, np.r_[qx, fx], np.r_[qy, fy]))
    m2.close(); ck2.close()


def scenario_each_reloads_its_own(make, tmp_path):
    """DESIGN.md 8: the library saves and reloads its file, the checker saves and reloads its own; both
    continue and agree (rowlen included) — the rows' sizes in the two files must be the same."""
    H = edge_history(seed=4, hiding=False)
    rows, qx, qy = H.queries()
    fo, fc = str(tmp_path / "ours.smx"), str(tmp_path / "checker.smx")
    m, ck = make(fo), cpu.CpuMatrix("port")
    H.apply(m, ck)
    m.close()
    ck.save(fc)
    ck.close()
    assert not hidden(smx_file.read(fc)), "the history must not hide cells in the checker's own file"
    m2, ck2 = make(fo), cpu.CpuMatrix("port", fc)
    ps.compare(m2, ck2, rows, qx, qy)
    F = follow_up(H, seed=5)
    frows, fx, fy = F.queries()
    F.apply(m2, ck2, after=lambda: ps.compare(m2, ck2, rows, np.r_[qx, fx], np.r_[qy, fy]))
    m2.close(); ck2.close()


def checker_files(tmp_path, H, layouts):
    """The checker's table for H, written once per layout -> (checker, {name: path})."""
    ck = cpu.CpuMatrix("port")
    H.apply(ck)
    out = {}
    for name, kw in layouts.items():
        out[name] = str(tmp_path / f"ck_{name}.smx")
        ck.save(out[name], **kw)
        f = smx_file.read(out[name])
        assert not hidden(f)
    return ck, out


LAYOUTS = {"plain": {}, "foreign": dict(shuffled=True, dead=True, unaligned=True, small_dir=True)}


def scenario_load_checker_files(make, open_sharded, tmp_path, worlds=(1, 2, 3)):
    """The checker's files (fresh, and laid out like an append-only writer's) load in the library — one
    handle, and sharded at each world — exactly as the checker's own positional load reads them."""
    H = tile_history()
    rows, qx, qy = H.queries()
    F = follow_up(H, seed=6)
    frows, fx, fy = F.queries()
    ck, files = checker_files(tmp_path, H, LAYOUTS)
    ck.close()
    for name, path in files.items():
        want = cpu.CpuMatrix("port", copy(path, str(tmp_path / f"want_{name}.smx")))
        m = make(copy(path, str(tmp_path / f"single_{name}.smx")))
        ps.compare(m, want, rows, qx, qy)
        for w in worlds:
            got = open_sharded(w, copy(path, str(tmp_path / f"w{w}_{name}.smx")), lambda s, r: answers(s, rows, qx, qy))
            for r in range(w):
                same(got[r], answers(want, rows, qx, qy), f"{name} file at world {w}, rank {r}")
        F.apply(m, want, after=lambda: ps.compare(m, want, rows, np.r_[qx, fx], np.r_[qy, fy]))   # the rowlen
        # automaton continues from the file's sizes
        m.close(); want.close()


def scenario_sharded_save(make, open_sharded, tmp_path, world):
    """A sharded snapshot passes the file checks against the checker's table, and the checker's load of it
    equals the library's."""
    H = edge_history(seed=7)
    rows, qx, qy = H.queries()
    ck = cpu.CpuMatrix("port")
    H.apply(ck)
    f = str(tmp_path / "sharded.smx")

    def build(s, r):
        sl = lambda a: a[r * len(a) // world:(r + 1) * len(a) // world]
        for op, xs, ys, vs in H.batches():
            getattr(s, op + "_batch")(sl(xs), sl(ys), sl(vs))
        return answers(s, rows, qx, qy)
    got = open_sharded(world, f, build)
    same(got[0], answers(ck, rows, qx, qy), f"the sharded table at world {world}")
    check_file(f, ck, rows)
    m, ck2 = make(copy(f, str(tmp_path / "single.smx"))), cpu.CpuMatrix("port", copy(f, str(tmp_path / "ck.smx")))
    ps.compare(m, ck2, rows, qx, qy)
    m.close(); ck2.close(); ck.close()


def scenario_hidden_cells(make, tmp_path):
    """The one deviation of a reload (DESIGN.md 8): in the reference's positional load, a zero-valued slot
    ahead of a non-zero cell in its probe run is cleared and hides that cell; the library re-inserts every
    non-zero cell.  The two differ exactly at the cells the file reader reports as hidden, nowhere else."""
    H = edge_history(seed=8, sizes=(16, 32))
    rows, qx, qy = H.queries()
    f = str(tmp_path / "checker.smx")
    ck = cpu.CpuMatrix("port")
    H.apply(ck)
    ck.save(f)
    ck.close()
    fr = smx_file.read(f)
    hid = hidden(fr)
    assert len(hid) >= 3, hid                             # the history makes some (and column 0 is one)
    ck2, m = cpu.CpuMatrix("port", copy(f, str(tmp_path / "ck.smx"))), make(copy(f, str(tmp_path / "m.smx")))
    a, b = np.asarray(m.get_batch(qx, qy)), ck2.get_many(qx, qy)
    differ = {(int(x), int(y)) for x, y in zip(qx[a != b], qy[a != b])}
    assert differ == {k for k in hid if k in set(zip(qx.tolist(), qy.tolist()))} == hid
    value = {(x, int(c)): int(v) for x, (size, cells) in fr.items() for c, v in smx_file.live(cells)}
    assert all(int(a[i]) == value[int(qx[i]), int(qy[i])] and b[i] == 0 for i in np.flatnonzero(a != b))
    assert (np.asarray(m.rowlen_batch(rows)) == ck2.rowlen_many(rows)).all()   # the recount sees hidden cells
    o1, p1 = m.getrow_batch(rows)
    o2, p2 = ck2.getrow_many(rows)
    assert (o1 == o2).all() and (cpu.sort_rows(o1, p1) == cpu.sort_rows(o2, p2)).all()
    m.close(); ck2.close()


# ---------------------------------------------------------------------------------------- helpers
def answers(m, rows, qx, qy):
    """gets, rowlens and column-sorted getrows of a library handle (collective when sharded) or the checker"""
    if isinstance(m, cpu.CpuMatrix):
        o, p = m.getrow_many(rows)
        return m.get_many(qx, qy), m.rowlen_many(rows), o, cpu.sort_rows(o, p)
    o, p = m.getrow_batch(rows)
    return (np.asarray(m.get_batch(qx, qy)).copy(), np.asarray(m.rowlen_batch(rows)).copy(),
            np.asarray(o).copy(), cpu.sort_rows(o, p))


def same(a, b, what):
    for k, name in enumerate(("get", "rowlen", "getrow offsets", "getrow pairs")):
        assert np.array_equal(np.asarray(a[k]), np.asarray(b[k])), f"{what}: {name} differs"
