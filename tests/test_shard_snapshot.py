"""File mode of the sharded matrix (include/smatrix_shard.h: smatrix_b200_shard_open_file / _snapshot) and the
device-side reader of .smx files (smatrix_b200_load_*), on the CPU: ranks are THREADS of this process driving
the simulator library, as in tests/test_router_threads.py.  Tiny windows and pieces make every load cross many
windows, pieces and tiles; one sharded .smx file must interchange with the single-GPU one in every direction."""
import hashlib
import os
import shutil
import struct
import threading

import numpy as np
import pytest

from libsmatrix_b200.matrix import SparseMatrix
from libsmatrix_b200.sharded import ShardedSparseMatrix
from oracle import cpu
import snapshot_suite as ss

U32 = np.uint32
_seq = [0]


@pytest.fixture(scope="module")
def sim():
    from hostsim import build as hb
    return hb.build()


@pytest.fixture(scope="module")
def sim32():
    from hostsim import build as hb
    return hb.build(defines=["-DSMX_SIM_WARP32"], suffix="_warp32")


@pytest.fixture(autouse=True)
def knobs(monkeypatch):
    monkeypatch.setenv("SMATRIX_DIR_LOG2", "8")
    monkeypatch.setenv("SMATRIX_LOAD_WINDOW", "4096")     # a few rows per pread; the 3000-column row grows it
    monkeypatch.setenv("SMATRIX_LOAD_CELLS", "700")       # and a few rows per piece
    monkeypatch.setenv("SMATRIX_SHARD_INBOX", "1024")     # the inboxes grow on demand
    monkeypatch.setenv("SMATRIX_SHARD_TIMEOUT", "60")


def ranks(world, fn):
    """fn(rank) on `world` threads -> list of results by rank; any rank's exception fails the test."""
    out, errors = [None] * world, []

    def main(r):
        try:
            out[r] = fn(r)
        except BaseException as e:                       # noqa: BLE001 - reported below
            import traceback
            errors.append(f"rank {r}: {e!r}\n{traceback.format_exc()}")
    ts = [threading.Thread(target=main, args=(r,)) for r in range(world)]
    for t in ts:
        t.start()
    for t in ts:
        t.join(timeout=280)
    assert not errors, "\n".join(errors)
    assert not any(t.is_alive() for t in ts), "a rank hangs"
    return out


def _name():
    _seq[0] += 1
    return f"smxsnap_{os.getpid()}_{_seq[0]}"


def open_sharded(lib, world, fname, fn):
    """fn(m, rank) on every rank of a sharded matrix over `fname`, then a collective close."""
    name = _name()

    def body(r):
        m = ShardedSparseMatrix(r, world, 0, name=name, _lib_path=lib, fname=fname)
        try:
            return fn(m, r)
        finally:
            m.close()
    return ranks(world, body)


def view(m, rows, qx, qy, sharded):
    """gets, rowlens, column-sorted getrows and the table totals — the same on every rank of a sharded matrix."""
    o, p = m.getrow_batch(rows)
    stats = [m.stat(k) for k in ("rows", "nnz", "value_sum")]
    if sharded:
        stats = [m.sum(v) % 2**64 for v in stats]
    return (np.asarray(m.get_batch(qx, qy)).copy(), np.asarray(m.rowlen_batch(rows)).copy(),
            o.copy(), cpu.sort_rows(o, p), stats)


def same(a, b, what):
    for k, (x, y) in enumerate(zip(a, b)):
        assert np.array_equal(np.asarray(x), np.asarray(y)), f"{what}: part {k} differs"


# ------------------------------------------------------------------ 1 / 5: save and reload at any world
@pytest.mark.parametrize("world", [2, 3, "2-warp32"])
def test_sharded_file_interchanges_with_single_gpu(sim, sim32, world, tmp_path):
    lib = sim
    if world == "2-warp32":      # the expansion kernels' ballots and prefixes on the 32-lane lock-step simulator
        lib, world = sim32, 2
    other = {2: 3, 3: 1}[world]
    fa, fb = str(tmp_path / "single.smx"), str(tmp_path / "sharded.smx")
    more = ss.safe_stream(np.random.default_rng(43), 6000, 160, 120, "incr", col0_rate=0.05)

    m = SparseMatrix(fa, _lib_path=lib)
    rows, qx, qy = ss._build(lambda op, x, y, v: getattr(m, op + "_batch")(x, y, v), np.random.default_rng(41))
    before = view(m, rows, qx, qy, False)
    o, p = before[2], before[3]
    zero_cells = int(((p[:, 1] == 0) & (p[:, 0] != 0)).sum())
    assert zero_cells == 10
    m.close()

    def build(m, r):
        sl = lambda a: a[r * len(a) // world:(r + 1) * len(a) // world]
        ss._build(lambda op, x, y, v: getattr(m, op + "_batch")(sl(x), sl(y), sl(v)), np.random.default_rng(41))
        return view(m, rows, qx, qy, True)
    built = open_sharded(lib, world, fb, build)
    same(built[0], before, "sharded build vs single-GPU build")
    assert built[world - 1] is not None

    def single(f):
        m = SparseMatrix(f, _lib_path=lib)
        got = view(m, rows, qx, qy, False)
        m.incr_batch(*more)
        after = view(m, rows, more[0][:2000], more[1][:2000], False)
        m.close()
        return got, after

    def sharded(f, w):
        def fn(m, r):
            got = view(m, rows, qx, qy, True)
            sl = lambda a: a[r * len(a) // w:(r + 1) * len(a) // w]
            m.incr_batch(sl(more[0]), sl(more[1]), sl(more[2]))
            return got, view(m, rows, more[0][:2000], more[1][:2000], True)
        out = open_sharded(lib, w, f, fn)
        for r in range(1, w):
            same(out[r][0], out[0][0], f"rank {r} vs rank 0")
        return out[0]

    copies = {}
    for k, f in (("a", fa), ("b", fb)):
        for j in range(2):
            copies[k, j] = str(tmp_path / f"{k}{j}.smx")
            shutil.copy(f, copies[k, j])
    results = {"A single": single(copies["a", 0]), "B single": single(copies["b", 0]),
               f"A sharded at {world}": sharded(copies["a", 1], world),
               f"B sharded at {other}": sharded(copies["b", 1], other)}
    ref_got, ref_after = results["A single"]
    want_stats = [before[4][0], before[4][1] - zero_cells, before[4][2]]
    assert ref_got[4] == want_stats, (ref_got[4], want_stats)
    assert ref_got[0][-510:-500].tolist() == [0] * 10            # the zero-valued cells are gone
    for what, (got, after) in results.items():
        same(got, ref_got, what)
        same(after, ref_after, what + ", after the follow-up stream")   # rowlen continues from the file's sizes


# ------------------------------------------------------------------ 2: a reference-style file
def _ref_file(path):
    """Two chained directory blocks (the first partly used), row blocks out of directory order, one at an
    offset that is not 8-byte aligned; sizes 1 .. 8192 with column-0 cells, zero-valued cells and rows with
    no live cell.  Returns the model: row -> {column: value} of the cells with a non-zero value."""
    rng = np.random.default_rng(5)
    rows = []                                                  # (key, size, cells[(col, val)] in slot order)
    for key, size in ((11, 1), (12, 2), (13, 16), (14, 64), (15, 1), (16, 8192), (17, 32), (18, 4), (19, 256)):
        cols = rng.choice(np.arange(1, 10 * size + 10), size, replace=False).astype(np.uint64)
        vals = rng.integers(1, 2**32, size, dtype=np.uint64)
        vals[rng.random(size) < 0.3] = 0                      # zero-valued cells
        empty = rng.random(size) < 0.2                          # empty slots
        cols[empty], vals[empty] = 0, 0
        if key in (11, 18):
            vals[:] = 0                                         # no live cell at all
        if key in (13, 16):
            cols[3 % size], vals[3 % size] = 0, 77 + key        # column 0
        rows.append((key, size, list(zip(cols.tolist(), vals.tolist()))))
    blocks = [(6, 4), (5, 5)]                                  # (slots, entries used)
    pos = 512 + sum(16 + 12 * b[0] for b in blocks)
    order = [4, 0, 7, 2, 8, 1, 6, 3, 5]                         # the file order of the row blocks
    rpos = {}
    body = b""
    for k, i in enumerate(order):
        if k == 3:
            body += b"\0" * 4                                   # the next row block is 4 bytes off alignment
        key, size, cells = rows[i]
        rpos[i] = pos + len(body)
        body += b"\x23" * 8 + struct.pack("<Q", size) + b"".join(struct.pack("<II", c, v) for c, v in cells)
    head = b"\x17" * 8 + struct.pack("<Q", 512) + b"\0" * 496
    d, at, e = b"", 512, 0
    for b, (slots, used) in enumerate(blocks):
        d += struct.pack("<QQ", slots, at + 16 + 12 * slots if b + 1 < len(blocks) else 0)
        for s in range(slots):
            d += struct.pack("<IQ", rows[e][0], rpos[e]) if s < used else struct.pack("<IQ", 0, 0)
            e += s < used
        at += 16 + 12 * slots
    assert e == len(rows)
    open(path, "wb").write(head + d + body)
    return {key: {c: v for c, v in cells if v != 0} for key, size, cells in rows}


def test_reference_style_file_loads_single_and_sharded(sim, tmp_path):
    f = str(tmp_path / "ref.smx")
    model = _ref_file(f)
    keys = np.array(sorted(model), U32)
    qx = np.array([k for k in model for c in list(model[k]) + [0, 123456]], U32)
    qy = np.array([c for k in model for c in list(model[k]) + [0, 123456]], U32)
    want_get = np.array([model[int(x)].get(int(y), 0) for x, y in zip(qx, qy)], U32)
    want_len = np.array([len(model[int(k)]) for k in keys], U32)
    want_rows = [sorted(model[int(k)].items()) for k in keys]

    def check(m, sharded):
        assert (np.asarray(m.get_batch(qx, qy)) == want_get).all()
        assert (np.asarray(m.rowlen_batch(keys)) == want_len).all()
        o, p = m.getrow_batch(keys)
        p = cpu.sort_rows(o, p)
        for i in range(len(keys)):
            assert [tuple(c) for c in p[o[i]:o[i + 1]].tolist()] == want_rows[i], f"row {keys[i]}"
        n_rows = m.sum(m.stat("rows")) if sharded else m.stat("rows")
        assert n_rows == len(keys)                               # rows without a live cell exist too
        return True

    g = shutil.copy(f, str(tmp_path / "g.smx"))
    m = SparseMatrix(g, _lib_path=sim)
    check(m, False)
    m.close()
    for w in (1, 2, 3):
        g = shutil.copy(f, str(tmp_path / f"s{w}.smx"))
        assert all(open_sharded(sim, w, g, lambda m, r: check(m, True)))


# ------------------------------------------------------------------ 3: corrupt files
def _good_file(sim, path):
    m = SparseMatrix(path, _lib_path=sim)
    m.incr_batch(np.repeat(np.arange(40, dtype=U32), 20), np.tile(np.arange(1, 21, dtype=U32), 40), None)
    m.close()
    data = bytearray(open(path, "rb").read())
    first = 512 + 16 + 4194304 * 12                             # the first row block
    return data, first


@pytest.mark.parametrize("damage", ["row-magic", "size-not-power-of-two", "truncated-row"])
def test_corrupt_file_fails_on_every_rank(sim, tmp_path, damage):
    f = str(tmp_path / "bad.smx")
    data, first = _good_file(sim, f)
    if damage == "row-magic":
        data[first + 7] = 0x24
    elif damage == "size-not-power-of-two":
        data[first + 8:first + 16] = struct.pack("<Q", 48)
    else:
        del data[-100:]
    open(f, "wb").write(bytes(data))
    digest = hashlib.sha256(bytes(data)).hexdigest()
    with pytest.raises(ValueError):
        SparseMatrix(f, _lib_path=sim)
    for w in (1, 3):
        name = _name()

        def body(r):
            with pytest.raises(RuntimeError):
                ShardedSparseMatrix(r, w, 0, name=name, _lib_path=sim, fname=f)
            return True
        assert all(ranks(w, body))
    assert hashlib.sha256(open(f, "rb").read()).hexdigest() == digest   # never overwritten


# ------------------------------------------------------------------ 4: a snapshot that fails
def test_failed_snapshot_returns_minus_one_everywhere(sim, tmp_path):
    d = tmp_path / "data"
    d.mkdir()
    f = str(d / "m.smx")
    name = _name()
    barrier = threading.Barrier(2)

    def body(r):
        m = ShardedSparseMatrix(r, 2, 0, name=name, _lib_path=sim, fname=f)
        m.incr_batch(np.arange(r * 50, r * 50 + 50, dtype=U32), np.ones(50, U32), None)
        assert m.snapshot() == 0
        good = open(f, "rb").read()
        barrier.wait()
        if r == 0:
            os.mkdir(f + ".tmp")                                # the temporary file cannot be created
        barrier.wait()
        m.incr_batch(np.arange(r * 50, r * 50 + 50, dtype=U32), np.ones(50, U32), None)
        rc = m.snapshot()
        barrier.wait()
        assert open(f, "rb").read() == good                     # the previous file is intact
        if r == 0:
            shutil.rmtree(d)                                    # no directory at all any more
        barrier.wait()
        rc2 = m.snapshot()
        m.close()                                               # says so loudly and closes anyway
        return rc, rc2
    assert ranks(2, body) == [(-1, -1), (-1, -1)]


# ------------------------------------------------------------------ 6: the interchange scenario at world 1
class _World1:
    """A sharded world-1 matrix with the single-op reads the scenario asks for."""

    def __init__(self, lib, f):
        self.m = ShardedSparseMatrix(0, 1, 0, name=_name(), _lib_path=lib, fname=f)

    def get(self, x, y):
        return int(self.m.get_batch(np.array([x], U32), np.array([y], U32))[0])

    def getRowLength(self, x):
        return int(self.m.rowlen_batch(np.array([x], U32))[0])

    def __getattr__(self, k):
        return getattr(self.m, k)


def test_snapshot_interchange_sharded_world1(sim, tmp_path):
    ss.scenario_snapshot_interchange(lambda f: _World1(sim, f), tmp_path)
