"""CPU tests that PIN the oracle: the C restatement (oracle/smatrix_oracle.c) and the Python
semantic model (oracle/model.py) against (a) the reference's own known-answer cases and (b) the
unmodified reference compiled into oracle/_ref (skipped only when that file is absent)."""
import numpy as np
import pytest

from oracle import cpu
from oracle.model import ModelMatrix, is_resize_count
from conftest import safe_stream

KINDS = ["port"] + (["reference"] if cpu.have_reference() else [])
need_ref = pytest.mark.skipif(not cpu.have_reference(), reason="oracle/_ref not built")


# ------------------------------------------------------------------ the reference's own KATs
# src/java/test/TestSparseMatrix.java:22-166, restated at the C-API level (SURVEY.md 4).
@pytest.mark.parametrize("kind", KINDS)
def test_reference_known_answers(kind):
    with cpu.CpuMatrix(kind) as m:
        m.set(42, 23, 17)                                   # :27-28
        assert m.get(42, 23) == 17
        m.set(4231, 2634, 0); m.incr(4231, 2634, 1)         # :37-39
        assert m.get(4231, 2634) == 1
        m.set(1231, 2634, 0); m.incr(1231, 2634, 1); m.incr(1231, 2634, 5)  # :48-51
        assert m.get(1231, 2634) == 6
        i, n = np.meshgrid(np.arange(1000, dtype=np.uint32), np.arange(1000, dtype=np.uint32))
        xs, ys = i.ravel(), n.ravel()                       # :60-78  set(i, n, 34) for n, i
        m.apply("set", xs, ys, np.full(xs.shape, 34, np.uint32))
        assert (m.get_many(xs, ys) == 34).all()
        xs = np.arange(1000, dtype=np.uint32)               # :87-94 (depends on the state above)
        m.apply("incr", xs, np.full(1000, 42, np.uint32), np.ones(1000, np.uint32))
        assert m.rowlen(42) == 1000
        m.apply("incr", xs, np.full(1000, 85, np.uint32), np.ones(1000, np.uint32))   # :103-112
        assert len(m.getrow(85)) == 1000
        m.apply("incr", xs, np.full(1000, 83, np.uint32), np.ones(1000, np.uint32))   # :120-129
        row = m.getrow(83)
        assert len(row[:230]) == 230 and len(row) == 1000


@pytest.mark.parametrize("kind", KINDS)
def test_example_program_answers(kind):
    """examples/smatrix_example.c:17-48 in memory mode: 4 x 100 x incr over (1..29, 1..49)."""
    with cpu.CpuMatrix(kind) as m:
        n, i = np.meshgrid(np.arange(1, 30, dtype=np.uint32), np.arange(1, 50, dtype=np.uint32),
                           indexing="ij")
        xs = np.tile(n.ravel(), 400)
        ys = np.tile(i.ravel(), 400)
        m.apply("incr", xs, ys, np.ones(xs.shape, np.uint32))
        assert (m.get_many(n.ravel(), i.ravel()) == 400).all()
        assert m.rowlen(23) == 49


@pytest.mark.parametrize("kind", KINDS)
def test_quirks(kind):
    """SURVEY.md 8a Q1, Q2, Q4, Q6, Q7."""
    with cpu.CpuMatrix(kind) as m:
        m.incr(5, 0, 1)
        for c in range(1, 10):
            m.incr(5, c, 1)
        assert m.rowlen(5) == 9 and len(m.getrow(5)) == 10            # Q1
        m.incr(5, 10, 1)
        assert m.rowlen(5) == 11
        m.set(2, 5, 0)
        assert m.rowlen(2) == 1 and m.getrow(2) == [(5, 0)]           # Q2
        m.set(8, 0, 0)
        assert m.rowlen(8) == 0 and m.getrow(8) == []
        assert len(m.getrow_raw(5, 0)) == 1                            # Q4: at least one pair
        assert len(m.getrow_raw(5, 20)) == 3                           # ceil(20/8)
        assert m.get(77, 1) == 0 and m.rowlen(77) == 0 and m.getrow(77) == []   # Q6
        assert m.get(77, 1) == 0 and m.rowlen(77) == 0
        assert m.set(9, 9, 7) == 7 and m.incr(9, 9, 2) == 9 and m.decr(9, 9, 10) == 2**32 - 1  # Q7
        assert m.decr(9, 10, 3) == 2**32 - 3


# ------------------------------------------------------------------ restatement vs reference
@need_ref
@pytest.mark.parametrize("seed", range(6))
def test_port_matches_reference_exactly(seed):
    """Same ops -> same return values, same rowlen, and the same getrow *in table order* (the
    restatement reproduces the layout, so even truncated reads agree).  Deliberately includes
    column-0 traffic outside the safe domain (Q3) — layout-identical means corruption-identical."""
    rng = np.random.default_rng(seed)
    ref, port = cpu.CpuMatrix("reference"), cpu.CpuMatrix("port")
    n = 40000
    for op in ("incr", "set", "decr", "incr"):
        xs = rng.integers(0, 300, n).astype(np.uint32) * np.uint32(2654435761 if seed % 2 else 1)
        ys = rng.integers(0, 200 if seed < 4 else 2**32, n, dtype=np.uint64).astype(np.uint32)
        vs = rng.integers(0, 4, n).astype(np.uint32) if seed % 3 == 0 else \
            rng.integers(0, 2**32, n, dtype=np.uint64).astype(np.uint32)
        a = ref.apply(op, xs, ys, vs, want_out=True)
        b = port.apply(op, xs, ys, vs, want_out=True)
        assert (a == b).all()
    rows = np.unique(xs)
    q = np.concatenate([rows, rng.integers(0, 2**32, 50, dtype=np.uint64).astype(np.uint32)])
    assert (ref.rowlen_many(q) == port.rowlen_many(q)).all()
    oa, pa = ref.getrow_many(q)
    ob, pb = port.getrow_many(q)
    assert (oa == ob).all() and (pa == pb).all()
    for x in rows[:20]:
        for nbytes in (0, 8, 12, 64, 100):
            assert (ref.getrow_raw(int(x), nbytes) == port.getrow_raw(int(x), nbytes)).all()
    qx = rng.integers(0, 300, 5000).astype(np.uint32) * np.uint32(2654435761 if seed % 2 else 1)
    qy = rng.integers(0, 220, 5000).astype(np.uint32)
    assert (ref.get_many(qx, qy) == port.get_many(qx, qy)).all()
    ref.close(); port.close()


@need_ref
def test_directory_growth_matches_reference():
    """> 49152 rows forces the 65536-entry directory to double (src/smatrix.c:698)."""
    ref, port = cpu.CpuMatrix("reference"), cpu.CpuMatrix("port")
    xs = (np.arange(120000, dtype=np.uint32) * np.uint32(2654435761))
    ys = (np.arange(120000, dtype=np.uint32) % 7)
    vs = np.arange(120000, dtype=np.uint32) + 1
    ref.apply("incr", xs, ys, vs); port.apply("incr", xs, ys, vs)
    assert (ref.get_many(xs, ys) == port.get_many(xs, ys)).all()
    assert (ref.get_many(xs, ys) == vs).all()
    assert (ref.rowlen_many(xs) == port.rowlen_many(xs)).all()
    ref.close(); port.close()


# ------------------------------------------------------------------ semantic model vs C oracles
@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("seed", range(8))
def test_model_matches_oracle_on_safe_domain(kind, seed):
    rng = np.random.default_rng(100 + seed)
    model, m = ModelMatrix(), cpu.CpuMatrix(kind)
    wide = seed % 2 == 1
    for rnd in range(4):
        op = ("incr", "set", "decr", "incr")[(seed + rnd) % 4]
        xs, ys, vs = safe_stream(rng, 3000, 40, 60 if seed < 6 else 600, op,
                                 col0_rate=(0.0, 0.05, 0.3)[seed % 3], wide_keys=wide,
                                 max_val=5 if seed % 4 == 0 else 2**32 - 1)
        if op == "decr":  # keep column 0 in the safe domain: never decrement it
            ys = np.where(ys == 0, np.uint32(1 if not wide else 12345), ys).astype(np.uint32)
        got = m.apply(op, xs, ys, vs, want_out=True)
        want = [getattr(model, op)(int(x), int(y), int(v)) for x, y, v in zip(xs, ys, vs)]
        assert (got == np.array(want, dtype=np.uint32)).all()
        rows = np.unique(xs)
        assert [model.rowlen(int(x)) for x in rows] == list(m.rowlen_many(rows))
        for x in rows[:15]:
            assert model.getrow(int(x)) == m.getrow(int(x))
    m.close()


def test_resize_counts():
    assert [n for n in range(1, 300) if is_resize_count(n)] == [10, 18, 34, 66, 130, 258]


@pytest.mark.parametrize("kind", KINDS)
def test_cf_rowlen_collapse(kind):
    """SURVEY.md 8a: when a row's first write is incr(x,0,1) (examples/cf_recommender.c:39),
    rowlen = n for n <= 9 and n + 1 for n >= 10 (n = non-zero columns)."""
    with cpu.CpuMatrix(kind) as m:
        for n in (1, 5, 9, 10, 11, 17, 18, 40, 100):
            x = 1000 + n
            m.incr(x, 0, 1)
            for c in range(1, n + 1):
                m.incr(x, c, 1)
            assert m.rowlen(x) == (n if n <= 9 else n + 1)


# ------------------------------------------------------------------ streams
def test_c2_stream_definition():
    """drv_gen_c2_* against an independent numpy evaluation of SURVEY.md 8(d)."""
    def splitmix(z):
        z = (z + np.uint64(0x9E3779B97F4A7C15))
        z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
        z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
        return z ^ (z >> np.uint64(31))
    with np.errstate(over="ignore"):
        i = np.arange(1000, 6000, dtype=np.uint64)
        r = splitmix(np.uint64(2) + i)
        x = ((r >> np.uint64(32)) % np.uint64(13_000_000)).astype(np.uint32) * np.uint32(2654435761)
        y = (np.uint64(1) + (r & np.uint64(0xFFFFFFFF)) % np.uint64(256)).astype(np.uint32)
    xs, ys = cpu.gen_c2_ops(2, 1000, 5000, 13_000_000, 256)
    assert (xs == x).all() and (ys == y).all()
    qx, qy = cpu.gen_c2_queries(3, 2, 0, 4000, 6000, 13_000_000, 256)
    assert (qy[1::2] > 256).all() and (qy[0::2] <= 256).all()


@pytest.mark.parametrize("kind", KINDS)
def test_pthread_harness_is_exact(kind):
    """BASELINE.md 2: multi-threaded incr totals are exact, so the harness is a valid oracle."""
    with cpu.CpuMatrix(kind if kind == "reference" else "port") as m:
        threads = 4 if kind == "reference" else 1   # the restatement has no locks
        secs = m.bench_c2_incr(threads, 2, 0, 200000, 500, 16)
        assert secs > 0
        xs, ys = cpu.gen_c2_ops(2, 0, 200000, 500, 16)
        keys, counts = np.unique(xs.astype(np.uint64) << np.uint64(32) | ys, return_counts=True)
        got = m.get_many((keys >> np.uint64(32)).astype(np.uint32), keys.astype(np.uint32))
        assert (got == counts).all()
        m.bench_c2_get(threads, 3, 2, 0, 50000, 200000, 500, 16)


# ------------------------------------------------------------------ committed golden fixtures
def _replay_golden(make_matrix):
    import os
    gdir = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
    files = sorted(f for f in os.listdir(gdir) if f.endswith(".npz"))
    assert len(files) >= 4
    for f in files:
        g = np.load(os.path.join(gdir, f))
        m = make_matrix()
        for k in range(int(g["n_batches"])):
            m.apply(str(g[f"op{k}"]), g[f"xs{k}"], g[f"ys{k}"], g[f"vs{k}"])
        assert (m.get_many(g["qx"], g["qy"]) == g["get"]).all(), f
        assert (m.rowlen_many(g["rows"]) == g["rowlen"]).all(), f
        o, p = m.getrow_many(g["rows"])
        assert (o == g["offsets"]).all() and (cpu.sort_rows(o, p) == g["pairs_sorted"]).all(), f
        m.close()


@pytest.mark.parametrize("kind", KINDS)
def test_golden_fixtures(kind):
    """tests/golden/*.npz were recorded from the unmodified reference (make_golden.py)."""
    _replay_golden(lambda: cpu.CpuMatrix(kind))


def test_lazy_rowlen_automaton_equals_stepwise():
    """DESIGN.md 2: catching the (S, d) state up lazily gives the reference's `used` as long as the
    state is synced right before column 0 turns non-zero."""
    from oracle.model import catch_up
    rng = np.random.default_rng(5)
    for _ in range(300):
        n_total = int(rng.integers(1, 700))
        flip = int(rng.integers(0, n_total + 1))          # column 0 becomes non-zero after `flip` inserts
        checkpoints = sorted(set(int(c) for c in rng.integers(0, n_total + 1, 4)) | {flip, n_total})
        # step-by-step reference automaton
        S, U, L, z = 16, 0, 0, False
        want = {}
        for n in range(n_total + 1):
            if n == flip:
                z = True
            if n in checkpoints:
                want[n] = U
            if n < n_total:
                if U > S // 2:
                    S *= 2
                    U = L + (1 if z else 0)
                U += 1
                L += 1
        # lazy: sync only at the flip, evaluate at arbitrary checkpoints
        slog, d, z = 4, 0, False
        for c in checkpoints:
            if c == flip:
                slog, d = catch_up(slog, d, c, False)     # the k_sync_rowlen moment
                z = True
            s2, d2 = catch_up(slog, d, c, z)
            assert c + d2 == want[c], (n_total, flip, c)


# ------------------------------------------------------------------ file mode
@need_ref
def test_file_mode_matches_reference(tmp_path):
    """The restatement's .smx writer and positional loader against the reference's file mode: each loads the
    other's file (and its own), and all four give the same answers, getrow in table order included."""
    import shutil
    rng = np.random.default_rng(77)
    rf = str(tmp_path / "ref.smx")
    ref, port = cpu.CpuMatrix("reference", rf), cpu.CpuMatrix("port")
    for op in ("incr", "set", "incr"):
        xs, ys, vs = safe_stream(rng, 20000, 120, 90, op, col0_rate=0.05, max_val=3)   # zero-valued cells too
        ref.apply(op, xs, ys, vs); port.apply(op, xs, ys, vs)
    rows = np.unique(xs)
    pf = str(tmp_path / "port.smx")
    port.save(pf, shuffled=True, dead=True, unaligned=True, small_dir=True)
    ref.close(); port.close()
    loaded = [cpu.CpuMatrix(kind, shutil.copy(src, str(tmp_path / f"{kind}_{k}.smx")))
              for k, src in enumerate((rf, pf)) for kind in ("reference", "port")]
    qx, qy = np.repeat(rows, 92), np.tile(np.arange(92, dtype=np.uint32), len(rows))
    want = loaded[0]
    for m in loaded[1:]:
        assert (m.get_many(qx, qy) == want.get_many(qx, qy)).all()
        assert (m.rowlen_many(rows) == want.rowlen_many(rows)).all()
        oa, pa = m.getrow_many(rows)
        ob, pb = want.getrow_many(rows)
        assert (oa == ob).all() and (pa == pb).all()
    for m in loaded:
        m.close()
