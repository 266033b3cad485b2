"""File-backed mode = snapshot on open/close (SURVEY.md 8f N2): our .smx files interchange with the
reference's, byte format src/smatrix.c:30-72.  Shared by the CPU host-logic tests (simulator) and the
GPU tests."""
from __future__ import annotations

import os
import shutil

import numpy as np

from oracle import cpu
from conftest import safe_stream
import parity_suite as ps

U32 = np.uint32


def _build(m_apply, rng):
    """A matrix with column-0 traffic, zero-valued cells, an empty row and a long row."""
    xs, ys, vs = safe_stream(rng, 20000, 150, 90, "incr", col0_rate=0.08)
    m_apply("incr", xs, ys, vs)
    zx = np.arange(10, 20, dtype=U32); zy = np.full(10, 7, U32)
    m_apply("set", zx, zy, np.zeros(10, U32))                    # zero-valued cells: dropped by a reload
    m_apply("set", np.array([4000], U32), np.array([0], U32), np.array([0], U32))   # an empty row
    lx = np.full(3000, 5000, U32); ly = np.arange(1, 3001, dtype=U32) * U32(2654435761)
    m_apply("incr", lx, ly, np.arange(1, 3001, dtype=U32))
    rows = np.concatenate([np.arange(152, dtype=U32), np.array([4000, 5000, 77777], U32)])
    qx = np.concatenate([xs[:3000], zx, lx[:500]]); qy = np.concatenate([ys[:3000], zy, ly[:500]])
    return rows, qx, qy


def scenario_snapshot_interchange(make, tmp_path):
    """make(fname) -> SparseMatrix.  Four files: ours and the reference's, each reopened by both."""
    if not cpu.have_reference():
        import pytest
        pytest.skip("needs oracle/_ref (the reference's file mode)")
    ours_f, ref_f = str(tmp_path / "ours.smx"), str(tmp_path / "ref.smx")
    m, ref = make(ours_f), cpu.CpuMatrix("reference", ref_f)
    rng1, rng2 = np.random.default_rng(41), np.random.default_rng(41)
    rows, qx, qy = _build(lambda op, x, y, v: getattr(m, op + "_batch")(x, y, v), rng1)
    _build(lambda op, x, y, v: ref.apply(op, x, y, v), rng2)
    ps.compare(m, ref, rows, qx, qy)
    m.close(); ref.close()                                         # both write their files
    assert os.path.getsize(ours_f) >= 512 + 16 + 4194304 * 12    # header + one directory block
    head = open(ours_f, "rb").read(16)
    assert head[:8] == b"\x17" * 8 and int.from_bytes(head[8:16], "little") == 512
    import shutil
    more = safe_stream(np.random.default_rng(43), 6000, 160, 120, "incr", col0_rate=0.05)
    # every file is reopened by BOTH libraries (each on its own copy: both persist what follows)
    for k, src in enumerate((ours_f, ref_f)):
        a, b = str(tmp_path / f"copy{k}_for_ours.smx"), str(tmp_path / f"copy{k}_for_ref.smx")
        shutil.copy(src, a); shutil.copy(src, b)
        m2, r2 = make(a), cpu.CpuMatrix("reference", b)
        ps.compare(m2, r2, rows, qx, qy)                            # zero-valued cells are gone in both
        assert m2.get(10, 7) == 0 and m2.getRowLength(4000) == 0 and m2.stat("rows") >= 150
        ps.apply_both(m2, r2, "incr", *more)       # the rowlen automaton continues from the file's row sizes
        ps.compare(m2, r2, rows, more[0][:2000], more[1][:2000])
        m2.close(); r2.close()
    # and the two original files describe the same matrix: ours(ours_f) == ours(ref_f)
    m3, m4 = make(ours_f), make(ref_f)
    assert (np.asarray(m3.get_batch(qx, qy)) == np.asarray(m4.get_batch(qx, qy))).all()
    assert (np.asarray(m3.rowlen_batch(rows)) == np.asarray(m4.rowlen_batch(rows))).all()
    m3.close(); m4.close()


def scenario_snapshot_roundtrip_big(make, tmp_path, n_rows=30000):
    """ours -> ours at a size that needs several row chunks; every cell comes back."""
    f = str(tmp_path / "big.smx")
    rng = np.random.default_rng(47)
    n = n_rows * 12
    xs = rng.integers(0, n_rows, n).astype(U32) * U32(2654435761)
    ys = rng.integers(0, 4000, n).astype(U32)
    vs = rng.integers(1, 1000, n).astype(U32)
    m = make(f)
    m.incr_batch(xs, ys, vs)
    want = np.asarray(m.get_batch(xs, ys)).copy()
    rl = np.asarray(m.rowlen_batch(np.unique(xs))).copy()
    nnz = m.stat("nnz")
    m.close()
    m2 = make(f)
    assert m2.stat("nnz") == nnz and m2.stat("rows") == len(np.unique(xs))
    assert (np.asarray(m2.get_batch(xs, ys)) == want).all()
    rows = np.unique(xs)
    ck = cpu.CpuMatrix("port", shutil.copy(f, str(tmp_path / "checker.smx")))   # the reference's positional load
    assert (np.asarray(m2.rowlen_batch(rows)) == ck.rowlen_many(rows)).all()     # rowlen: the recount of the file
    assert (np.asarray(m2.get_batch(xs, ys)) == ck.get_many(xs, ys)).all()
    o1, p1 = m2.getrow_batch(rows)
    o2, p2 = ck.getrow_many(rows)
    assert (o1 == o2).all() and (cpu.sort_rows(o1, p1) == cpu.sort_rows(o2, p2)).all()
    ck.close()
    m2.close()
