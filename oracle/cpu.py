"""oracle/cpu.py — ctypes front-end for the CPU checkers.

TEST / BASELINE INFRASTRUCTURE ONLY (tests/, __graft_entry__.smoke(), bench.py's CPU legs).

Two interchangeable back-ends behind one class:
  kind="reference"  oracle/_ref/libsmatrix_ref.so — the UNMODIFIED reference compiled by
                    oracle/Makefile from /root/reference/src/smatrix.c (prebuilt file travels to
                    the GPU box; /root/reference itself is never read at run time)
  kind="port"       oracle/liboracle.so — our C restatement (smatrix_oracle.c)
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
REF_SO = os.path.join(HERE, "_ref", "libsmatrix_ref.so")
PORT_SO = os.path.join(HERE, "liboracle.so")
DRIVER_SO = os.path.join(HERE, "libsmxdriver.so")

_u32p = C.POINTER(C.c_uint32)
_u64p = C.POINTER(C.c_uint64)


def build(ref: bool = True) -> None:
    """Compile the checkers (gcc only).  `make ref` is a no-op without the reference checkout."""
    targets = ["oracle"] + (["ref"] if ref else [])
    subprocess.run(["make", "-s", "-C", HERE] + targets, check=True, stdout=subprocess.DEVNULL)


def have_reference() -> bool:
    return os.path.exists(REF_SO)


def _ptr(a: np.ndarray, t=_u32p):
    return a.ctypes.data_as(t)


def _u32(a) -> np.ndarray:
    return np.ascontiguousarray(a, dtype=np.uint32)


_driver = None


def driver():
    global _driver
    if _driver is None:
        if not os.path.exists(DRIVER_SO):
            build(ref=False)
        d = C.CDLL(DRIVER_SO)
        d.drv_getrow_many.restype = C.c_uint64
        d.drv_bench_c2_incr.restype = C.c_double
        d.drv_bench_c2_get.restype = C.c_double
        d.drv_bench_c2_incr.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_uint64, C.c_uint64,
                                        C.c_uint64, C.c_uint32, C.c_uint32]
        d.drv_bench_c2_get.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_uint64, C.c_uint64,
                                       C.c_uint64, C.c_uint64, C.c_uint64, C.c_uint32, C.c_uint32]
        d.drv_gen_c2_ops.argtypes = [C.c_uint64, C.c_uint64, C.c_size_t, C.c_uint32, C.c_uint32,
                                     _u32p, _u32p]
        d.drv_gen_c2_queries.argtypes = [C.c_uint64, C.c_uint64, C.c_uint64, C.c_size_t,
                                         C.c_uint64, C.c_uint32, C.c_uint32, _u32p, _u32p]
        d.drv_gen_c3_ops.argtypes = [C.c_uint64, C.c_uint64, C.c_size_t, _u64p, C.c_uint32, _u32p, _u32p]
        d.drv_gen_c3_queries.argtypes = [C.c_uint64, C.c_uint64, C.c_uint64, C.c_size_t, C.c_uint64, _u64p,
                                         C.c_uint32, _u32p, _u32p]
        d.drv_gen_c4_lens.argtypes = [C.c_uint64, C.c_uint64, C.c_size_t, _u64p, C.c_uint32, _u32p]
        d.drv_gen_c4_ops.argtypes = [C.c_uint64, C.c_uint64, C.c_size_t, _u64p, C.c_uint32, _u32p, _u32p, _u32p]
        d.drv_bench_apply.restype = C.c_double
        d.drv_bench_apply.argtypes = [C.c_void_p, C.c_void_p, C.c_int, _u32p, _u32p, _u32p, C.c_size_t]
        d.drv_bench_get.restype = C.c_double
        d.drv_bench_get.argtypes = [C.c_void_p, C.c_void_p, C.c_int, _u32p, _u32p, C.c_size_t]
        d.drv_bench_getrow.restype = C.c_double
        d.drv_bench_getrow.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, _u32p, C.c_size_t, _u64p]
        _driver = d
    return _driver


class CpuMatrix:
    """One matrix on the CPU, through either back-end; mirrors src/smatrix.h:87-94 plus bulk
    helpers that loop in C (oracle/smx_driver.c)."""

    def __init__(self, kind: str = "reference", fname: str | None = None):
        if kind == "reference":
            if not have_reference():
                raise FileNotFoundError(f"{REF_SO} missing: run `make -C oracle ref` where "
                                        "/root/reference exists")
            self.lib = C.CDLL(REF_SO)
            pre = "smatrix_"
        elif kind == "port":
            if not os.path.exists(PORT_SO):
                build(ref=False)
            self.lib = C.CDLL(PORT_SO)
            pre = "smx_oracle_"
        else:
            raise ValueError(kind)
        self.kind = kind
        L = self.lib
        self._f = {n: getattr(L, pre + n) for n in
                   ("open", "close", "get", "set", "incr", "decr", "rowlen", "getrow")}
        self._f["open"].restype = C.c_void_p
        self._f["open"].argtypes = [C.c_char_p]
        self._f["close"].argtypes = [C.c_void_p]
        self._f["close"].restype = None
        for n in ("set", "incr", "decr"):
            self._f[n].restype = C.c_uint32
            self._f[n].argtypes = [C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32]
        self._f["get"].restype = C.c_uint32
        self._f["get"].argtypes = [C.c_void_p, C.c_uint32, C.c_uint32]
        self._f["rowlen"].restype = C.c_uint32
        self._f["rowlen"].argtypes = [C.c_void_p, C.c_uint32]
        self._f["getrow"].restype = C.c_uint32
        self._f["getrow"].argtypes = [C.c_void_p, C.c_uint32, _u32p, C.c_size_t]
        self.h = C.c_void_p(self._f["open"](fname.encode() if fname else None))
        if not self.h:
            raise ValueError(f"cannot load {fname}") if fname else MemoryError("open failed")

    def fnptr(self, name: str) -> C.c_void_p:
        return C.cast(self._f[name], C.c_void_p)

    # single ops ---------------------------------------------------------------------------
    def get(self, x, y):
        return self._f["get"](self.h, x, y)

    def set(self, x, y, v):
        return self._f["set"](self.h, x, y, v)

    def incr(self, x, y, v):
        return self._f["incr"](self.h, x, y, v)

    def decr(self, x, y, v):
        return self._f["decr"](self.h, x, y, v)

    def rowlen(self, x):
        return self._f["rowlen"](self.h, x)

    # the restatement only: its row sizes and its file writer --------------------------------
    def rowsize(self, x) -> int:
        """Slot capacity S of row x (0 if the row does not exist)."""
        f = self.lib.smx_oracle_rowsize
        f.restype, f.argtypes = C.c_uint32, [C.c_void_p, C.c_uint32]
        return f(self.h, x)

    def save(self, fname: str, shuffled: bool = False, dead: bool = False, unaligned: bool = False,
             small_dir: bool = False) -> None:
        """Write the matrix as a .smx file (the rows' cell arrays as they are in memory).  The layout
        switches make the file look like one the reference's append-only writer leaves behind
        (oracle/smatrix_oracle.h: SMX_ORACLE_SAVE_*); the rows and cells are the same either way."""
        if self.kind != "port":
            raise NotImplementedError("the reference writes its file at close")
        flags = 1 * shuffled | 2 * dead | 4 * unaligned | 8 * small_dir
        f = self.lib.smx_oracle_save
        f.restype, f.argtypes = C.c_int, [C.c_void_p, C.c_char_p, C.c_int]
        if f(self.h, fname.encode(), flags) != 0:
            raise OSError(f"cannot write {fname}")

    def getrow_raw(self, x, ret_len_bytes: int, slack_pairs: int = 2) -> np.ndarray:
        """The literal C call with a caller buffer of `ret_len_bytes` (plus slack for the
        reference's one-pair / 4-byte overruns, SURVEY.md Q4).  Returns the (n, 2) pairs."""
        buf = np.zeros(2 * (ret_len_bytes // 8 + slack_pairs + 1), dtype=np.uint32)
        n = self._f["getrow"](self.h, x, _ptr(buf), ret_len_bytes)
        return buf[: 2 * n].reshape(-1, 2).copy()

    def getrow(self, x) -> list[tuple[int, int]]:
        """Whole row, sorted by column."""
        pairs = self.getrow_raw(x, (self.rowlen(x) + 2) * 8)
        return sorted((int(k), int(v)) for k, v in pairs)

    # bulk (loops in C) --------------------------------------------------------------------
    def apply(self, op: str, xs, ys, vs, want_out: bool = False):
        xs, ys, vs = _u32(xs), _u32(ys), _u32(vs)
        out = np.empty(len(xs), dtype=np.uint32) if want_out else None
        driver().drv_apply(self.fnptr(op), self.h, _ptr(xs), _ptr(ys), _ptr(vs),
                           C.c_size_t(len(xs)), _ptr(out) if want_out else None)
        return out

    def get_many(self, xs, ys) -> np.ndarray:
        xs, ys = _u32(xs), _u32(ys)
        out = np.empty(len(xs), dtype=np.uint32)
        driver().drv_get_many(self.fnptr("get"), self.h, _ptr(xs), _ptr(ys),
                              C.c_size_t(len(xs)), _ptr(out))
        return out

    def rowlen_many(self, xs) -> np.ndarray:
        xs = _u32(xs)
        out = np.empty(len(xs), dtype=np.uint32)
        driver().drv_rowlen_many(self.fnptr("rowlen"), self.h, _ptr(xs), C.c_size_t(len(xs)),
                                 _ptr(out))
        return out

    def getrow_many(self, xs):
        """(offsets[n+1] uint64, pairs[total, 2] uint32) in the back-end's table order."""
        xs = _u32(xs)
        lens = self.rowlen_many(xs).astype(np.uint64)
        cap = int(lens.sum() + 2 * len(xs) + 2)
        offsets = np.zeros(len(xs) + 1, dtype=np.uint64)
        pairs = np.zeros(2 * cap, dtype=np.uint32)
        total = driver().drv_getrow_many(self.fnptr("rowlen"), self.fnptr("getrow"), self.h,
                                         _ptr(xs), C.c_size_t(len(xs)), _ptr(offsets, _u64p),
                                         _ptr(pairs), C.c_uint64(cap))
        assert total != 0xFFFFFFFFFFFFFFFF
        return offsets, pairs[: 2 * total].reshape(-1, 2)

    # timing (pthread harness, src/smatrix_benchmark.c:98-132 shape) -----------------------
    def bench_c2_incr(self, threads, seed, first, count, rows, ycols) -> float:
        return driver().drv_bench_c2_incr(self.fnptr("incr"), self.h, threads, seed, first, count,
                                          rows, ycols)

    def bench_c2_get(self, threads, seed_get, seed_build, first, count, n_build, rows,
                     ycols) -> float:
        return driver().drv_bench_c2_get(self.fnptr("get"), self.h, threads, seed_get, seed_build,
                                         first, count, n_build, rows, ycols)

    # the same harness over pre-generated arrays (any workload)
    def bench_apply(self, op: str, threads: int, xs, ys, vs=None) -> float:
        xs, ys = _u32(xs), _u32(ys)
        vs = _u32(vs) if vs is not None else None
        return driver().drv_bench_apply(self.fnptr(op), self.h, threads, _ptr(xs), _ptr(ys),
                                        _ptr(vs) if vs is not None else None, len(xs))

    def bench_get(self, threads: int, xs, ys) -> float:
        xs, ys = _u32(xs), _u32(ys)
        return driver().drv_bench_get(self.fnptr("get"), self.h, threads, _ptr(xs), _ptr(ys), len(xs))

    def bench_getrow(self, threads: int, xs):
        """rowlen + getrow (full-size buffers) of every row in xs -> (seconds, pairs returned)"""
        xs = _u32(xs)
        pairs = C.c_uint64(0)
        secs = driver().drv_bench_getrow(self.fnptr("rowlen"), self.fnptr("getrow"), self.h, threads,
                                         _ptr(xs), len(xs), C.byref(pairs))
        return secs, int(pairs.value)

    def close(self):
        if self.h:
            self._f["close"](self.h)
            self.h = None

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()


def sort_rows(offsets: np.ndarray, pairs: np.ndarray) -> np.ndarray:
    """Sort each CSR row's pairs by column (the contract's comparison order, SURVEY.md Q5)."""
    out = pairs.copy()
    n = len(offsets) - 1
    if len(out) == 0:
        return out
    row_id = np.repeat(np.arange(n, dtype=np.uint64), np.diff(offsets).astype(np.int64))
    order = np.lexsort((out[:, 0], row_id))
    return out[order]


def gen_c2_ops(seed, first, count, rows, ycols):
    xs = np.empty(count, dtype=np.uint32)
    ys = np.empty(count, dtype=np.uint32)
    driver().drv_gen_c2_ops(seed, first, count, rows, ycols, _ptr(xs), _ptr(ys))
    return xs, ys


def gen_c2_queries(seed_get, seed_build, first, count, n_build, rows, ycols):
    xs = np.empty(count, dtype=np.uint32)
    ys = np.empty(count, dtype=np.uint32)
    driver().drv_gen_c2_queries(seed_get, seed_build, first, count, n_build, rows, ycols,
                                _ptr(xs), _ptr(ys))
    return xs, ys


# ---- C3 / C4 streams (SURVEY.md 8d): inverse-CDF thresholds + the generators of smx_driver.c -------
from libsmatrix_b200.workloads import zipf_thresholds  # noqa: E402,F401 - ONE definition for host and device


def gen_c3_ops(seed, first, count, thr):
    xs = np.empty(count, dtype=np.uint32)
    ys = np.empty(count, dtype=np.uint32)
    driver().drv_gen_c3_ops(seed, first, count, _ptr(thr, _u64p), len(thr), _ptr(xs), _ptr(ys))
    return xs, ys


def gen_c3_queries(seed_get, seed_build, first, count, n_build, thr):
    xs = np.empty(count, dtype=np.uint32)
    ys = np.empty(count, dtype=np.uint32)
    driver().drv_gen_c3_queries(seed_get, seed_build, first, count, n_build, _ptr(thr, _u64p), len(thr),
                                _ptr(xs), _ptr(ys))
    return xs, ys


def gen_c4_lens(seed, first, count, thr):
    lens = np.empty(count, dtype=np.uint32)
    driver().drv_gen_c4_lens(seed, first, count, _ptr(thr, _u64p), len(thr), _ptr(lens))
    return lens


def gen_c4_ops(seed, first, count, offs):
    """offs: exclusive prefix of the row lengths, rows + 1 entries (uint64)"""
    offs = np.ascontiguousarray(offs, dtype=np.uint64)
    xs = np.empty(count, dtype=np.uint32)
    ys = np.empty(count, dtype=np.uint32)
    vs = np.empty(count, dtype=np.uint32)
    driver().drv_gen_c4_ops(seed, first, count, _ptr(offs, _u64p), len(offs) - 1, _ptr(xs), _ptr(ys), _ptr(vs))
    return xs, ys, vs
