"""SparseMatrix — the host-side mirror of the reference's binding classes over the C-ABI.

Method names and argument meaning follow the reference's Java class
(src/java/com/paulasmuth/libsmatrix/SparseMatrix.java:17-146: get/set/incr/decr/getRowLength/
getRow(x[, maxlen])/close/getFilename) and Ruby class (src/smatrix_ruby.c:166-174:
get/set/incr/decr returning the new value), so the parity tests read like the reference's own
TestSparseMatrix.java.  The `*_batch` methods call the batched C-ABI entry points; they accept
numpy arrays (host pointers) or CUDA torch tensors (device pointers, zero-copy).

No computation happens here: every method is one call into libsmatrix_b200.so.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import binding


def _is_torch(a) -> bool:
    return type(a).__module__.startswith("torch")


TOPK_MAX_K = 1024


def _topk_call(fn, items, k):
    """fn(items_ptr, n, k, counts_ptr, ids_ptr, scores_ptr) on outputs allocated where `items` lives."""
    if isinstance(k, bool) or not isinstance(k, (int, np.integer)) or not 1 <= int(k) <= TOPK_MAX_K:
        raise ValueError(f"k must be an integer in 1..{TOPK_MAX_K}, got {k!r}")
    k = int(k)
    if _is_torch(items) and items.is_cuda:
        import torch
        if items.dtype not in (torch.int32, torch.uint32):
            raise TypeError("torch batch arrays must be int32/uint32")
        items = items.contiguous()
        n = items.numel()
        counts = torch.empty(n, dtype=torch.int32, device=items.device)
        ids = torch.empty((n, k), dtype=torch.int32, device=items.device)
        scores = torch.empty((n, k), dtype=torch.float64, device=items.device)
        torch.cuda.current_stream(items.device).synchronize()      # the items may still be in flight on torch's stream
        fn(items.data_ptr(), n, k, counts.data_ptr(), ids.data_ptr(), scores.data_ptr())
        return counts, ids, scores
    if _is_torch(items):
        items = items.numpy()
    items = np.ascontiguousarray(items, dtype=np.uint32)
    n = len(items)
    counts = np.empty(n, dtype=np.uint32)
    ids = np.empty((n, k), dtype=np.uint32)
    scores = np.empty((n, k), dtype=np.float64)
    fn(items.ctypes.data, n, k, counts.ctypes.data, ids.ctypes.data, scores.ctypes.data)
    return counts, ids, scores


def _rec_call(fn, basket_offsets, items, k):
    """fn(off_ptr, items_ptr, n_baskets, k, counts_ptr, ids_ptr, scores_ptr) on outputs allocated where the baskets
    live; the offsets, the items and k are checked here, before any call into the library."""
    if isinstance(k, bool) or not isinstance(k, (int, np.integer)) or not 1 <= int(k) <= TOPK_MAX_K:
        raise ValueError(f"k must be an integer in 1..{TOPK_MAX_K}, got {k!r}")
    k = int(k)
    on_cuda = [_is_torch(a) and a.is_cuda for a in (basket_offsets, items)]
    if on_cuda[0] != on_cuda[1]:
        raise ValueError("basket offsets and items must both be CUDA tensors or both be host arrays")
    if on_cuda[0]:
        import torch
        if basket_offsets.device != items.device:
            raise ValueError("basket offsets and items must be on the same device")
        if basket_offsets.dtype != torch.int64 or items.dtype not in (torch.int32, torch.uint32):
            raise TypeError("torch baskets: int64 offsets and int32/uint32 items")
        off, items = basket_offsets.contiguous(), items.contiguous()
        if off.dim() != 1 or off.numel() < 1:
            raise ValueError("basket offsets need n_baskets + 1 entries")
        n = off.numel() - 1
        ok = torch.stack([off[0] == 0, off[-1] == items.numel(), (off[1:] >= off[:-1]).all()]).all()
        if not bool(ok):
            raise ValueError("basket offsets must start at 0, never decrease and end at len(items)")
        counts = torch.empty(n, dtype=torch.int32, device=items.device)
        ids = torch.empty((n, k), dtype=torch.int32, device=items.device)
        scores = torch.empty((n, k), dtype=torch.float64, device=items.device)
        torch.cuda.current_stream(items.device).synchronize()      # the inputs may still be in flight on torch's stream
        fn(off.data_ptr(), items.data_ptr(), n, k, counts.data_ptr(), ids.data_ptr(), scores.data_ptr())
        return counts, ids, scores
    if _is_torch(basket_offsets):
        basket_offsets = basket_offsets.numpy()
    if _is_torch(items):
        items = items.numpy()
    raw = np.asarray(basket_offsets)
    if raw.ndim != 1 or len(raw) < 1 or (len(raw) and raw.dtype.kind not in "iu"):
        raise ValueError("basket offsets need n_baskets + 1 integer entries")
    items = np.ascontiguousarray(items, dtype=np.uint32)
    if raw[0] != 0 or raw[-1] != len(items) or (np.diff(raw.astype(np.int64)) < 0).any():
        raise ValueError("basket offsets must start at 0, never decrease and end at len(items)")
    off = np.ascontiguousarray(raw, dtype=np.uint64)
    n = len(off) - 1
    counts = np.empty(n, dtype=np.uint32)
    ids = np.empty((n, k), dtype=np.uint32)
    scores = np.empty((n, k), dtype=np.float64)
    fn(off.ctypes.data, items.ctypes.data, n, k, counts.ctypes.data, ids.ctypes.data, scores.ctypes.data)
    return counts, ids, scores


def _check_key(name, v) -> int:
    if isinstance(v, bool) or not isinstance(v, (int, np.integer)) or not 0 <= int(v) <= 0xFFFFFFFF:
        raise ValueError(f"{name} must be an integer row key in 0..2^32 - 1, got {v!r}")
    return int(v)


def _check_count(name, v) -> int:
    if isinstance(v, bool) or not isinstance(v, (int, np.integer)) or int(v) < 1:
        raise ValueError(f"{name} must be an integer >= 1, got {v!r}")
    return int(v)


def _list_rows(fn, start, limit, bound, device, dev):
    """fn(from, keys_ptr, cap) -> m, into an array of min(limit, bound) keys (bound >= m) on the host or on CUDA
    device `dev`; -> the first min(limit, m) keys."""
    n = bound if limit is None else min(limit, bound)
    if device:
        import torch
        keys = torch.empty(n, dtype=torch.int32, device=torch.device("cuda", dev))
        ptr = keys.data_ptr()
    else:
        keys = np.empty(n, dtype=np.uint32)
        ptr = keys.ctypes.data
    got = min(int(fn(start, ptr if n else None, n)), n)
    if got == n:
        return keys
    return keys[:got].clone() if device else keys[:got].copy()


def _getrow_sorted(fn, xs):
    """fn(xs_ptr, n, offsets_ptr, pairs_ptr, cap) -> total: a CUDA tensor in -> (int64 offsets, int32 pairs) on its
    device; anything else -> numpy (uint64 offsets, uint32 pairs)."""
    if _is_torch(xs) and xs.is_cuda:
        import torch
        if xs.dtype not in (torch.int32, torch.uint32):
            raise TypeError("torch batch arrays must be int32/uint32")
        xs = xs.contiguous()
        n = xs.numel()
        offsets = torch.empty(n + 1, dtype=torch.int64, device=xs.device)
        torch.cuda.current_stream(xs.device).synchronize()      # the rows may still be in flight on torch's stream
        total = int(fn(xs.data_ptr(), n, None, None, 0))
        pairs = torch.empty((total, 2), dtype=torch.int32, device=xs.device)
        assert int(fn(xs.data_ptr(), n, offsets.data_ptr(), pairs.data_ptr() if total else None, total)) == total
        return offsets, pairs
    xs = np.ascontiguousarray(xs.numpy() if _is_torch(xs) else xs, dtype=np.uint32)
    n = len(xs)
    offsets = np.zeros(n + 1, dtype=np.uint64)
    total = int(fn(xs.ctypes.data, n, None, None, 0))          # the size query; the offsets come down once
    pairs = np.zeros((total, 2), dtype=np.uint32)
    assert int(fn(xs.ctypes.data, n, offsets.ctypes.data, pairs.ctypes.data if total else None, total)) == total
    return offsets, pairs


def _pages(m, start, rows_per_page, device):
    while True:
        keys = m.rows(start, rows_per_page, device)
        if len(keys) == 0:
            return
        yield (keys,) + tuple(m.getrow_sorted_batch(keys))
        last = int(keys[-1]) & 0xFFFFFFFF
        if len(keys) < rows_per_page or last == 0xFFFFFFFF:
            return
        start = last + 1


class DevPtr:
    """A raw device array of `n` uint32 (library- or peer-allocated memory that is not a tensor)."""
    __slots__ = ("ptr", "n")

    def __init__(self, ptr: int, n: int):
        self.ptr, self.n = int(ptr), int(n)

    def __len__(self):
        return self.n


class SparseMatrix:
    def __init__(self, file_path: str | None = None, device: int | None = None,
                 _lib_path: str | None = None, arena_gib: float | None = None):
        self._lib = binding.load(_lib_path)
        self.filename = file_path
        fname = file_path.encode() if file_path is not None else None
        if arena_gib is not None:       # explicit slab arena (otherwise $SMATRIX_ARENA_GIB, default: on demand)
            self._h = self._lib.smatrix_b200_open_arena(fname, int(device or 0), int(arena_gib * (1 << 30)))
        elif device is None:
            self._h = self._lib.smatrix_open(fname)
        else:
            self._h = self._lib.smatrix_b200_open(fname, int(device))
        if not self._h:
            # src/smatrix_jni.c:61-62 turns a NULL handle into IllegalArgumentException
            raise ValueError("smatrix_open() failed")

    @classmethod
    def _borrow(cls, lib, handle):
        """Wrap a handle somebody else owns (the C router's local shard); close() is the owner's job."""
        m = cls.__new__(cls)
        m._lib, m._h, m.filename = lib, handle, None
        return m

    # ---- handle plumbing -------------------------------------------------------------------
    def _handle(self):
        if not self._h:
            # src/smatrix_jni.c:15 ERR_PTRNOTFOUND
            raise ValueError("can't find native object. maybe close() was already called")
        return self._h

    def close(self):
        if self._h:
            self._lib.smatrix_close(self._h)
            self._h = None

    def __del__(self):  # src/smatrix_ruby.c:157-164: the GC finalizer closes the matrix
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def getFilename(self):
        return self.filename

    # ---- file mode ---------------------------------------------------------------------------
    def snapshot(self) -> int:
        """Write the whole .smx file now (temporary file, fsync, rename): 0, or -1 on failure or without a file."""
        return int(self._lib.smatrix_b200_snapshot(self._handle()))

    def checkpoint(self) -> int:
        """Persist only what changed: append the blocks of the rows written since the file last matched the table,
        a new directory, then switch the header to it (smatrix_b200_checkpoint).  The file loads to what a snapshot
        taken now would load to.  0, or -1 on failure or without a file; stat("dirty_rows") counts the rows the
        next checkpoint writes."""
        return int(self._lib.smatrix_b200_checkpoint(self._handle()))

    # ---- the reference API -----------------------------------------------------------------
    def get(self, x: int, y: int) -> int:
        return self._lib.smatrix_get(self._handle(), x & 0xFFFFFFFF, y & 0xFFFFFFFF)

    def set(self, x: int, y: int, val: int) -> int:
        return self._lib.smatrix_set(self._handle(), x & 0xFFFFFFFF, y & 0xFFFFFFFF, val & 0xFFFFFFFF)

    def incr(self, x: int, y: int, val: int) -> int:
        return self._lib.smatrix_incr(self._handle(), x & 0xFFFFFFFF, y & 0xFFFFFFFF, val & 0xFFFFFFFF)

    def decr(self, x: int, y: int, val: int) -> int:
        return self._lib.smatrix_decr(self._handle(), x & 0xFFFFFFFF, y & 0xFFFFFFFF, val & 0xFFFFFFFF)

    def getRowLength(self, x: int) -> int:
        return self._lib.smatrix_rowlen(self._handle(), x & 0xFFFFFFFF)

    rowlen = getRowLength

    def getrow_raw(self, x: int, ret_len_bytes: int, slack_pairs: int = 2) -> np.ndarray:
        """The literal smatrix_getrow call with a `ret_len_bytes` buffer -> (n, 2) pairs."""
        buf = np.zeros(2 * (ret_len_bytes // 8 + slack_pairs + 1), dtype=np.uint32)
        n = self._lib.smatrix_getrow(self._handle(), x & 0xFFFFFFFF, buf.ctypes.data, ret_len_bytes)
        return buf[: 2 * n].reshape(-1, 2).copy()

    def getRow(self, x: int, maxlen: int = 0) -> dict[int, int]:
        """Like src/smatrix_jni.c:114-149: rowlen -> buffer -> getrow -> (truncated) sorted map."""
        pairs = self.getrow_raw(x, (self.getRowLength(x) + 2) * 8)
        if maxlen > 0:
            pairs = pairs[:maxlen]
        return dict(sorted((int(k), int(v)) for k, v in pairs))

    # ---- batched entry points --------------------------------------------------------------
    @staticmethod
    def _arg(a, keep: list):
        """-> raw pointer (int) of a uint32 numpy array (host) or CUDA/CPU torch tensor."""
        if a is None:
            return None
        if isinstance(a, DevPtr):
            keep.append(a)
            return a.ptr
        if _is_torch(a):
            import torch
            if a.dtype not in (torch.int32, torch.uint32):
                raise TypeError("torch batch arrays must be int32/uint32")
            a = a.contiguous()
            keep.append(a)
            return a.data_ptr()
        a = np.ascontiguousarray(a, dtype=np.uint32)
        keep.append(a)
        return a.ctypes.data

    @staticmethod
    def _len(a) -> int:
        return a.n if isinstance(a, DevPtr) else (a.numel() if _is_torch(a) else len(a))

    @staticmethod
    def _on_device(a) -> bool:
        return isinstance(a, DevPtr) or (_is_torch(a) and a.is_cuda)

    @classmethod
    def _check_same(cls, arrays):
        """All batch arrays: the same length and all host or all device — the C side reads n entries from
        each raw pointer and abort()s the process on mixed placement, so refuse here instead."""
        arrays = [a for a in arrays if a is not None]
        n = cls._len(arrays[0])
        if any(cls._len(a) != n for a in arrays):
            raise ValueError("batch arrays must have the same length: " + ", ".join(str(cls._len(a)) for a in arrays))
        if len({cls._on_device(a) for a in arrays}) > 1:
            raise ValueError("batch arrays must be all host or all device arrays")
        return n

    @classmethod
    def _check_out(cls, out, n: int, like):
        if cls._len(out) < n:
            raise ValueError(f"out holds {cls._len(out)} entries, the batch has {n}")
        if cls._on_device(out) != cls._on_device(like):
            raise ValueError("out must live where the batch arrays live (host or device)")
        if _is_torch(out):
            import torch
            if out.dtype not in (torch.int32, torch.uint32) or not out.is_contiguous():
                raise TypeError("out must be a contiguous int32 / uint32 tensor")
        elif isinstance(out, np.ndarray):
            if out.dtype != np.uint32 or not out.flags.c_contiguous or not out.flags.writeable:
                raise TypeError("out must be a writable C-contiguous uint32 array")

    def _write(self, fn, xs, ys, vals):
        keep: list = []
        px, py, pv = self._arg(xs, keep), self._arg(ys, keep), self._arg(vals, keep)
        n = self._check_same(keep)
        fn(self._handle(), px, py, pv, n)

    def incr_batch(self, xs, ys, vals=None):
        self._write(self._lib.smatrix_incr_batch, xs, ys, vals)

    def decr_batch(self, xs, ys, vals=None):
        self._write(self._lib.smatrix_decr_batch, xs, ys, vals)

    def set_batch(self, xs, ys, vals=None):
        self._write(self._lib.smatrix_set_batch, xs, ys, vals)

    def _write_out(self, fn, xs, ys, vals):
        """-> out[i] = what the single-op call i would have returned (input order)."""
        keep: list = []
        px, py, pv = self._arg(xs, keep), self._arg(ys, keep), self._arg(vals, keep)
        self._check_same(keep)
        if _is_torch(keep[0]):
            import torch
            n = keep[0].numel()
            out = torch.empty(n, dtype=torch.int32, device=keep[0].device)
            fn(self._handle(), px, py, pv, n, out.data_ptr())
            return out
        n = len(keep[0])
        out = np.empty(n, dtype=np.uint32)
        fn(self._handle(), px, py, pv, n, out.ctypes.data)
        return out

    def incr_batch_out(self, xs, ys, vals=None):
        return self._write_out(self._lib.smatrix_incr_batch_out, xs, ys, vals)

    def decr_batch_out(self, xs, ys, vals=None):
        return self._write_out(self._lib.smatrix_decr_batch_out, xs, ys, vals)

    def set_batch_out(self, xs, ys, vals=None):
        return self._write_out(self._lib.smatrix_set_batch_out, xs, ys, vals)

    def get_batch(self, xs, ys, out=None):
        keep: list = []
        px, py = self._arg(xs, keep), self._arg(ys, keep)
        self._check_same(keep)
        if isinstance(keep[0], DevPtr):
            assert isinstance(out, DevPtr) and out.n >= keep[0].n
            self._lib.smatrix_get_batch(self._handle(), px, py, keep[0].n, out.ptr)
            return out
        if _is_torch(keep[0]):
            import torch
            n = keep[0].numel()
            if out is None:
                out = torch.empty(n, dtype=torch.int32, device=keep[0].device)
            self._check_out(out, n, keep[0])
            po = out.data_ptr()
        else:
            n = len(keep[0])
            if out is None:
                out = np.empty(n, dtype=np.uint32)
            self._check_out(out, n, keep[0])
            po = out.ctypes.data
        self._lib.smatrix_get_batch(self._handle(), px, py, n, po)
        return out

    def rowlen_batch(self, xs, out=None):
        keep: list = []
        px = self._arg(xs, keep)
        if isinstance(keep[0], DevPtr):
            assert isinstance(out, DevPtr)
            self._lib.smatrix_rowlen_batch(self._handle(), px, keep[0].n, out.ptr)
            return out
        if _is_torch(keep[0]):
            import torch
            if out is None:
                out = torch.empty(keep[0].numel(), dtype=torch.int32, device=keep[0].device)
            self._check_out(out, keep[0].numel(), keep[0])
            self._lib.smatrix_rowlen_batch(self._handle(), px, keep[0].numel(), out.data_ptr())
            return out
        if out is None:
            out = np.empty(len(keep[0]), dtype=np.uint32)
        self._check_out(out, len(keep[0]), keep[0])
        self._lib.smatrix_rowlen_batch(self._handle(), px, len(keep[0]), out.ctypes.data)
        return out

    def getrow_batch(self, xs):
        """-> (offsets[n+1] uint64, pairs[total, 2] uint32), host arrays; rows in table order."""
        keep: list = []
        px = self._arg(np.asarray(xs) if not _is_torch(xs) else xs.cpu().numpy(), keep)
        n = len(keep[0])
        offsets = np.zeros(n + 1, dtype=np.uint64)
        total = self._lib.smatrix_getrow_batch(self._handle(), px, n, offsets.ctypes.data, None, 0)
        pairs = np.zeros((int(total), 2), dtype=np.uint32)
        if total:
            got = self._lib.smatrix_getrow_batch(self._handle(), px, n, offsets.ctypes.data,
                                                 pairs.ctypes.data, int(total))
            assert got == total
        return offsets, pairs

    def cf_neighbors_batch(self, items):
        """examples/cf_recommender.c:50-86 for a batch of items -> (offsets[n+1], ids[total], scores[total])."""
        items = np.ascontiguousarray(items, dtype=np.uint32)
        n = len(items)
        offsets = np.zeros(n + 1, dtype=np.uint64)
        total = int(self._lib.smatrix_cf_neighbors_batch(self._handle(), items.ctypes.data, n,
                                                         offsets.ctypes.data, None, None, 0))
        ids = np.zeros(total, dtype=np.uint32)
        scores = np.zeros(total, dtype=np.float64)
        if total:
            self._lib.smatrix_cf_neighbors_batch(self._handle(), items.ctypes.data, n, offsets.ctypes.data,
                                                 ids.ctypes.data, scores.ctypes.data, total)
        return offsets, ids, scores

    def cf_topk_batch(self, items, k: int):
        """The k best neighbours of every item, ranked on the device (score descending, then id ascending) ->
        (counts[n], ids[n, k], scores[n, k]); slots past counts[i] hold id 0xFFFFFFFF and score -1.0.
        numpy (or any host sequence) in -> numpy out; a CUDA torch tensor in -> tensors on its device out
        (int32 counts and ids, float64 scores), with no copy through the host."""
        return _topk_call(lambda *a: self._lib.smatrix_cf_topk_batch(self._handle(), *a), items, k)

    def cf_recommend_batch(self, basket_offsets, items, k: int):
        """Per basket (items[basket_offsets[i]:basket_offsets[i+1]], e.g. one user's items), the k best other items
        by their summed neighbour scores, summed in basket order, ranked on the device (score descending, then id
        ascending) -> (counts[n], ids[n, k], scores[n, k]); slots past counts[i] hold id 0xFFFFFFFF and score -1.0.
        The basket's own items and id 0 are never recommended.  numpy in -> numpy out; CUDA torch tensors in (int64
        offsets, int32 items) -> tensors on their device out, with no copy through the host."""
        return _rec_call(lambda *a: self._lib.smatrix_cf_recommend_batch(self._handle(), *a), basket_offsets, items, k)

    # ---- enumeration -------------------------------------------------------------------------
    def rows(self, start: int = 0, limit: int | None = None, device: bool = False):
        """The row keys >= start in ascending order, at most `limit` of them (all by default): the rows a snapshot
        lists, including rows without pairs.  A uint32 numpy array, or with device=True an int32 CUDA tensor on the
        matrix's GPU that is filled without a copy through the host.  One pass over the directory per call."""
        start = _check_key("start", start)
        limit = None if limit is None else _check_count("limit", limit)
        return _list_rows(lambda *a: self._lib.smatrix_list_rows(self._handle(), *a), start, limit,
                          self.stat("rows"), device, self.device)

    def getrow_sorted_batch(self, xs):
        """getrow_batch with every row's pairs in ascending column order -> (offsets[n+1], pairs[total, 2]): numpy
        (uint64, uint32) for host rows, or int64 / int32 tensors on the device of a CUDA tensor of rows, with no copy
        through the host."""
        return _getrow_sorted(lambda *a: self._lib.smatrix_getrow_sorted_batch(self._handle(), *a), xs)

    def iter_rows(self, start: int = 0, rows_per_page: int = 1 << 20, device: bool = False):
        """Every row with key >= start exactly once, in key order, a page of at most rows_per_page rows at a time:
        yields (keys, offsets, pairs) = (rows(...), *getrow_sorted_batch(keys)), numpy or (device=True) CUDA tensors."""
        start = _check_key("start", start)
        rows_per_page = _check_count("rows_per_page", rows_per_page)
        return _pages(self, start, rows_per_page, device)

    # ---- device controls (include/smatrix_b200.h) --------------------------------------------
    def stat(self, name: str) -> int:
        return int(self._lib.smatrix_b200_stat(self._handle(), binding.STAT[name]))

    def sync(self):
        self._lib.smatrix_b200_sync(self._handle())

    def timer_start(self):
        self._lib.smatrix_b200_timer_start(self._handle())

    def timer_stop_ms(self) -> float:
        return float(self._lib.smatrix_b200_timer_stop_ms(self._handle()))

    def set_kernel_timing(self, on: bool):
        self._lib.smatrix_b200_set_kernel_timing(self._handle(), 1 if on else 0)

    def set_get_slices(self, mode: int):
        """0: point reads in input order; 1: by directory slice when rows repeat (default); 2: always."""
        self._lib.smatrix_b200_set_get_slices(self._handle(), int(mode))

    @property
    def device(self) -> int:
        return int(self._lib.smatrix_b200_device(self._handle()))

    @property
    def stream(self) -> int:
        return int(self._lib.smatrix_b200_stream(self._handle()) or 0)

    def dev_alloc(self, nbytes: int) -> int:
        return int(self._lib.smatrix_b200_dev_alloc(self._handle(), nbytes))

    def dev_free(self, ptr: int):
        self._lib.smatrix_b200_dev_free(self._handle(), ptr)

    def memcpy(self, dst: int, src: int, nbytes: int):
        self._lib.smatrix_b200_memcpy(self._handle(), dst, src, nbytes)

    def gen_c2_ops(self, seed, first, count, rows, ycols, d_xs: int, d_ys: int):
        self._lib.smatrix_b200_gen_c2_ops(self._handle(), seed, first, count, rows, ycols, d_xs, d_ys)

    def gen_c2_queries(self, seed_get, seed_build, first, count, n_build, rows, ycols, d_xs: int,
                       d_ys: int):
        self._lib.smatrix_b200_gen_c2_queries(self._handle(), seed_get, seed_build, first, count,
                                              n_build, rows, ycols, d_xs, d_ys)

    def gen_c3_ops(self, seed, first, count, d_thr: int, items: int, d_xs: int, d_ys: int):
        self._lib.smatrix_b200_gen_c3_ops(self._handle(), seed, first, count, d_thr, items, d_xs, d_ys)

    def gen_c3_queries(self, seed_get, seed_build, first, count, n_build, d_thr: int, items: int, d_xs: int, d_ys: int):
        self._lib.smatrix_b200_gen_c3_queries(self._handle(), seed_get, seed_build, first, count, n_build, d_thr,
                                              items, d_xs, d_ys)

    def gen_c4_lens(self, seed, first, count, d_thr: int, kmax: int, d_lens: int):
        self._lib.smatrix_b200_gen_c4_lens(self._handle(), seed, first, count, d_thr, kmax, d_lens)

    def gen_c4_ops(self, seed, first, count, d_offs: int, rows: int, d_xs: int, d_ys: int, d_vs: int):
        self._lib.smatrix_b200_gen_c4_ops(self._handle(), seed, first, count, d_offs, rows, d_xs, d_ys, d_vs)

    def probe_random_read(self, footprint_bytes: int, accesses: int, width: int = 32) -> float:
        return float(self._lib.smatrix_b200_probe_random_read(self._handle(), footprint_bytes,
                                                              accesses, width))

    def probe_random_atomic(self, footprint_bytes: int, accesses: int) -> float:
        return float(self._lib.smatrix_b200_probe_random_atomic(self._handle(), footprint_bytes,
                                                                accesses))
