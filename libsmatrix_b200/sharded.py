"""One matrix row-sharded over the GPUs of one box (SURVEY.md 8e).

ShardedSparseMatrix is a thin ctypes wrapper over the C router (include/smatrix_shard.h,
csrc/smx_router.c): rendezvous through POSIX shared memory, batches routed by the partition
kernel's own stores over NVLink, no NCCL and no Python on the data path.

    owner(x) = mix_owner(x) mod world        (smatrix_b200_owner; independent of the directory hash)

One rank per GPU, as threads of one process or as one process per GPU.  Every rank holds a
complete private table for the rows it owns.  A batch call is collective: each rank passes ITS
slice of the batch (device tensors, or host arrays that are staged piece by piece); the ops travel
to the owners of their rows, and each rank updates only its own shard.

Input order.  The collective batch is the concatenation of the ranks' slices in rank order.
Routing permutes ops, and two results depend on order: which duplicate `set` wins, and the
history-dependent rowlen when column 0 turns non-zero in the same batch as new columns (SURVEY.md
Q1).  With `ordered=True` (default) every op travels with its global index and the owner applies
the batch through smatrix_b200_apply_ordered, which is bit-exact with the sequential reference.
`ordered=False` skips the index for incr/decr streams that never write column 0 (BASELINE configs
2 and 5): values never depend on order (addition mod 2^32 commutes), so the result is identical.
"""
from __future__ import annotations

import os

import numpy as np
import torch
import torch.distributed as dist

from .matrix import (DevPtr, SparseMatrix, _check_count, _check_key, _getrow_sorted, _list_rows, _rec_call,
                     _topk_call)

_seq = [0]


def default_name() -> str:
    """A rendezvous name every rank of one launch agrees on.  With a torch.distributed group already up,
    rank 0 picks it (pid + counter) and broadcasts it — plumbing only, once per matrix.  Otherwise it is
    derived from what the ranks of one launch share: the launcher's pid (torchrun agent / the test that
    spawned the ranks), the rendezvous port, and how many sharded matrices this process has opened so
    far (every rank opens them in the same order)."""
    _seq[0] += 1
    if dist.is_available() and dist.is_initialized():
        box = [f"smx_{os.getpid()}_{_seq[0]}" if dist.get_rank() == 0 else None]
        dist.broadcast_object_list(box, src=0)
        return box[0]
    return f"smx_{os.getppid()}_{os.environ.get('MASTER_PORT', '0')}_{_seq[0]}"


class ShardedSparseMatrix:
    """ctypes wrapper of smatrix_b200_shard_* — no computation and no routing logic here."""

    def __init__(self, rank: int, world: int, device: int = 0, name: str | None = None,
                 _lib_path: str | None = None, arena_gib: float | None = None, fname: str | None = None):
        """fname: file mode (include/smatrix_shard.h, smatrix_b200_shard_open_file) — the matrix is loaded from
        that .smx file if it exists and is non-empty and written back by snapshot() and close(); every rank
        passes the same path."""
        from . import binding
        self._lib = binding.load(_lib_path)
        self.rank, self.world = rank, world
        self._name = name or default_name()
        self.filename = fname
        if fname is not None:
            arena = (int(arena_gib * (1 << 30)) if arena_gib is not None
                     else int(os.environ.get("SMATRIX_ARENA_GIB") or "0", 0) << 30)
            self._h = self._lib.smatrix_b200_shard_open_file(self._name.encode(), rank, world, int(device), arena,
                                                             fname.encode())
        elif arena_gib is not None:
            self._h = self._lib.smatrix_b200_shard_open_arena(self._name.encode(), rank, world, int(device),
                                                              int(arena_gib * (1 << 30)))
        else:
            self._h = self._lib.smatrix_b200_shard_open(self._name.encode(), rank, world, int(device))
        if not self._h:
            raise RuntimeError("smatrix_b200_shard_open failed (no CUDA device or no peer access"
                               + (", or the file cannot be opened or is corrupt)" if fname is not None else ")"))
        self.local = SparseMatrix._borrow(self._lib, self._lib.smatrix_b200_shard_local(self._h))
        self._cuda = _lib_path is None

    def _handle(self):
        if not self._h:
            raise ValueError("sharded matrix is closed")
        return self._h

    @staticmethod
    def _n(a) -> int:
        return 0 if a is None else (a.numel() if torch.is_tensor(a) else len(a))

    def _write(self, fn, xs, ys, vals, *extra):
        keep: list = []
        A = SparseMatrix._arg
        px, py, pv = A(xs, keep), A(ys, keep), A(vals, keep)
        if torch.is_tensor(xs) and xs.is_cuda:
            torch.cuda.current_stream(xs.device).synchronize()   # inputs may still be in flight on torch's stream
        fn(self._handle(), px, py, pv, self._n(xs), *extra)

    def incr_batch(self, xs, ys, vals=None, ordered: bool = True):
        self._write(self._lib.smatrix_b200_shard_incr_batch, xs, ys, vals, 1 if ordered else 0)

    def decr_batch(self, xs, ys, vals=None, ordered: bool = True):
        self._write(self._lib.smatrix_b200_shard_decr_batch, xs, ys, vals, 1 if ordered else 0)

    def set_batch(self, xs, ys, vals=None):
        self._write(self._lib.smatrix_b200_shard_set_batch, xs, ys, vals)

    def _write_out(self, fn, xs, ys, vals, out):
        """-> out[i] = what single call i of the COLLECTIVE batch would have returned (input order)."""
        keep: list = []
        A = SparseMatrix._arg
        px, py, pv = A(xs, keep), A(ys, keep), A(vals, keep)
        if isinstance(xs, DevPtr):
            if not isinstance(out, DevPtr):
                raise ValueError("raw device arrays need a raw device `out`")
            po = out.ptr
        else:
            out = self._out_like(xs, out)
            po = out.data_ptr() if torch.is_tensor(out) else out.ctypes.data
        if torch.is_tensor(xs) and xs.is_cuda:
            torch.cuda.current_stream(xs.device).synchronize()
        fn(self._handle(), px, py, pv, self._n(xs), po)
        return out

    def incr_batch_out(self, xs, ys, vals=None, out=None):
        return self._write_out(self._lib.smatrix_b200_shard_incr_batch_out, xs, ys, vals, out)

    def decr_batch_out(self, xs, ys, vals=None, out=None):
        return self._write_out(self._lib.smatrix_b200_shard_decr_batch_out, xs, ys, vals, out)

    def set_batch_out(self, xs, ys, vals=None, out=None):
        return self._write_out(self._lib.smatrix_b200_shard_set_batch_out, xs, ys, vals, out)

    def _out_like(self, xs, out):
        n = self._n(xs)
        if out is not None:
            return out
        if torch.is_tensor(xs):
            return torch.empty(n, dtype=torch.int32, device=xs.device)
        return np.empty(n, dtype=np.uint32)

    def get_batch(self, xs, ys, out=None):
        keep: list = []
        A = SparseMatrix._arg
        out = self._out_like(xs, out)
        if torch.is_tensor(xs) and xs.is_cuda:
            torch.cuda.current_stream(xs.device).synchronize()
        self._lib.smatrix_b200_shard_get_batch(self._handle(), A(xs, keep), A(ys, keep), self._n(xs),
                                               out.data_ptr() if torch.is_tensor(out) else out.ctypes.data)
        return out

    def rowlen_batch(self, xs, out=None):
        keep: list = []
        out = self._out_like(xs, out)
        if torch.is_tensor(xs) and xs.is_cuda:
            torch.cuda.current_stream(xs.device).synchronize()
        self._lib.smatrix_b200_shard_rowlen_batch(self._handle(), SparseMatrix._arg(xs, keep), self._n(xs),
                                                  out.data_ptr() if torch.is_tensor(out) else out.ctypes.data)
        return out

    def getrow_batch(self, xs):
        """-> (offsets[n+1] uint64, pairs[total, 2] uint32) host arrays (rows in input order)."""
        xs = xs.cpu().numpy().view(np.uint32) if torch.is_tensor(xs) else np.ascontiguousarray(xs, dtype=np.uint32)
        n = len(xs)
        offsets = np.zeros(n + 1, dtype=np.uint64)
        h = self._handle()
        total = int(self._lib.smatrix_b200_shard_getrow_batch(h, xs.ctypes.data, n, offsets.ctypes.data, None, 0))
        # the fill is collective too: every rank makes the second call, with room for its own total
        pairs = np.zeros((max(total, 1), 2), dtype=np.uint32)
        got = int(self._lib.smatrix_b200_shard_getrow_batch(h, xs.ctypes.data, n, offsets.ctypes.data,
                                                            pairs.ctypes.data, max(total, 1)))
        assert got == total
        return offsets, pairs[:total]

    def cf_neighbors_batch(self, items):
        """examples/cf_recommender.c:50-86 for THIS rank's items -> (offsets[n+1], ids[total], scores[total]);
        collective (every rank calls it, each with its own items)."""
        items = np.ascontiguousarray(items, dtype=np.uint32)
        n = len(items)
        offsets = np.zeros(n + 1, dtype=np.uint64)
        h = self._handle()
        total = int(self._lib.smatrix_b200_shard_cf_neighbors_batch(h, items.ctypes.data, n, offsets.ctypes.data,
                                                                    None, None, 0))
        ids = np.zeros(max(total, 1), dtype=np.uint32)
        scores = np.zeros(max(total, 1), dtype=np.float64)
        got = int(self._lib.smatrix_b200_shard_cf_neighbors_batch(h, items.ctypes.data, n, offsets.ctypes.data,
                                                                  ids.ctypes.data, scores.ctypes.data, max(total, 1)))
        assert got == total
        return offsets, ids[:total], scores[:total]

    def cf_topk_batch(self, items, k: int):
        """The k best neighbours of THIS rank's items (contract of SparseMatrix.cf_topk_batch); collective."""
        return _topk_call(lambda *a: self._lib.smatrix_b200_shard_cf_topk_batch(self._handle(), *a), items, k)

    def cf_recommend_batch(self, basket_offsets, items, k: int):
        """Recommendations for THIS rank's baskets (contract of SparseMatrix.cf_recommend_batch); collective, and a
        rank may pass no baskets (offsets [0])."""
        return _rec_call(lambda *a: self._lib.smatrix_b200_shard_cf_recommend_batch(self._handle(), *a),
                         basket_offsets, items, k)

    def rows(self, start: int = 0, limit: int | None = None, device: bool = False):
        """Collective: SparseMatrix.rows of the whole sharded matrix.  Every rank passes the same start and limit
        and gets the same keys (device=True: on this rank's GPU)."""
        start = _check_key("start", start)
        limit = None if limit is None else _check_count("limit", limit)
        fn = lambda *a: self._lib.smatrix_b200_shard_list_rows(self._handle(), *a)
        return _list_rows(fn, start, limit, int(fn(start, None, 0)), device, self.local.device)

    def getrow_sorted_batch(self, xs):
        """Collective: SparseMatrix.getrow_sorted_batch for THIS rank's rows (a rank may pass none)."""
        return _getrow_sorted(lambda *a: self._lib.smatrix_b200_shard_getrow_sorted_batch(self._handle(), *a), xs)

    def getrow_batch_into(self, d_xs, n: int, d_offsets: int, d_pairs: int, pairs_cap: int) -> int:
        """The raw collective call on device (or host) pointers; returns the total number of pairs."""
        return int(self._lib.smatrix_b200_shard_getrow_batch(self._handle(), d_xs, n, d_offsets, d_pairs, pairs_cap))

    def reserve_route(self, max_ops_per_rank: int, max_pairs_per_rank: int = 0) -> bool:
        self._lib.smatrix_b200_shard_reserve(self._handle(), int(max_ops_per_rank), int(max_pairs_per_rank))
        return True

    def route_stats(self, reset: bool = False) -> dict:
        g = lambda k: int(self._lib.smatrix_b200_shard_stat(self._handle(), k))
        d = {"route_ms": g(0) / 1e6, "apply_ms": g(1) / 1e6, "routes": g(2), "remote_bytes": g(3), "max_inbox_ops": g(4)}
        if reset:
            self._lib.smatrix_b200_shard_stat_reset(self._handle())
        return d

    def snapshot(self) -> int:
        """Collective: write the .smx file now (smatrix_b200_shard_snapshot); 0, or -1 on every rank."""
        return int(self._lib.smatrix_b200_shard_snapshot(self._handle()))

    def checkpoint(self) -> int:
        """Collective: append the rows written since the file last matched the table and switch its header to a
        new directory (smatrix_b200_shard_checkpoint); 0, or -1 on every rank."""
        return int(self._lib.smatrix_b200_shard_checkpoint(self._handle()))

    def barrier(self):
        self._lib.smatrix_b200_shard_barrier(self._handle())

    def sum(self, v: int) -> int:
        return int(self._lib.smatrix_b200_shard_sum(self._handle(), int(v)))

    def max(self, v: int) -> int:
        return int(self._lib.smatrix_b200_shard_max(self._handle(), int(v)))

    def stat(self, name):
        return self.local.stat(name)

    _LOCAL_CONTROLS = frozenset((
        "timer_start", "timer_stop_ms", "set_kernel_timing", "set_get_slices", "sync", "gen_c2_ops", "gen_c2_queries",
        "gen_c3_ops", "gen_c3_queries", "gen_c4_lens", "gen_c4_ops", "probe_random_read",
        "probe_random_atomic", "dev_alloc", "dev_free", "memcpy", "device", "stream"))

    def __getattr__(self, name):
        # only controls of the local shard are forwarded; a call that is not sharded (single ops,
        # getRow, ...) must not silently run on one shard
        if name in ShardedSparseMatrix._LOCAL_CONTROLS:
            return getattr(self.local, name)
        raise AttributeError(f"{type(self).__name__} has no sharded '{name}' (it would only see this rank's rows)")

    def close(self):
        if self._h:
            self.local._h = None          # borrowed: the router closes it
            self._lib.smatrix_b200_shard_close(self._h)
            self._h = None

    def __del__(self):
        pass   # closing is collective: never from a finalizer


def open_sharded(rank: int, world: int, device: int = 0, name: str | None = None,
                 arena_gib: float | None = None, fname: str | None = None) -> ShardedSparseMatrix:
    """Collective: open this rank's part of a sharded matrix, file-backed when `fname` is given.  Raises
    RuntimeError on every rank alike (shard_open agrees on the outcome before anyone returns) when the router
    cannot be set up or the file cannot be opened or read."""
    return ShardedSparseMatrix(rank, world, device, name=name, arena_gib=arena_gib, fname=fname)
