"""One matrix row-sharded over the GPUs of one box (SURVEY.md 8e).

Two implementations of the same collective API:

  ShardedSparseMatrix       the product: a thin ctypes wrapper over the C router
                            (include/smatrix_shard.h, csrc/smx_router.c) — rendezvous through POSIX
                            shared memory, batches routed by the partition kernel's own stores over
                            NVLink, no NCCL and no Python on the data path.
  TorchShardedSparseMatrix  the fallback when peer memory cannot be mapped, and the gloo / CPU test
                            vehicle: torch.distributed all-to-all-v (described below).

open_sharded() picks the C router and falls back (on every rank alike) when it cannot be set up.

TorchShardedSparseMatrix

    owner(x) = mix_owner(x) mod world        (smatrix_b200_owner; independent of the directory hash)

One process per GPU (torch.distributed, backend nccl over NVLink/NVSwitch).  Every rank holds a
complete private table for the rows it owns.  A batch call is collective: each rank passes ITS
slice of the batch (device tensors, or host arrays that are staged piece by piece); the slice is
bucketed by owner on the device (K8) and moved to the owners, and each rank updates only its own
shard.  Two routes:

  * peer memory (default on CUDA): the per-owner counts are all-gathered (world x world, tiny) and
    ONE scatter kernel writes every owner's run straight into that owner's inbox — symmetric
    buffers mapped through CUDA IPC, plain stores over NVLink (smatrix_b200_route_p2p).  Reads: the
    owners' look-up kernels write the answers straight into the requester's answer buffer, in a
    staggered order so that no GPU is ever the target of all the others at once, and the
    requester un-permutes them (smatrix_b200_gather).
  * NCCL (fallback; gloo on CPU for the tests): partition into a send buffer, one all-to-all-v of
    the (x, y, value) triples, reverse all-to-all-v for reads.

Input order.  The collective batch is the concatenation of the ranks' slices in rank order.
Routing permutes ops, and two results depend on order: which duplicate `set` wins, and the
history-dependent rowlen when column 0 turns non-zero in the same batch as new columns (SURVEY.md
Q1).  With `ordered=True` (default) every op travels with its global index (16 B/op instead of
12) and the owner applies the batch through smatrix_b200_apply_ordered, which is bit-exact with
the sequential reference.  `ordered=False` skips the index for incr/decr streams that never
write column 0 (BASELINE configs 2 and 5): values never depend on order (addition mod 2^32
commutes), so the result is identical.
"""
from __future__ import annotations

import contextlib
import os

import numpy as np
import torch
import torch.distributed as dist

import ctypes as C

from .matrix import DevPtr, SparseMatrix, _topk_call


class _PeerBuffers:
    """Symmetric buffers for the fused route: per generation an inbox (x, y, v, order index) that
    the other ranks' scatter kernels write into, and an answer buffer that owners' read kernels
    write into — all peer-mapped through CUDA IPC, i.e. plain stores over NVLink / NVSwitch."""
    GENS = 3            # routed / in flight / being applied (see ShardedSparseMatrix._write)
    ARRAYS = ("x", "y", "v", "o", "b")
    LOCAL_ONLY = ("p",)  # inverse permutation of my own queries: never touched by a peer

    def __init__(self, sm: "TorchShardedSparseMatrix", cap_ops: int):
        self.sm, self.cap, self.gen = sm, int(cap_ops), 0
        lib, h = sm._lib, sm.router._handle()
        self.local = {(g, a): int(lib.smatrix_b200_dev_alloc(h, self.cap * 4))
                      for g in range(self.GENS) for a in self.ARRAYS + self.LOCAL_ONLY}
        mine = {}
        for k, ptr in self.local.items():
            if k[1] in self.LOCAL_ONLY:
                continue
            buf = (C.c_ubyte * 64)()
            if lib.smatrix_b200_ipc_export(h, ptr, buf) != 0:
                raise RuntimeError("cudaIpcGetMemHandle failed")
            mine[k] = bytes(buf)
        everyone = [None] * sm.world
        dist.all_gather_object(everyone, mine, group=sm.group)
        self.peer = []
        for r in range(sm.world):
            if r == sm.rank:
                self.peer.append(dict(self.local))
                continue
            opened = {}
            for k, hb in everyone[r].items():
                p = lib.smatrix_b200_ipc_open(h, (C.c_ubyte * 64).from_buffer_copy(hb))
                if not p:
                    raise RuntimeError("cudaIpcOpenMemHandle failed")
                opened[k] = int(p)
            self.peer.append(opened)
        if os.environ.get("SMX_ROUTE_WARM", "1") != "0":
            # first stores through a freshly opened IPC mapping are slow (the mapping is completed
            # lazily): push every peer array once now, so the first routed batch runs at NVLink speed
            for r in range(sm.world):
                if r != sm.rank:
                    for k, p in self.peer[r].items():
                        lib.smatrix_b200_memcpy(h, p, self.local[k], self.cap * 4)
            dist.barrier(group=sm.group)

    def next_gen(self) -> int:
        self.gen = (self.gen + 1) % self.GENS
        return self.gen

    def close(self):
        lib, h = self.sm._lib, self.sm.router._handle()
        for r, d in enumerate(self.peer):
            if r != self.sm.rank:
                for p in d.values():
                    lib.smatrix_b200_ipc_close(h, p)
        dist.barrier(group=self.sm.group)     # nobody frees memory a peer still maps
        for p in self.local.values():
            lib.smatrix_b200_dev_free(h, p)


class TorchShardedSparseMatrix:
    def __init__(self, rank: int, world: int, device: int = 0, group=None, _lib_path: str | None = None,
                 p2p: bool | None = None):
        self.rank, self.world, self.group = rank, world, group
        self._use_p2p = (_lib_path is None) if p2p is None else p2p   # CUDA build: peer memory; else NCCL/gloo
        self._peers: _PeerBuffers | None = None
        self.local = SparseMatrix(device=device, _lib_path=_lib_path)
        arena = os.environ.pop("SMATRIX_ARENA_GIB", None)               # the router holds no data:
        os.environ["SMATRIX_STREAM_HIGH_PRIORITY"] = "1"                 # no arena, and a high-priority
        try:                                                             # stream so K8 interleaves with
            self.router = SparseMatrix(device=device, _lib_path=_lib_path)   # an update in flight
        finally:
            os.environ.pop("SMATRIX_STREAM_HIGH_PRIORITY", None)
            if arena is not None:
                os.environ["SMATRIX_ARENA_GIB"] = arena
        self._lib = self.local._lib
        self._pool = None
        self._bufs: dict[str, torch.Tensor] = {}
        self._gen = 0
        self._side = self._side_down = None      # upload / download streams of the host-array path
        self._cuda = _lib_path is None
        self.dev = torch.device("cuda", device) if self._cuda else torch.device("cpu")

    # ------------------------------------------------------------------ plumbing
    def _buf(self, n, like=None):
        return torch.empty(n, dtype=torch.int32, device=self.dev)

    def _slot(self, name: str, n: int):
        """Grow-only reusable device buffer (no allocator traffic in steady state)."""
        b = self._bufs.get(name)
        if b is None or b.numel() < n:
            b = torch.empty(max(n + n // 8, 1024), dtype=torch.int32, device=self.dev)
            self._bufs[name] = b
        return b[:n]

    def _up(self, name: str, t):
        """Host arrays (numpy or CPU tensors, ideally pinned) are staged into a reusable device
        buffer on torch's current stream; device tensors pass through."""
        if t is None:
            return None
        if isinstance(t, np.ndarray):
            t = torch.from_numpy(t.view(np.int32))
        if t.device == self.dev:
            return t
        d = self._slot("up_" + name, t.numel())
        d.copy_(t, non_blocking=True)
        return d

    HOST_PIECE = 1 << 24

    def _host_pieces(self, arrays, n: int):
        """Order-free host batches: yield (lo, hi, device tensors) piece by piece; the upload of
        piece k+1 runs on a side stream while the caller routes / applies piece k.  Collective: every
        rank yields the same number of pieces (its own may be empty)."""
        pieces = max(1, -(-self._nmax(n) // self.HOST_PIECE))
        if self._side is None and self._cuda:
            self._side = torch.cuda.Stream(self.dev)
        as_t = lambda t: None if t is None else (torch.from_numpy(t.view(np.int32)) if isinstance(t, np.ndarray) else t)
        arrays = [as_t(t) for t in arrays]

        def issue(k):
            lo, hi = k * n // pieces, (k + 1) * n // pieces
            out = []
            ctx = torch.cuda.stream(self._side) if self._side is not None else contextlib.nullcontext()
            with ctx:
                for i, t in enumerate(arrays):
                    if t is None:
                        out.append(None)
                        continue
                    d = self._slot(f"hp{k & 1}_{i}", hi - lo)
                    d.copy_(t[lo:hi], non_blocking=True)
                    out.append(d)
                ev = None
                if self._side is not None:
                    ev = torch.cuda.Event()
                    ev.record(self._side)
            return lo, hi, out, ev

        cur = issue(0)
        for k in range(pieces):
            nxt = issue(k + 1) if k + 1 < pieces else None
            if cur[3] is not None:
                cur[3].synchronize()
            yield cur[0], cur[1], cur[2]
            cur = nxt

    def _sync_torch(self):
        if self._cuda:
            torch.cuda.current_stream(self.dev).synchronize()

    def _partition(self, xs, ys, vals, want_src: bool, want_pos: bool = False):
        n = xs.numel()
        g = self._gen = (self._gen + 1) % 3      # three generations: routed / in flight / being applied
        oxs = self._slot(f"ox{g}", n)
        oys = self._slot(f"oy{g}", n) if ys is not None else None
        ovs = self._slot(f"ov{g}", n) if vals is not None else None
        osrc = self._slot(f"os{g}", n) if want_src else None
        opos = self._slot(f"op{g}", n) if want_pos else None
        counts = np.zeros(self.world, dtype=np.uint64)
        p = lambda t: t.data_ptr() if t is not None else None
        self._sync_torch()   # inputs may have been produced on torch's stream
        # the router has its own handle (own stream + mutex) so that routing the next sub-batch can
        # overlap the update of the current one
        self._lib.smatrix_b200_partition2(self.router._handle(), p(xs), p(ys), p(vals), n, self.world,
                                          counts.ctypes.data, p(oxs), p(oys), p(ovs), p(osrc), p(opos))
        return [int(c) for c in counts], oxs, oys, ovs, osrc, opos

    def _exchange_counts(self, send):
        t = torch.tensor(send, dtype=torch.int64, device=self.dev)
        r = torch.empty_like(t)
        dist.all_to_all_single(r, t, group=self.group)
        return [int(v) for v in r.tolist()]

    def _a2a(self, t, send, recv, name=None):
        out = self._slot(name, sum(recv)) if name else self._buf(sum(recv))
        dist.all_to_all_single(out, t, output_split_sizes=recv, input_split_sizes=send, group=self.group)
        return out

    def _route(self, xs, ys, vals, want_src=False, ordered=False, want_pos=False):
        send, oxs, oys, ovs, osrc, opos = self._partition(xs, ys, vals, want_src or ordered, want_pos)
        recv = self._exchange_counts(send)
        g = self._gen
        rx = self._a2a(oxs, send, recv, f"rx{g}")
        ry = self._a2a(oys, send, recv, f"ry{g}") if oys is not None else None
        rv = self._a2a(ovs, send, recv, f"rv{g}") if ovs is not None else None
        rord = None
        if ordered:   # global index = (ops in the slices of lower ranks) + index inside my slice
            sizes = torch.zeros(self.world, dtype=torch.int64, device=self.dev)
            sizes[self.rank] = xs.numel()
            dist.all_reduce(sizes, group=self.group)
            if int(sizes.sum()) >= 2**32 - 1:
                raise ValueError("ordered collective batches are limited to 2^32 - 2 ops")
            base = int(sizes[: self.rank].sum())
            gidx = (osrc.long() + base).to(torch.int32)   # wraps into uint32 bit pattern
            rord = self._a2a(gidx, send, recv)
        self._sync_torch()   # the library runs on its own stream
        return send, recv, rx, ry, rv, (opos if want_pos else osrc), rord

    # ------------------------------------------------------------------ fused route over peer memory
    def _ensure_peers(self, nmax: int) -> bool:
        """(Re)create the symmetric buffers for batches of up to nmax ops per rank.  Collective:
        every rank calls it with the same nmax."""
        if not self._use_p2p or self.world == 1:
            return False
        need = int(nmax * 1.25) + 65536
        if self._peers is None or self._peers.cap < need:
            peers, err = None, None
            try:
                if self._peers is not None:
                    self._peers.close()
                    self._peers = None
                peers = _PeerBuffers(self, need)
            except Exception as e:            # no peer access on this box
                err = e
            # agree on the outcome: one failed rank and EVERY rank falls back to the NCCL path together
            # (a rank that stayed on the peer route alone would wait for collectives nobody else calls)
            ok = torch.tensor([0 if err else 1], device=self.dev)
            dist.all_reduce(ok, op=dist.ReduceOp.MIN, group=self.group)
            if int(ok.item()) == 0:
                if peers is not None:
                    peers.close()
                self._peers, self._use_p2p = None, False
                print(f"[smatrix sharded] peer-memory route unavailable ({err or 'a peer failed'}); "
                      "using NCCL all-to-all", flush=True)
                return False
            self._peers = peers
        return True

    def reserve_route(self, max_ops_per_rank: int) -> bool:
        """Collective set-up of the peer-memory route for batches of up to max_ops_per_rank ops
        (symmetric inboxes + CUDA IPC exchange, ~15 x 5 B/op of HBM per rank).  Optional: the first
        batch does it lazily; call it to keep that cost out of a timed region."""
        return self._ensure_peers(self._nmax(max_ops_per_rank))

    def _route_p2p(self, xs, ys, vals, ordered=False, want_pos=False):
        """K8 fused with the exchange: count per owner, all-gather the world x world count matrix
        (tiny), then ONE scatter kernel writes every owner's run straight into that owner's inbox
        over NVLink.  Returns None (on every rank alike) if some inbox would overflow."""
        pb, W, me, n = self._peers, self.world, self.rank, xs.numel()
        lib, rh = self._lib, self.router._handle()
        ptr = lambda t: t.data_ptr() if t is not None else None
        self._sync_torch()
        counts = np.zeros(W, dtype=np.uint64)
        if n:
            lib.smatrix_b200_partition_count(rh, ptr(xs), n, W, counts.ctypes.data)
        mine = torch.from_numpy(counts.astype(np.int64)).to(self.dev)
        allc = torch.empty(W * W, dtype=torch.int64, device=self.dev)
        dist.all_gather_into_tensor(allc, mine, group=self.group)
        cnt = allc.view(W, W).cpu().numpy()              # cnt[s][o]: ops sender s has for owner o
        if int(cnt.sum(axis=0).max()) > pb.cap or int(cnt.sum(axis=1).max()) > pb.cap:
            return None
        g = pb.next_gen()
        in_base = cnt[:me].sum(axis=0)                   # where my run starts inside owner o's inbox
        send_base = np.concatenate([[0], np.cumsum(cnt[me])[:-1]])   # my routed order: runs by owner
        tab = np.zeros(5 * W, dtype=np.uint64)
        for o in range(W):
            off = 4 * int(in_base[o])
            tab[o] = pb.peer[o][(g, "x")] + off
            tab[W + o] = pb.peer[o][(g, "y")] + off if ys is not None else 0
            tab[2 * W + o] = pb.peer[o][(g, "v")] + off if vals is not None else 0
            tab[3 * W + o] = pb.peer[o][(g, "o")] + off if ordered else 0
            tab[4 * W + o] = int(send_base[o])
        opos = DevPtr(pb.local[(g, "p")], n) if want_pos else None     # preallocated with the inboxes
        bias = int(cnt[:me].sum())                       # global index of my first op (rank-major order)
        if n:
            lib.smatrix_b200_route_p2p(rh, ptr(xs), ptr(ys), ptr(vals), n, W, tab.ctypes.data,
                                       bias & 0xFFFFFFFF, opos.ptr if opos else None)
        dist.barrier(group=self.group)                   # every rank's runs have landed
        n_recv = int(cnt[:, me].sum())
        dp = lambda a, used: DevPtr(pb.local[(g, a)], n_recv) if used else None
        return cnt, g, dp("x", True), dp("y", ys is not None), dp("v", vals is not None), dp("o", ordered), opos

    # overlapped pieces (helper thread routes piece j+1 while piece j updates): measured slower than one
    # fused route per batch on B200 (7.4 vs 6.7 ms per 2^26 ops at N=2), so off unless asked for
    PIPELINE_MIN = int(os.environ.get("SMX_PIPELINE_MIN", 1 << 62))
    PIPELINE_PIECE = int(os.environ.get("SMX_PIPELINE_PIECE", 1 << 25))

    def _nmax(self, n: int) -> int:
        t = torch.tensor([n], dtype=torch.int64, device=self.dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX, group=self.group)
        return int(t)

    def _routed(self, xs, ys, vals, ordered=False, nmax=None):
        """-> (rx, ry, rv, rord, n_recv) through peer memory when possible, else NCCL all-to-all."""
        for attempt in (0, 1):
            if attempt == 0 and (self._peers is None or not self._use_p2p):
                continue      # nothing set up yet: size the inboxes first (collective decision below)
            if attempt == 1 and not self._ensure_peers(nmax if nmax is not None else self._nmax(xs.numel())):
                break
            # with inboxes in place the count matrix itself tells every rank whether they suffice,
            # so the steady state needs no extra all-reduce
            r = self._route_p2p(xs, ys, vals, ordered=ordered)
            if r is not None:
                _, _, rx, ry, rv, rord, _ = r
                return rx, ry, rv, rord, rx.n
        _, _, rx, ry, rv, _, rord = self._route(xs, ys, vals, ordered=ordered)
        return rx, ry, rv, rord, rx.numel()

    def _write(self, op: int, xs, ys, vals, ordered: bool):
        n = xs.numel()
        piped = self.PIPELINE_MIN < (1 << 40)
        # every rank must take the same decisions (the exchanges are collective)
        nmax = self._nmax(n) if (piped or self._peers is None) else None
        if ordered:
            rx, ry, rv, rord, n_recv = self._routed(xs, ys, vals, ordered=True, nmax=nmax)
            if n_recv:
                p = lambda t: None if t is None else (t.ptr if isinstance(t, DevPtr) else t.data_ptr())
                self._lib.smatrix_b200_apply_ordered(self.local._handle(), op, p(rx), p(ry), p(rv), p(rord),
                                                     n_recv)
            return
        apply = (self.local.incr_batch, self.local.decr_batch)[op]
        pieces = max(1, -(-nmax // self.PIPELINE_PIECE)) if (piped and nmax >= self.PIPELINE_MIN) else 1
        if pieces == 1:
            rx, ry, rv, _, n_recv = self._routed(xs, ys, vals, nmax=nmax)
            if n_recv:
                apply(rx, ry, rv)
            return
        # route piece j+1 (router handle + NCCL, helper thread) while piece j updates the shard
        import concurrent.futures as cf
        if self._pool is None:
            self._pool = cf.ThreadPoolExecutor(max_workers=1)
        cut = lambda t, j: None if t is None else t[j * n // pieces:(j + 1) * n // pieces]

        piece_max = -(-nmax // pieces) + 1
        self._ensure_peers(piece_max)      # size the inboxes once, before the helper thread starts

        def route(j):
            if self._cuda:
                torch.cuda.set_device(self.dev)
            return self._routed(cut(xs, j), cut(ys, j), cut(vals, j), nmax=piece_max)
        fut = self._pool.submit(route, 0)
        for j in range(pieces):
            rx, ry, rv, _, n_recv = fut.result()
            if j + 1 < pieces:
                fut = self._pool.submit(route, j + 1)
            if n_recv:
                apply(rx, ry, rv)

    # ------------------------------------------------------------------ collective batch API
    # xs / ys / vals: this rank's slice, as device tensors (zero-copy) or host arrays (staged first)
    def _is_dev(self, t) -> bool:
        return torch.is_tensor(t) and t.device == self.dev

    def _write_any(self, op: int, xs, ys, vals, ordered: bool):
        if self._is_dev(xs) or ordered:
            # ordered batches keep the documented global order (rank-major over whole slices): one piece
            self._write(op, self._up("x", xs), self._up("y", ys), self._up("v", vals), ordered)
            return
        for _, _, (px, py, pv) in self._host_pieces([xs, ys, vals], len(xs)):
            self._write(op, px, py, pv, False)

    def incr_batch(self, xs, ys, vals=None, ordered: bool = True):
        self._write_any(0, xs, ys, vals, ordered)

    def decr_batch(self, xs, ys, vals=None, ordered: bool = True):
        self._write_any(1, xs, ys, vals, ordered)

    def set_batch(self, xs, ys, vals=None):
        # last writer in GLOBAL input order wins
        self._write(2, self._up("x", xs), self._up("y", ys), self._up("v", vals), True)

    def _read_p2p(self, fn, xs, ys, out):
        """Queries travel through the inboxes; every owner's read kernel writes its answers straight
        into the requester's answer buffer (peer memory), which the requester then gathers into
        input order."""
        import time as _t
        dbg = os.environ.get("SMX_ROUTE_DEBUG") in ("1", "2")
        t0 = _t.perf_counter()
        r = self._route_p2p(xs, ys, None, want_pos=True)
        if r is None:
            return None
        cnt, g, rx, ry, _, _, opos = r
        t1 = _t.perf_counter()
        pb, me = self._peers, self.rank
        starts = np.concatenate([[0], np.cumsum(cnt[:, me])])   # sender s's run inside my inbox
        for i in range(self.world):               # one launch per sender's run, staggered: at any moment
            s_ = (me + i) % self.world            # the ranks answer DIFFERENT requesters (a shift
            c, off = int(cnt[s_][me]), int(starts[s_])   # permutation), not all the same one
            if c:
                dst = DevPtr(pb.peer[s_][(g, "b")] + 4 * int(cnt[s_][:me].sum()), c)
                qx = DevPtr(rx.ptr + 4 * off, c)
                if ry is not None:
                    fn(qx, DevPtr(ry.ptr + 4 * off, c), out=dst)
                else:
                    fn(qx, out=dst)
        t2 = _t.perf_counter()
        dist.barrier(group=self.group)             # all answers have landed
        t3 = _t.perf_counter()
        n = xs.numel()
        if out is None:
            out = self._buf(n)
        if n:
            self._lib.smatrix_b200_gather(self.router._handle(), out.data_ptr(), pb.local[(g, "b")],
                                          opos.ptr, n)
        if dbg and (self.rank == 0 or os.environ.get("SMX_ROUTE_DEBUG") == "2"):
            print(f"[route] rank {self.rank} read n={n}: route {1e3*(t1-t0):.2f} ms, owners' kernels {1e3*(t2-t1):.2f}, "
                  f"barrier {1e3*(t3-t2):.2f}, gather {1e3*(_t.perf_counter()-t3):.2f}", file=__import__("sys").stderr, flush=True)
        return out

    def _read_routed(self, fn, xs, ys, out):
        for attempt in (0, 1):
            if attempt == 0 and (self._peers is None or not self._use_p2p):
                continue
            if attempt == 1 and not self._ensure_peers(self._nmax(xs.numel())):
                break
            r = self._read_p2p(fn, xs, ys, out)
            if r is not None:
                return r
        return None

    def get_batch(self, xs, ys, out=None):
        if not self._is_dev(xs):      # host arrays: piece-wise, uploads and downloads overlap the look-ups
            n = len(xs)
            host_out = out if out is not None else np.empty(n, dtype=np.uint32)
            h = torch.from_numpy(host_out.view(np.int32)) if isinstance(host_out, np.ndarray) else host_out
            down_ev = [None, None]          # answers go down on their own stream: PCIe is full duplex
            for k, (lo, hi, (px, py)) in enumerate(self._host_pieces([xs, ys], n)):
                if down_ev[k & 1] is not None:
                    down_ev[k & 1].synchronize()           # the answer buffer of piece k-2 is free again
                ans = self.get_batch(px, py, self._slot(f"hp_ans{k & 1}", hi - lo))
                if self._cuda:
                    if self._side_down is None:
                        self._side_down = torch.cuda.Stream(self.dev)
                    with torch.cuda.stream(self._side_down):
                        h[lo:hi].copy_(ans, non_blocking=True)     # `ans` is complete: the library call is synchronous
                        down_ev[k & 1] = torch.cuda.Event()
                        down_ev[k & 1].record(self._side_down)
                else:
                    h[lo:hi].copy_(ans)
            if self._cuda:
                self._side_down.synchronize()
            return host_out
        r = self._read_routed(self.local.get_batch, xs, ys, out)
        if r is not None:
            return r
        send, recv, rx, ry, _, opos, _ = self._route(xs, ys, None, want_pos=True)
        ans = self.local.get_batch(rx, ry) if rx.numel() else self._buf(0)
        self._sync_torch()
        back = self._a2a(ans, recv, send)           # answers travel the reverse way
        return self._unpermute(back, opos, out)

    def _unpermute(self, back, opos, out=None):
        """out[i] = back[opos[i]] — answers arrive in routed order."""
        if out is None:
            out = self._buf(opos.numel())
        self._sync_torch()
        self._lib.smatrix_b200_gather(self.router._handle(), out.data_ptr(), back.data_ptr(),
                                      opos.data_ptr(), opos.numel())
        return out

    def rowlen_batch(self, xs):
        r = self._read_routed(self.local.rowlen_batch, xs, None, None)
        if r is not None:
            return r
        send, recv, rx, _, _, opos, _ = self._route(xs, None, None, want_pos=True)
        ans = self.local.rowlen_batch(rx) if rx.numel() else self._buf(0)
        self._sync_torch()
        back = self._a2a(ans, recv, send)
        return self._unpermute(back, opos)

    def getrow_batch(self, xs):
        """-> (offsets[n+1] uint64, pairs[total, 2] uint32) host arrays for THIS rank's rows xs, rows
        in input order, pairs in the owners' table order (src/smatrix.c:189-210 with full buffers).
        Row ids travel to their owners, each owner answers with the CSR of its run, and the asking
        rank puts the rows back into input order."""
        xs_np = xs.cpu().numpy().view(np.uint32) if torch.is_tensor(xs) else np.ascontiguousarray(xs, dtype=np.uint32)
        n = len(xs_np)
        dx = self._up("gx", torch.from_numpy(xs_np.view(np.int32).copy())) if n else self._buf(0)
        send, recv, rx, _, _, opos, _ = self._route(dx, None, None, want_pos=True)
        if rx.numel():
            off_l, pairs_l = self.local.getrow_batch(rx.cpu().numpy().view(np.uint32))
        else:
            off_l, pairs_l = np.zeros(1, np.uint64), np.zeros((0, 2), np.uint32)
        cnt_l = np.diff(off_l).astype(np.int64)                       # pairs per received row, inbox order
        self._sync_torch()
        back_cnt = self._a2a(torch.from_numpy(cnt_l.astype(np.int32)).to(self.dev), recv, send)
        edges = np.concatenate([[0], np.cumsum(recv)]).astype(np.int64)
        pairs_to = [int(cnt_l[edges[r]:edges[r + 1]].sum()) for r in range(self.world)]   # pairs I send to rank r
        cnt_back = back_cnt.cpu().numpy().astype(np.int64)            # pairs per row, MY routed order
        sedges = np.concatenate([[0], np.cumsum(send)]).astype(np.int64)
        pairs_from = [int(cnt_back[sedges[r]:sedges[r + 1]].sum()) for r in range(self.world)]
        flat = torch.from_numpy(pairs_l.reshape(-1).view(np.int32).copy()).to(self.dev)
        got = torch.empty(2 * sum(pairs_from), dtype=torch.int32, device=self.dev)
        dist.all_to_all_single(got, flat, output_split_sizes=[2 * c for c in pairs_from],
                               input_split_sizes=[2 * c for c in pairs_to], group=self.group)
        got = got.cpu().numpy().view(np.uint32).reshape(-1, 2)
        pos = opos.cpu().numpy().astype(np.int64) if n else np.zeros(0, np.int64)
        roff = np.concatenate([[0], np.cumsum(cnt_back)]).astype(np.int64)   # CSR in routed order
        lens = cnt_back[pos] if n else np.zeros(0, np.int64)
        offsets = np.concatenate([[0], np.cumsum(lens)]).astype(np.uint64)
        total = int(offsets[-1])
        take = np.repeat(roff[pos] - offsets[:-1].astype(np.int64), lens) + np.arange(total, dtype=np.int64)
        return offsets, got[take] if total else np.zeros((0, 2), np.uint32)

    # ------------------------------------------------------------------ local controls
    def stat(self, name):
        return self.local.stat(name)

    _LOCAL_CONTROLS = frozenset((
        "timer_start", "timer_stop_ms", "set_kernel_timing", "set_get_slices", "sync", "gen_c2_ops", "gen_c2_queries",
        "gen_c3_ops", "gen_c3_queries", "gen_c4_lens", "gen_c4_ops", "probe_random_read",
        "probe_random_atomic", "dev_alloc", "dev_free", "memcpy", "device", "stream"))

    def __getattr__(self, name):
        # only controls of the local shard are forwarded; a data-path call that is not sharded here
        # (cf_neighbors_batch, *_batch_out, single ops) must not silently run on one shard
        if name in TorchShardedSparseMatrix._LOCAL_CONTROLS:
            return getattr(self.local, name)
        raise AttributeError(f"{type(self).__name__} has no sharded '{name}' (it would only see this rank's rows)")

    def close(self):
        if self._pool is not None:
            self._pool.shutdown(wait=True)
            self._pool = None
        self._bufs: dict[str, torch.Tensor] = {}
        self._gen = 0
        if self._peers is not None:
            self._peers.close()
            self._peers = None
        self.router.close()
        self.local.close()


# ====================================================================================================
# the product: the C router (include/smatrix_shard.h) behind the same collective API
# ====================================================================================================
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
                 _lib_path: str | None = None, arena_gib: float | None = None):
        from . import binding
        self._lib = binding.load(_lib_path)
        self.rank, self.world = rank, world
        self._name = name or default_name()
        if arena_gib is not None:
            self._h = self._lib.smatrix_b200_shard_open_arena(self._name.encode(), rank, world, int(device),
                                                              int(arena_gib * (1 << 30)))
        else:
            self._h = self._lib.smatrix_b200_shard_open(self._name.encode(), rank, world, int(device))
        if not self._h:
            raise RuntimeError("smatrix_b200_shard_open failed (no CUDA device or no peer access)")
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

    def barrier(self):
        self._lib.smatrix_b200_shard_barrier(self._handle())

    def sum(self, v: int) -> int:
        return int(self._lib.smatrix_b200_shard_sum(self._handle(), int(v)))

    def max(self, v: int) -> int:
        return int(self._lib.smatrix_b200_shard_max(self._handle(), int(v)))

    def stat(self, name):
        return self.local.stat(name)

    def __getattr__(self, name):
        if name in TorchShardedSparseMatrix._LOCAL_CONTROLS:
            return getattr(self.local, name)
        raise AttributeError(f"{type(self).__name__} has no sharded '{name}' (it would only see this rank's rows)")

    def close(self):
        if self._h:
            self.local._h = None          # borrowed: the router closes it
            self._lib.smatrix_b200_shard_close(self._h)
            self._h = None

    def __del__(self):
        pass   # closing is collective: never from a finalizer


def open_sharded(rank: int, world: int, device: int = 0, group=None, name: str | None = None,
                 arena_gib: float | None = None):
    """The C router when it can be set up, else (every rank alike — shard_open agrees on the outcome
    before anyone returns) the torch.distributed fallback.  $SMX_ROUTER=torch forces the fallback."""
    if os.environ.get("SMX_ROUTER", "c") != "torch":
        try:
            return ShardedSparseMatrix(rank, world, device, name=name, arena_gib=arena_gib)
        except RuntimeError as e:
            print(f"[smatrix sharded] rank {rank}: C router unavailable ({e}); using torch.distributed", flush=True)
    if arena_gib:      # the fallback's tables read the arena size from the environment at open
        os.environ["SMATRIX_ARENA_GIB"] = str(int(arena_gib))
    try:
        return TorchShardedSparseMatrix(rank, world, device, group=group)
    finally:
        if arena_gib:
            os.environ.pop("SMATRIX_ARENA_GIB", None)
