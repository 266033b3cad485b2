"""The C router (csrc/smx_router.c, include/smatrix_shard.h) on the CPU: ranks are THREADS of this
process driving the serial simulator library (tests/hostsim) — the same code path a C / JNI host uses
to drive several GPUs from one process (peer pointers, no IPC).  Checks the host logic of the router:
rendezvous, count exchange, inbox layout, staged host pieces, reverse route of answers, the getrow
offset round trip — bit-exact against the CPU oracle fed the whole collective batch."""
import ctypes as C
import os
import threading

import numpy as np
import pytest

from libsmatrix_b200.sharded import ShardedSparseMatrix
from oracle import cpu

U32 = np.uint32


@pytest.fixture(scope="module")
def sim():
    from hostsim import build as hb
    return hb.build()


class DevArrays:
    """uint32 arrays in the simulator's "device" memory (so the router takes its device-pointer path)."""

    def __init__(self, m):
        self.m, self.ptrs = m, []

    def up(self, a):
        a = np.ascontiguousarray(a, dtype=U32)
        p = self.m.local.dev_alloc(max(a.nbytes, 4))
        self.m.local.memcpy(p, a.ctypes.data, a.nbytes)
        self.ptrs.append(p)
        from libsmatrix_b200.matrix import DevPtr
        return DevPtr(p, len(a))

    def down(self, d):
        out = np.empty(d.n, dtype=U32)
        self.m.local.memcpy(out.ctypes.data, d.ptr, out.nbytes)
        return out

    def free(self):
        for p in self.ptrs:
            self.m.local.dev_free(p)


def _rank_main(sim, name, rank, world, errors, device_arrays):
    try:
        m = ShardedSparseMatrix(rank, world, 0, name=name, _lib_path=sim)
        ref = cpu.CpuMatrix("port")
        rng = np.random.default_rng(99)                  # the same global stream on every rank
        n = 30000
        xs = rng.integers(0, 2500, n).astype(U32) * U32(2654435761)
        ys = rng.integers(0, 50, n).astype(U32)          # includes column 0: order matters for rowlen
        vs = rng.integers(0, 1000, n).astype(U32)
        sl = lambda k: slice(rank * k // world, (rank + 1) * k // world)
        dev = DevArrays(m)
        put = (lambda a: dev.up(a)) if device_arrays else (lambda a: a)
        ref.apply("incr", xs, ys, vs)
        m.incr_batch(put(xs[sl(n)]), put(ys[sl(n)]), put(vs[sl(n)]))                 # ordered (default)
        gx = rng.integers(0, 60, 5000).astype(U32) * U32(2654435761)
        gy = rng.integers(1, 20, 5000).astype(U32)
        gv = rng.integers(1, 2**32, 5000, dtype=np.uint64).astype(U32)
        ref.apply("set", gx, gy, gv)                                                 # last writer in GLOBAL order
        m.set_batch(put(gx[sl(5000)]), put(gy[sl(5000)]), put(gv[sl(5000)]))
        nz = ys != 0
        k = int(nz.sum())
        ref.apply("incr", xs[nz], ys[nz], np.ones(k, U32))
        m.incr_batch(put(xs[nz][sl(k)]), put(ys[nz][sl(k)]), None, ordered=False)    # order-free, all ones
        ref.apply("decr", xs[nz][::2], ys[nz][::2], vs[nz][::2])
        k2 = len(xs[nz][::2])
        m.decr_batch(put(xs[nz][::2][sl(k2)]), put(ys[nz][::2][sl(k2)]), put(vs[nz][::2][sl(k2)]), ordered=False)
        if rank == world - 1:                            # an empty slice is a valid contribution
            m.incr_batch(np.zeros(0, U32), np.zeros(0, U32), None, ordered=False)
        else:
            ex = np.full(7, 12345, U32); ey = np.arange(1, 8, dtype=U32)
            m.incr_batch(ex, ey, None, ordered=False)
        for r in range(world - 1):
            ref.apply("incr", np.full(7, 12345, U32), np.arange(1, 8, dtype=U32), np.ones(7, U32))
        allx = np.concatenate([xs, gx, [12345]]).astype(U32); ally = np.concatenate([ys, gy, [3]]).astype(U32)
        qx = np.concatenate([allx[rank::5], rng.integers(0, 2**32, 200, dtype=np.uint64).astype(U32)])
        qy = np.concatenate([ally[rank::5], rng.integers(0, 60, 200).astype(U32)])
        if device_arrays:
            dq = dev.up(np.zeros(len(qx), U32))
            m._lib.smatrix_b200_shard_get_batch(m._handle(), dev.up(qx).ptr, dev.up(qy).ptr, len(qx), dq.ptr)
            got = dev.down(dq)
        else:
            got = m.get_batch(qx, qy)
        assert (got == ref.get_many(qx, qy)).all(), f"rank {rank}: sharded get mismatch"
        if os.environ.get("SMATRIX_GET_SLICE_MIN") == "64":      # the owners answered in directory-slice order
            assert m.stat("sliced_gets") > 0 and m.stat("wide_chunks") > 0, (m.stat("sliced_gets"), m.stat("wide_chunks"))
        rows = np.unique(allx)[rank::world] if rank else np.unique(allx)           # overlapping requests are fine
        rows = np.concatenate([rows, np.array([7, 8, 9], U32)])                      # rows nobody has
        assert (m.rowlen_batch(rows) == ref.rowlen_many(rows)).all(), f"rank {rank}: sharded rowlen mismatch"
        o1, p1 = m.getrow_batch(rows)
        o2, p2 = ref.getrow_many(rows)
        assert (o1 == o2).all(), f"rank {rank}: sharded getrow offsets mismatch"
        assert (cpu.sort_rows(o1, p1) == cpu.sort_rows(o2, p2)).all(), f"rank {rank}: sharded getrow pairs mismatch"
        o0, p0 = m.getrow_batch(np.zeros(0, U32))                                    # empty request (collective)
        assert len(o0) == 1 and len(p0) == 0
        owned = sum(1 for x in np.unique(allx) if m._lib.smatrix_b200_owner(int(x), world) == rank)
        assert m.stat("rows") == owned, f"rank {rank}: the shard holds {m.stat('rows')} rows, it owns {owned}"
        rows_total, nnz_total = m.sum(m.stat("rows")), m.sum(m.stat("nnz"))
        assert rows_total == len(np.unique(allx)), (rows_total, len(np.unique(allx)))
        assert nnz_total == len(ref.getrow_many(np.unique(allx))[1])
        # the CF read side across ranks (examples/cf_recommender.c:50-86): bit-exact doubles
        items = np.concatenate([np.unique(allx)[rank::7][:60], np.array([7], U32)])
        co, cids, cscores = m.cf_neighbors_batch(items)
        o3, p3 = ref.getrow_many(items)
        assert (co == o3).all(), f"rank {rank}: cf offsets mismatch"
        for i, a in enumerate(items):
            lo, hi = int(co[i]), int(co[i + 1])
            got = dict(zip(cids[lo:hi].tolist(), cscores[lo:hi].tolist()))
            a_total, want = ref.get(int(a), 0), {}
            for b, cc in p3[lo:hi]:
                den = np.sqrt(np.float64(a_total)) * np.sqrt(np.float64(ref.get(int(b), 0) or 1))
                want[int(b)] = 0.0 if (den == 0.0 or np.float64(cc) > den) else float(np.float64(cc) / den)
            assert got == want, f"rank {rank}: cf scores of item {a}"
        # per-op return values across ranks (SURVEY.md 8f N1): heavy key duplication, column 0, all three ops
        for op in ("incr", "decr", "set", "incr"):
            bx = (rng.zipf(1.4, 6000) % 50).astype(U32) * U32(2654435761)
            by = (rng.zipf(1.3, 6000) % 9).astype(U32)
            bv = rng.integers(1, 1000, 6000).astype(U32)
            want = ref.apply(op, bx, by, bv, want_out=True)
            s6 = sl(6000)
            dout = dev.up(np.zeros(len(bx[s6]), U32)) if device_arrays else None
            got = getattr(m, op + "_batch_out")(put(bx[s6]), put(by[s6]), put(bv[s6]), out=dout)
            got = dev.down(got) if device_arrays else np.asarray(got)
            assert (got == want[s6]).all(), f"rank {rank}: sharded {op}_batch_out mismatch"
        with pytest.raises(AttributeError):                                          # not a sharded call: must refuse
            m.getRow
        dev.free()
        m.close(); ref.close()
    except BaseException as e:                           # noqa: BLE001 - reported by the main thread
        import traceback
        errors.append(f"rank {rank}: {e!r}\n{traceback.format_exc()}")


@pytest.fixture(scope="module")
def sim32():
    from hostsim import build as hb
    return hb.build(defines=["-DSMX_SIM_WARP32"], suffix="_warp32")


@pytest.mark.parametrize("device_arrays", [False, True], ids=["host-arrays", "device-arrays"])
@pytest.mark.parametrize("world", [2, 3, "2-sliced", "2-sliced-warp32"])
def test_c_router_ranks_as_threads(sim, sim32, world, device_arrays, monkeypatch):
    if world == "2-sliced-warp32":   # the same on the 32-lane lock-step simulator: the route's partition kernels, the
        sim, world = sim32, "2-sliced"  # gathers and the shards' kernels with their warp collectives, one fiber scheduler per rank
    if world == "2-sliced":     # the owners' shards order their inboxes by directory slice (writes: 256 slices for the
        world = 2               # order-free batches without column 0; reads: every asking rank's run of queries)
        monkeypatch.setenv("SMATRIX_PARTITION_MIN", "256")
        monkeypatch.setenv("SMATRIX_SLICE_LOG2", "3")
        monkeypatch.setenv("SMATRIX_GET_SLICE_MIN", "64")
    monkeypatch.setenv("SMATRIX_DIR_LOG2", "8")
    monkeypatch.setenv("SMATRIX_SHARD_PIECE", "4096")      # host slices are staged in several pieces ...
    monkeypatch.setenv("SMATRIX_SHARD_TAPER_MIN", "256")   # ... the last of them cut into 1/2, 1/4, 1/4
    monkeypatch.setenv("SMATRIX_SHARD_INBOX", "1024")      # the inboxes must grow on demand
    monkeypatch.setenv("SMATRIX_SHARD_TIMEOUT", "60")
    name = f"smxtest_{os.getpid()}_{world}_{int(device_arrays)}_{os.environ.get('SMATRIX_GET_SLICE_MIN', 'd')}_{int(sim is sim32)}"
    errors: list = []
    ts = [threading.Thread(target=_rank_main, args=(sim, name, r, world, errors, device_arrays)) for r in range(world)]
    for t in ts:
        t.start()
    for t in ts:
        t.join(timeout=280)
    assert not errors, "\n".join(errors)
    assert not any(t.is_alive() for t in ts), "a rank hangs"
