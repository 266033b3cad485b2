"""Worker for tests/test_gpu_sharded.py: one rank (= one GPU) of an NCCL group driving the
C router (include/smatrix_shard.h) on the real CUDA library."""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from libsmatrix_b200.sharded import ShardedSparseMatrix  # noqa: E402
from oracle import cpu  # noqa: E402

U32 = np.uint32


def main():
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    kind = os.environ.get("SMX_SHARD_KIND", "c")
    sliced = kind == "c-sliced"                       # shards forced onto their slice-ordered paths
    m = ShardedSparseMatrix(rank, world, rank)
    ref = cpu.CpuMatrix("reference" if cpu.have_reference() else "port")
    rng = np.random.default_rng(321)                  # the same global stream on every rank
    n = 400_000
    xs = rng.integers(0, 20000, n).astype(U32) * U32(2654435761)
    ys = rng.integers(0, 120, n).astype(U32)          # includes column 0: order matters for rowlen
    vs = rng.integers(0, 1000, n).astype(U32)
    t = lambda a: torch.from_numpy(a.view(np.int32).copy()).to(dev)
    sl = lambda k: slice(rank * k // world, (rank + 1) * k // world)
    ref.apply("incr", xs, ys, vs)
    m.incr_batch(xs[sl(n)], ys[sl(n)], vs[sl(n)])                          # ordered (default); host arrays are staged
    gx = rng.integers(0, 300, 50000).astype(U32) * U32(2654435761)
    gy = rng.integers(1, 40, 50000).astype(U32)
    gv = rng.integers(1, 2**32, 50000, dtype=np.uint64).astype(U32)
    ref.apply("set", gx, gy, gv)
    m.set_batch(t(gx[sl(50000)]), t(gy[sl(50000)]), t(gv[sl(50000)]))      # last writer in GLOBAL order
    nz = ys != 0
    ref.apply("incr", xs[nz], ys[nz], np.ones(int(nz.sum()), U32))
    k = int(nz.sum())
    m.incr_batch(t(xs[nz][sl(k)]), t(ys[nz][sl(k)]), None, ordered=False)  # order-free stream
    allx = np.concatenate([xs, gx]); ally = np.concatenate([ys, gy])
    qx = np.concatenate([allx[rank::7], rng.integers(0, 2**32, 1000, dtype=np.uint64).astype(U32)])
    qy = np.concatenate([ally[rank::7], rng.integers(0, 130, 1000).astype(U32)])
    got = m.get_batch(t(qx), t(qy)).cpu().numpy().view(U32)
    assert (got == ref.get_many(qx, qy)).all(), f"rank {rank}: sharded get mismatch"
    assert (m.get_batch(qx, qy) == got).all(), f"rank {rank}: host-array get differs from device-array get"
    if sliced:
        assert m.stat("sliced_gets") > 0 and m.stat("wide_chunks") > 0, (m.stat("sliced_gets"), m.stat("wide_chunks"))
    rows = np.unique(allx)[rank::world]
    got = m.rowlen_batch(t(rows)).cpu().numpy().view(U32)
    assert (got == ref.rowlen_many(rows)).all(), f"rank {rank}: sharded rowlen mismatch"
    # getrow across ranks (src/smatrix.c:189-210): overlapping requests, rows nobody has, an empty request
    grows = np.concatenate([np.unique(allx)[rank::3], np.array([3, 5], U32)])
    o1, p1 = m.getrow_batch(grows)
    o2, p2 = ref.getrow_many(grows)
    assert (o1 == o2).all(), f"rank {rank}: sharded getrow offsets mismatch"
    assert (cpu.sort_rows(o1, p1) == cpu.sort_rows(o2, p2)).all(), f"rank {rank}: sharded getrow pairs mismatch"
    o0, p0 = m.getrow_batch(np.zeros(0, U32))
    assert len(o0) == 1 and len(p0) == 0
    for op in ("incr", "decr", "set", "incr"):        # per-op return values across ranks (SURVEY.md 8f N1)
        bx = (rng.zipf(1.4, 60000) % 500).astype(U32) * U32(2654435761)
        by = (rng.zipf(1.3, 60000) % 9).astype(U32)
        bv = rng.integers(1, 1000, 60000).astype(U32)
        want = ref.apply(op, bx, by, bv, want_out=True)
        s6 = sl(60000)
        got = getattr(m, op + "_batch_out")(bx[s6], by[s6], bv[s6])
        assert (np.asarray(got) == want[s6]).all(), f"rank {rank}: sharded {op}_batch_out mismatch (host arrays)"
    bx = (rng.zipf(1.4, 60000) % 500).astype(U32) * U32(2654435761)
    by = (rng.zipf(1.3, 60000) % 9 + 1).astype(U32)
    want = ref.apply("incr", bx, by, np.ones(60000, U32), want_out=True)
    got = m.incr_batch_out(t(bx[sl(60000)]), t(by[sl(60000)]), None)          # device arrays, all ones
    assert (got.cpu().numpy().view(U32) == want[sl(60000)]).all(), f"rank {rank}: sharded incr_batch_out mismatch (device)"
    allx = np.concatenate([allx, bx]); ally = np.concatenate([ally, by])
    items = np.unique(allx)[rank::11][:200]           # the CF read side across ranks: bit-exact doubles
    co, cids, cscores = m.cf_neighbors_batch(items)
    o3, p3 = ref.getrow_many(items)
    assert (co == o3).all(), f"rank {rank}: cf offsets mismatch"
    for i, a in enumerate(items[:40]):
        lo, hi = int(co[i]), int(co[i + 1])
        got = dict(zip(cids[lo:hi].tolist(), cscores[lo:hi].tolist()))
        a_total, want = ref.get(int(a), 0), {}
        for b, cc in p3[lo:hi]:
            den = np.sqrt(np.float64(a_total)) * np.sqrt(np.float64(ref.get(int(b), 0) or 1))
            want[int(b)] = 0.0 if (den == 0.0 or np.float64(cc) > den) else float(np.float64(cc) / den)
        assert got == want, f"rank {rank}: cf scores of item {a}"
    tot = torch.tensor([m.stat("rows"), m.stat("nnz")], device=dev)
    dist.all_reduce(tot)
    o, p = ref.getrow_many(np.unique(allx))
    assert int(tot[0]) == len(np.unique(allx)) and int(tot[1]) == len(p)
    m.close(); ref.close()
    dist.barrier()
    dist.destroy_process_group()
    print(f"rank {rank} ok ({kind})")


if __name__ == "__main__":
    main()
