"""Top-k recommender queries (smatrix_cf_topk_batch, smatrix_b200_topk_segments, the sharded call): bit-exact
against the CPU checker's ranking (tests/topk_suite.py).  CPU: three simulator builds of tests/hostsim/ — the
1-lane one, the 32-lane one, and one with the size classes and the digit width lowered so that rows of a few
thousand pairs take the multi-pass select.  GPU (`-m gpu`): the same at full size, device and torch in/out, and
the config-3 table at bench size."""
import os
import subprocess
import sys
import threading

import numpy as np
import pytest

import topk_suite as ts
from libsmatrix_b200 import SparseMatrix
from libsmatrix_b200.matrix import DevPtr

HERE = os.path.dirname(os.path.abspath(__file__))
U32 = np.uint32
LOWERED = ["-DTOPK_WARP_MAX=16u", "-DTOPK_BLOCK_MAX=1024u", "-DTOPK_DIGIT_BITS=4u"]
CLASSES = {"sim": (256, 4096), "sim32": (256, 4096), "sim_lowered": (16, 1024)}


@pytest.fixture(scope="module")
def sim():
    from hostsim import build as hb
    return hb.build()


@pytest.fixture(scope="module")
def sim32():
    from hostsim import build as hb
    return hb.build(defines=["-DSMX_SIM_WARP32"], suffix="_warp32")


@pytest.fixture(scope="module")
def sim_lowered():
    from hostsim import build as hb
    return hb.build(defines=LOWERED, suffix="_topk_lowered")


def _pieces(make, monkeypatch, pairs):
    def f():
        monkeypatch.setenv("SMATRIX_TOPK_PAIRS", str(pairs))
        try:
            return make()
        finally:
            monkeypatch.delenv("SMATRIX_TOPK_PAIRS")
    return f


def _check_stats(st, ks):
    assert st["tie_big"] == len(ks) and st["straddle_big"] == len(ks)   # the big class ran where intended ...
    assert st["tie_passes"] > 8 * len(ks)                              # ... into the id digits (> 8 passes each)
    assert st["straddle_passes"] > 8 * (len(ks) - 1)                   # k = 1 ends inside the score digits
    assert st["small_big"] == 0 and st["small_passes"] == 0            # ... and not where it was not
    assert st["allocs_again"] == 0


# ------------------------------------------------------------------ CPU: the simulator builds
@pytest.mark.parametrize("lib", ["sim", "sim32", "sim_lowered"])
def test_boundaries_sim(lib, request, monkeypatch):
    so = request.getfixturevalue(lib)
    warp_max, block_max = CLASSES[lib]
    make = lambda: SparseMatrix(_lib_path=so)
    ks = (1, 7, 32, 1024)
    st = ts.scenario_boundaries(make, warp_max, block_max, ks, big_times=3,
                                make_pieces=_pieces(make, monkeypatch, block_max // 2 + 7))
    _check_stats(st, ks)


def test_d2h_sim(sim):
    ts.scenario_d2h(lambda: SparseMatrix(_lib_path=sim))


def test_k_is_checked(sim):
    m = SparseMatrix(_lib_path=sim)
    for k in (0, 1025, -3, 2.0, True):
        with pytest.raises(ValueError):
            m.cf_topk_batch(np.arange(3, dtype=U32), k)
    m.close()
    code = ("import ctypes, numpy as np\n"
            "from libsmatrix_b200 import binding\n"
            f"lib = binding.load({sim!r}); h = lib.smatrix_open(None)\n"
            "c = np.zeros(1, np.uint32); i = np.zeros(1025, np.uint32); s = np.zeros(1025)\n"
            "lib.smatrix_cf_topk_batch(h, c.ctypes.data, 1, 1025, c.ctypes.data, i.ctypes.data, s.ctypes.data)\n")
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True,
                       cwd=os.path.dirname(HERE), timeout=120)
    assert r.returncode != 0 and "libsmatrix error: cf_topk_batch: k = 1025" in r.stdout, (r.returncode, r.stdout)


def _dev(m, a):
    a = np.ascontiguousarray(a)
    p = m.dev_alloc(max(a.nbytes, 8))
    m.memcpy(p, a.ctypes.data, a.nbytes)
    return p


def _down(m, p, like):
    out = np.empty_like(like)
    m.memcpy(out.ctypes.data, p, out.nbytes)
    return out


def test_device_arrays_sim(sim):
    """Device items and outputs; and smatrix_b200_topk_segments on a CSR of its own: negative scores, infinities,
    ties, segments of every class."""
    ms, ref, rows = ts.build(lambda: SparseMatrix(_lib_path=sim), 256, 4096, ks=(7,), big_times=2)
    m = ms[0]
    q = ts.query_items(rows, np.random.default_rng(5))
    k, n = 7, len(q)
    c0, i0, s0 = np.zeros(n, U32), np.zeros((n, k), U32), np.zeros((n, k))
    ptrs = [_dev(m, q), _dev(m, c0), _dev(m, i0), _dev(m, s0)]
    m._lib.smatrix_cf_topk_batch(m._handle(), ptrs[0], n, k, *ptrs[1:])
    got = (_down(m, ptrs[1], c0), _down(m, ptrs[2], i0), _down(m, ptrs[3], s0))
    ts.assert_same(got, ts.oracle_topk(ref, q, k), "device arrays")
    ts.assert_same(m.cf_topk_batch(q, k), got, "host arrays")
    rng = np.random.default_rng(11)
    lens = np.array([0, 1, 5, 255, 256, 257, 3000, 4096, 4097, 9000, 20000])
    off = np.concatenate([[0], np.cumsum(lens)]).astype(np.uint64)
    ids = np.concatenate([rng.permutation(2 * L + 1)[:L] for L in lens]).astype(U32)
    sc = rng.choice(np.array([-np.inf, -3.5, -1e-300, 0.0, 1e-300, 0.25, 0.5, 7.0, np.inf]), int(off[-1]))
    for k in (1, 32, 1024):
        out = (np.zeros(len(lens), U32), np.zeros((len(lens), k), U32), np.zeros((len(lens), k)))
        dp = [_dev(m, a) for a in (off, ids, sc) + out]
        m._lib.smatrix_b200_topk_segments(m._handle(), len(lens), dp[0], dp[1], dp[2], k, dp[3], dp[4], dp[5])
        ts.assert_same(tuple(_down(m, p, a) for p, a in zip(dp[3:], out)), ts.rank(off, ids, sc, k), f"segments k={k}")
        for p in dp:
            m.dev_free(p)
    for p in ptrs:
        m.dev_free(p)
    m.close(); ref.close()


def _rank_main(sim, name, rank, world, errors, device_arrays, rows, want):
    try:
        from libsmatrix_b200.sharded import ShardedSparseMatrix
        m = ShardedSparseMatrix(rank, world, 0, name=name, _lib_path=sim)
        xs, ys, vs = (np.concatenate([o[i] for o in rows.ops]).astype(U32) for i in range(3))
        sl = lambda a: a[rank * len(a) // world:(rank + 1) * len(a) // world]
        m.set_batch(sl(xs), sl(ys), sl(vs))
        for k, (q, w) in want.items():
            mine = q[rank::world]
            wanted = tuple(a[rank::world] for a in w)
            if device_arrays:
                n = len(mine)
                outs = (np.zeros(n, U32), np.zeros((n, k), U32), np.zeros((n, k)))
                loc = m.local
                ptrs = [_dev(loc, mine)] + [_dev(loc, a) for a in outs]
                m._lib.smatrix_b200_shard_cf_topk_batch(m._handle(), ptrs[0], n, k, *ptrs[1:])
                got = tuple(_down(loc, p, a) for p, a in zip(ptrs[1:], outs))
                for p in ptrs:
                    loc.dev_free(p)
            else:
                got = m.cf_topk_batch(mine, k)
            ts.assert_same(got, wanted, f"rank {rank} k={k}")
        m.close()
    except BaseException as e:                           # noqa: BLE001 - reported by the main thread
        import traceback
        errors.append(f"rank {rank}: {e!r}\n{traceback.format_exc()}")


@pytest.mark.parametrize("device_arrays", [False, True], ids=["host-arrays", "device-arrays"])
@pytest.mark.parametrize("world", [2, 3])
def test_router_ranks_as_threads(sim, world, device_arrays, monkeypatch):
    """The C router with ranks as threads equals the single-table answer (a rank whose items are all absent, or
    that asks for none, still takes part)."""
    monkeypatch.setenv("SMATRIX_DIR_LOG2", "8")
    monkeypatch.setenv("SMATRIX_SHARD_INBOX", "1024")
    monkeypatch.setenv("SMATRIX_SHARD_TIMEOUT", "60")
    rows = ts.Rows(seed=4, pool=12000)
    for L in (0, 1, 6, 7, 8, 200, 300, 4097, 9000):
        rows.add(L)
    rows.add(5000, "tie")
    ref_m = SparseMatrix(_lib_path=sim)
    ref = ts.checker()
    rows.apply([ref_m], ref)
    q = ts.query_items(rows, np.random.default_rng(6))
    want = {}
    for k in (7, 1024):
        w = ref_m.cf_topk_batch(q, k)
        ts.assert_same(w, ts.oracle_topk(ref, q, k), f"single table k={k}")
        want[k] = (q, w)
    want[3] = (ts.ABSENT.copy(), ts.oracle_topk(ref, ts.ABSENT, 3))   # with world 3 one rank asks for nothing
    ref_m.close(); ref.close()
    name = f"smxtopk_{os.getpid()}_{world}_{int(device_arrays)}"
    errors: list = []
    th = [threading.Thread(target=_rank_main, args=(sim, name, r, world, errors, device_arrays, rows, want))
          for r in range(world)]
    for t in th:
        t.start()
    for t in th:
        t.join(timeout=280)
    assert not errors, "\n".join(errors)
    assert not any(t.is_alive() for t in th), "a rank hangs"


# ------------------------------------------------------------------ GPU: full size
@pytest.mark.gpu
def test_boundaries(monkeypatch):
    make = lambda: SparseMatrix()
    ks = (1, 7, 32, 1024)
    st = ts.scenario_boundaries(make, 256, 4096, ks, big_times=40, make_pieces=_pieces(make, monkeypatch, 20000))
    _check_stats(st, ks)


@pytest.mark.gpu
def test_d2h():
    ts.scenario_d2h(lambda: SparseMatrix())


@pytest.mark.gpu
def test_torch_in_out():
    import torch
    ms, ref, rows = ts.build(lambda: SparseMatrix(), 256, 4096, ks=(32,), big_times=8)
    m = ms[0]
    q = ts.query_items(rows, np.random.default_rng(8))
    dq = torch.from_numpy(q.view(np.int32)).cuda()
    for k in (32, 100):
        c, i, s = m.cf_topk_batch(dq, k)
        assert c.is_cuda and i.is_cuda and s.is_cuda and i.shape == (len(q), k) and s.dtype == torch.float64
        got = (c.cpu().numpy().view(U32), i.cpu().numpy().view(U32), s.cpu().numpy())
        ts.assert_same(got, ts.oracle_topk(ref, q, k), f"torch k={k}")
        a0, h0 = m.stat("allocs"), m.stat("d2h_bytes")
        m.cf_topk_batch(dq, k)                                   # again: no cudaMalloc, no answers through the host
        assert m.stat("allocs") == a0 and m.stat("d2h_bytes") - h0 < 4096
    m.close(); ref.close()


def rank_torch(m, items, k, chunk=2000):
    """The baseline: cf_neighbors_batch into device tensors, ranked with torch sorts (chunks of items)."""
    import torch
    n = len(items)
    counts = torch.empty(n, dtype=torch.int32, device="cuda")
    ids = torch.empty((n, k), dtype=torch.int32, device="cuda")
    scores = torch.empty((n, k), dtype=torch.float64, device="cuda")
    for lo in range(0, n, chunk):
        it = torch.from_numpy(np.ascontiguousarray(items[lo:lo + chunk]).view(np.int32)).cuda()
        c, i, s = rank_segments(m, it, k)
        counts[lo:lo + len(it)], ids[lo:lo + len(it)], scores[lo:lo + len(it)] = c, i, s
    return counts, ids, scores


def rank_segments(m, items, k):
    import torch
    n = items.numel()
    off = torch.empty(n + 1, dtype=torch.int64, device="cuda")
    total = int(m._lib.smatrix_cf_neighbors_batch(m._handle(), items.data_ptr(), n, off.data_ptr(), None, None, 0))
    nb = torch.empty(max(total, 1), dtype=torch.int32, device="cuda")
    sc = torch.empty(max(total, 1), dtype=torch.float64, device="cuda")
    m._lib.smatrix_cf_neighbors_batch(m._handle(), items.data_ptr(), n, off.data_ptr(), nb.data_ptr(), sc.data_ptr(),
                                      max(total, 1))
    nb, sc = nb[:total], sc[:total]
    lens = off[1:] - off[:-1]
    seg = torch.repeat_interleave(torch.arange(n, device="cuda"), lens)
    o = torch.argsort(nb.to(torch.int64) & 0xFFFFFFFF, stable=True)
    o = o[torch.argsort(-sc[o], stable=True)]
    o = o[torch.argsort(seg[o], stable=True)]
    s_seg = seg[o]
    pos = torch.arange(total, device="cuda") - off[s_seg]
    keep = pos < k
    ids = torch.full((n, k), -1, dtype=torch.int32, device="cuda")
    out = torch.full((n, k), -1.0, dtype=torch.float64, device="cuda")
    ids[s_seg[keep], pos[keep]] = nb[o][keep]
    out[s_seg[keep], pos[keep]] = sc[o][keep]
    return torch.clamp(lens, max=k).to(torch.int32), ids, out


def build_c3(m, baskets=1 << 24, items=4_000_000, seed=3):
    """The config-3 table at bench size, built on the device (Zipf(1.1) baskets of 8, all pairs + totals)."""
    import torch
    from libsmatrix_b200.workloads import zipf_thresholds
    thr = torch.from_numpy(zipf_thresholds(items, 1.1).view(np.int64)).cuda()
    B = 1 << 26
    xs = torch.empty(B, dtype=torch.int32, device="cuda")
    ys = torch.empty(B, dtype=torch.int32, device="cuda")
    for first in range(0, baskets * 64, B):
        n = min(B, baskets * 64 - first)
        m.gen_c3_ops(seed, first, n, thr.data_ptr(), items, xs.data_ptr(), ys.data_ptr())
        m.incr_batch(xs[:n], ys[:n], None)


@pytest.mark.gpu
def test_config3_table():
    import torch
    m = SparseMatrix(arena_gib=40)
    build_c3(m)
    assert m.rowlen(1) > 10**6
    rng = np.random.default_rng(12)
    sets = {"hottest": np.arange(1, 10_001, dtype=U32),
            "random": rng.integers(1, 4_000_001, 100_000).astype(U32)}
    for name, items in sets.items():
        for k in (10, 100):
            want = rank_torch(m, items, k)
            got = m.cf_topk_batch(torch.from_numpy(items.view(np.int32)).cuda(), k)
            for g, w, what in zip(got, want, ("counts", "ids", "scores")):
                if what == "scores":
                    g, w = g.view(torch.int64), w.view(torch.int64)
                assert torch.equal(g, w), f"{name} k={k}: {what} differ"
            if name == "hottest":
                assert m.stat("topk_big") > 0
    m.close()


@pytest.mark.gpu
def test_world2():
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    env = dict(os.environ, WORLD_SIZE="2", SMX_TOPK_NAME=f"smxtopk_{os.getpid()}")
    procs = [subprocess.Popen([sys.executable, os.path.join(HERE, "topk_gpu_worker.py")],
                              env=dict(env, RANK=str(r)), stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
             for r in range(2)]
    outs = [p.communicate(timeout=600)[0] for p in procs]
    for r, (p, o) in enumerate(zip(procs, outs)):
        assert p.returncode == 0, f"rank {r} failed:\n{o[-3000:]}"
        assert f"rank {r} ok" in o
