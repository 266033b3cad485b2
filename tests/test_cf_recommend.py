"""Basket recommendations (smatrix_cf_recommend_batch, smatrix_b200_basket_topk, the sharded call): bit-exact against
the CPU checker's lists summed in position order (tests/recommend_suite.py).  CPU: three simulator builds of
tests/hostsim/ — the 1-lane one, the 32-lane one, and one with the size classes lowered so that baskets of a few
thousand pairs take the global-sort class.  GPU (`-m gpu`): the same at full size, device and torch in/out, and
baskets of the config-3 stream on the config-3 table at bench size."""
import os
import subprocess
import sys
import threading

import numpy as np
import pytest

import recommend_suite as rs
import topk_suite as ts
from libsmatrix_b200 import SparseMatrix

HERE = os.path.dirname(os.path.abspath(__file__))
U32 = np.uint32
LOWERED = ["-DTOPK_WARP_MAX=16u", "-DTOPK_BLOCK_MAX=1024u"]
CLASSES = {"sim": (256, 4096), "sim32": (256, 4096), "sim_lowered": (16, 1024)}
KS = (1, 7, 32, 1024)


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
    return hb.build(defines=LOWERED, suffix="_rec_lowered")


def _pieces(make, monkeypatch, pairs):
    def f():
        monkeypatch.setenv("SMATRIX_TOPK_PAIRS", str(pairs))
        try:
            return make()
        finally:
            monkeypatch.delenv("SMATRIX_TOPK_PAIRS")
    return f


def _check_stats(st):
    assert st["n_big"] > 0
    assert st["rec_big"] == [st["n_big"]] * len(KS)                  # the global sort ran for the big baskets ...
    assert st.get("rec_big_pieces", st["rec_big"]) == st["rec_big"]  # ... in one piece or in many
    assert st["small_big"] == 0                                      # ... and not for the others
    assert st["allocs_again"] == 0


def _dev(m, a):
    a = np.ascontiguousarray(a)
    p = m.dev_alloc(max(a.nbytes, 8))
    m.memcpy(p, a.ctypes.data, a.nbytes)
    return p


def _down(m, p, like):
    out = np.empty_like(like)
    m.memcpy(out.ctypes.data, p, out.nbytes)
    return out


# ------------------------------------------------------------------ CPU: the simulator builds
@pytest.mark.parametrize("lib", ["sim", "sim32", "sim_lowered"])
def test_baskets_sim(lib, request, monkeypatch):
    so = request.getfixturevalue(lib)
    warp_max, block_max = CLASSES[lib]
    make = lambda: SparseMatrix(_lib_path=so)
    st = rs.scenario_baskets(make, warp_max, block_max, KS,
                             make_pieces=_pieces(make, monkeypatch, block_max // 2 + 7))
    _check_stats(st)


@pytest.mark.parametrize("lib", ["sim", "sim_lowered"])
def test_single_item_is_topk_sim(lib, request):
    so = request.getfixturevalue(lib)
    rs.scenario_single_vs_topk(lambda: SparseMatrix(_lib_path=so), *CLASSES[lib], KS)


def test_d2h_sim(sim):
    rs.scenario_d2h(lambda: SparseMatrix(_lib_path=sim))


def test_checked_in_python(sim):
    m = SparseMatrix(_lib_path=sim)
    off, items = np.array([0, 2, 3], np.uint64), np.arange(1, 4, dtype=U32)
    for k in (0, 1025, -3, 2.0, True):
        with pytest.raises(ValueError):
            m.cf_recommend_batch(off, items, k)
    for bad in ([], [1, 3], [0, 2, 1, 3], [0, 2], [0, 4], [[0, 3]]):
        with pytest.raises(ValueError):
            m.cf_recommend_batch(np.array(bad, np.int64), items, 5)
    c, i, s = m.cf_recommend_batch(np.zeros(1, np.uint64), np.zeros(0, U32), 5)   # no baskets
    assert c.shape == (0,) and i.shape == (0, 5) and s.shape == (0, 5)
    m.close()


@pytest.mark.parametrize("case", ["k", "offsets", "decreasing"])
def test_checked_in_c(sim, case):
    k, off = {"k": (1025, "[0, 1, 2]"), "offsets": (5, "[1, 1, 2]"), "decreasing": (5, "[0, 2, 1]")}[case]
    code = ("import numpy as np\n"
            "from libsmatrix_b200 import binding\n"
            f"lib = binding.load({sim!r}); h = lib.smatrix_open(None)\n"
            f"o = np.array({off}, np.uint64); it = np.arange(1, 3, dtype=np.uint32)\n"
            f"c = np.zeros(2, np.uint32); i = np.zeros(2 * {k}, np.uint32); s = np.zeros(2 * {k})\n"
            f"lib.smatrix_cf_recommend_batch(h, o.ctypes.data, it.ctypes.data, 2, {k}, c.ctypes.data, i.ctypes.data,"
            " s.ctypes.data)\n")
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True,
                       cwd=os.path.dirname(HERE), timeout=120)
    want = "k = 1025 is outside" if case == "k" else "malformed basket offsets"
    assert r.returncode != 0 and f"libsmatrix error: cf_recommend_batch: {want}" in r.stdout, (r.returncode, r.stdout)


def test_device_arrays_sim(sim):
    """Device offsets, items and outputs; and smatrix_b200_basket_topk on lists of its own."""
    ms, ref, t, baskets, named = rs.setup(lambda: SparseMatrix(_lib_path=sim), 256, 4096)
    m = ms[0]
    off, items = rs.flatten(baskets)
    k, n = 32, len(baskets)
    want = rs.oracle(ref, off, items, k)
    outs = (np.zeros(n, U32), np.zeros((n, k), U32), np.zeros((n, k)))
    ptrs = [_dev(m, off), _dev(m, items)] + [_dev(m, a) for a in outs]
    m._lib.smatrix_cf_recommend_batch(m._handle(), ptrs[0], ptrs[1], n, k, *ptrs[2:])
    got = tuple(_down(m, p, a) for p, a in zip(ptrs[2:], outs))
    ts.assert_same(got, want, "device arrays")
    a0 = m.stat("allocs")
    m._lib.smatrix_cf_recommend_batch(m._handle(), ptrs[0], ptrs[1], n, k, *ptrs[2:])
    assert m.stat("allocs") == a0
    ts.assert_same(m.cf_recommend_batch(off, items, k), got, "host arrays")
    # lists that are not a table's: negative and tiny scores, repeated ids at one position, ids equal to items
    rng = np.random.default_rng(11)
    b_off = np.array([0, 0, 1, 3, 3, 7, 9], np.uint64)
    b_items = rng.integers(1, 40, int(b_off[-1])).astype(U32)
    lens = rng.integers(0, 3000, len(b_items))
    lens[2] = 0
    l_off = np.concatenate([[0], np.cumsum(lens)]).astype(np.uint64)
    l_ids = rng.integers(0, 60, int(l_off[-1])).astype(U32)
    l_sc = rng.choice(np.array([-3.5, -1e-300, 0.0, 1e-300, 1e-17, 0.25, 0.5, 7.0, 1e16]), int(l_off[-1]))
    for k in (1, 32, 1024):
        outs = (np.zeros(len(b_off) - 1, U32), np.zeros((len(b_off) - 1, k), U32), np.zeros((len(b_off) - 1, k)))
        dp = [_dev(m, a) for a in (b_off, b_items, l_off, l_ids, l_sc) + outs]
        m._lib.smatrix_b200_basket_topk(m._handle(), len(b_off) - 1, *dp[:5], k, *dp[5:])
        ts.assert_same(tuple(_down(m, p, a) for p, a in zip(dp[5:], outs)),
                       rs.recommend_from_lists(b_off, b_items, l_off, l_ids, l_sc, k), f"basket_topk k={k}")
        for p in dp:
            m.dev_free(p)
    for p in ptrs:
        m.dev_free(p)
    m.close(); ref.close()


def _rank_main(sim, name, rank, world, errors, device_arrays, ops, mine, k):
    try:
        from libsmatrix_b200.sharded import ShardedSparseMatrix
        m = ShardedSparseMatrix(rank, world, 0, name=name, _lib_path=sim)
        xs, ys, vs = ops
        sl = lambda a: a[rank * len(a) // world:(rank + 1) * len(a) // world]
        m.set_batch(sl(xs), sl(ys), sl(vs))
        (off, items), want = mine
        if device_arrays:
            n = len(off) - 1
            outs = (np.zeros(n, U32), np.zeros((n, k), U32), np.zeros((n, k)))
            loc = m.local
            ptrs = [_dev(loc, off), _dev(loc, items)] + [_dev(loc, a) for a in outs]
            m._lib.smatrix_b200_shard_cf_recommend_batch(m._handle(), ptrs[0], ptrs[1], n, k, *ptrs[2:])
            got = tuple(_down(loc, p, a) for p, a in zip(ptrs[2:], outs))
            for p in ptrs:
                loc.dev_free(p)
        else:
            got = m.cf_recommend_batch(off, items, k)
        ts.assert_same(got, want, f"rank {rank}")
        m.close()
    except BaseException as e:                           # noqa: BLE001 - reported by the main thread
        import traceback
        errors.append(f"rank {rank}: {e!r}\n{traceback.format_exc()}")


@pytest.mark.parametrize("device_arrays", [False, True], ids=["host-arrays", "device-arrays"])
@pytest.mark.parametrize("world", [2, 3])
def test_router_ranks_as_threads(sim, world, device_arrays, monkeypatch):
    """The C router with ranks as threads equals the oracle of the whole table; the last rank passes no baskets."""
    monkeypatch.setenv("SMATRIX_DIR_LOG2", "8")
    monkeypatch.setenv("SMATRIX_SHARD_INBOX", "1024")
    monkeypatch.setenv("SMATRIX_SHARD_TIMEOUT", "60")
    ms, ref, t, baskets, named = rs.setup(lambda: SparseMatrix(_lib_path=sim), 256, 4096)
    ms[0].close()
    k = 7
    parts = [baskets[r::world - 1] for r in range(world - 1)] + [[]]
    mine = []
    for part in parts:
        off, items = rs.flatten(part)
        mine.append(((off, items), rs.oracle(ref, off, items, k)))
    ref.close()
    name = f"smxrec_{os.getpid()}_{world}_{int(device_arrays)}"
    errors: list = []
    th = [threading.Thread(target=_rank_main, args=(sim, name, r, world, errors, device_arrays, t.ops(), mine[r], k))
          for r in range(world)]
    for x in th:
        x.start()
    for x in th:
        x.join(timeout=280)
    assert not errors, "\n".join(errors)
    assert not any(x.is_alive() for x in th), "a rank hangs"


# ------------------------------------------------------------------ GPU: full size
@pytest.mark.gpu
def test_baskets(monkeypatch):
    make = lambda: SparseMatrix()
    st = rs.scenario_baskets(make, 256, 4096, KS, make_pieces=_pieces(make, monkeypatch, 3000))
    _check_stats(st)


@pytest.mark.gpu
def test_single_item_is_topk():
    rs.scenario_single_vs_topk(lambda: SparseMatrix(), 256, 4096, KS)


@pytest.mark.gpu
def test_d2h():
    rs.scenario_d2h(lambda: SparseMatrix())


@pytest.mark.gpu
def test_torch_in_out():
    import torch
    ms, ref, t, baskets, named = rs.setup(lambda: SparseMatrix(), 256, 4096)
    m = ms[0]
    off, items = rs.flatten(baskets)
    d_off = torch.from_numpy(off.astype(np.int64)).cuda()
    d_items = torch.from_numpy(items.view(np.int32)).cuda()
    with pytest.raises(ValueError):
        m.cf_recommend_batch(off, d_items, 5)                    # mixed placement
    for k in (32, 100):
        c, i, s = m.cf_recommend_batch(d_off, d_items, k)
        assert c.is_cuda and i.is_cuda and s.is_cuda and i.shape == (len(baskets), k) and s.dtype == torch.float64
        got = (c.cpu().numpy().view(U32), i.cpu().numpy().view(U32), s.cpu().numpy())
        ts.assert_same(got, rs.oracle(ref, off, items, k), f"torch k={k}")
        a0, h0 = m.stat("allocs"), m.stat("d2h_bytes")
        m.cf_recommend_batch(d_off, d_items, k)                  # again: no cudaMalloc, no answers through the host
        assert m.stat("allocs") == a0 and m.stat("d2h_bytes") - h0 < 4096
    m.close(); ref.close()


def stream_baskets(m, first_basket, n, seed=3, items=4_000_000):
    """Baskets of the config-3 stream: basket i = the 8 Zipf items of build ops 64 i .. 64 i + 63."""
    import torch
    from libsmatrix_b200.workloads import zipf_thresholds
    thr = torch.from_numpy(zipf_thresholds(items, 1.1).view(np.int64)).cuda()
    xs = torch.empty(64 * n, dtype=torch.int32, device="cuda")
    ys = torch.empty(64 * n, dtype=torch.int32, device="cuda")
    m.gen_c3_ops(seed, 64 * first_basket, 64 * n, thr.data_ptr(), items, xs.data_ptr(), ys.data_ptr())
    m.sync()
    return xs.view(n, 8, 8)[:, :, 0].reshape(-1).cpu().numpy().view(U32)


@pytest.mark.gpu
def test_config3_stream_baskets():
    """64 baskets sampled from the config-3 stream on the bench-size table (item 1 is in some), bit-exact against
    the oracle fed by the library's own cf_neighbors_batch lists."""
    from test_cf_topk import build_c3
    m = SparseMatrix(arena_gib=40)
    build_c3(m)
    rng = np.random.default_rng(21)
    picks = np.sort(rng.choice(1 << 24, 64, replace=False))
    items = np.concatenate([stream_baskets(m, int(b), 1) for b in picks])
    off = np.arange(0, 8 * 64 + 1, 8, dtype=np.uint64)
    assert (items == 1).any(), "no sampled basket holds the hottest item"
    lists = m.cf_neighbors_batch(items)
    for k in (10, 100):
        b0 = m.stat("rec_big")
        got = m.cf_recommend_batch(off, items, k)
        ts.assert_same(got, rs.recommend_from_lists(off, items, *lists, k), f"config-3 k={k}")
        assert m.stat("rec_big") > b0
    m.close()


@pytest.mark.gpu
def test_world2():
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    env = dict(os.environ, WORLD_SIZE="2", SMX_REC_NAME=f"smxrec_{os.getpid()}")
    procs = [subprocess.Popen([sys.executable, os.path.join(HERE, "recommend_gpu_worker.py")],
                              env=dict(env, RANK=str(r)), stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
             for r in range(2)]
    outs = [p.communicate(timeout=600)[0] for p in procs]
    for r, (p, o) in enumerate(zip(procs, outs)):
        assert p.returncode == 0, f"rank {r} failed:\n{o[-3000:]}"
        assert f"rank {r} ok" in o
