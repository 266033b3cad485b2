"""Matrix enumeration (smatrix_list_rows, smatrix_getrow_sorted_batch, smatrix_b200_sort_rows and the sharded calls)
against the CPU checker's file and rows (tests/export_suite.py).  CPU: three simulator builds of tests/hostsim/ — the
1-lane one, the 32-lane one, and one with the size classes lowered so that rows of a few thousand pairs take the
radix class.  GPU (`-m gpu`): the same at full size, torch in and out, a config-3 hot item, and the config-4 table
at bench size exported page by page."""
import os
import subprocess
import sys
import threading

import numpy as np
import pytest

import export_suite as es
from libsmatrix_b200 import SparseMatrix

HERE = os.path.dirname(os.path.abspath(__file__))
U32 = np.uint32
LOWERED = ["-DTOPK_WARP_MAX=16u", "-DTOPK_BLOCK_MAX=1024u"]
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
    return hb.build(defines=LOWERED, suffix="_rec_lowered")


def _pieces(make, monkeypatch, pairs):
    def f():
        monkeypatch.setenv("SMATRIX_TOPK_PAIRS", str(pairs))
        try:
            return make()
        finally:
            monkeypatch.delenv("SMATRIX_TOPK_PAIRS")
    return f


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
def test_shapes_sim(lib, request, monkeypatch):
    so = request.getfixturevalue(lib)
    warp_max, block_max = CLASSES[lib]
    make = lambda: SparseMatrix(_lib_path=so)
    st = es.scenario_shapes(make, warp_max, block_max, 10**5,
                            make_pieces=_pieces(make, monkeypatch, 2 * block_max + 400))   # groups of 2 rows
    assert st["n_big"] >= 6 and st["sort_big_pieces"] == st["n_big"]


@pytest.mark.parametrize("lib", ["sim", "sim_lowered"])
def test_follows_writes_sim(lib, request, monkeypatch, tmp_path):
    so = request.getfixturevalue(lib)
    monkeypatch.setenv("SMATRIX_DIR_LOG2", "8")
    es.scenario_follows_writes(lambda fname=None: SparseMatrix(fname, _lib_path=so), tmp_path)


@pytest.mark.parametrize("lib", ["sim", "sim32", "sim_lowered"])
def test_sort_rows_sim(lib, request):
    so = request.getfixturevalue(lib)
    m = SparseMatrix(_lib_path=so)
    es.scenario_sort_rows(m, *CLASSES[lib], _dev, _down)
    m.close()


def test_device_arrays_sim(sim):
    """Device keys, offsets and pairs through the C calls, against the host-array answers."""
    m, ref = SparseMatrix(_lib_path=sim), es.port()
    st = es.Stream([m], ref)
    es.build_shapes(st, 256, 4096, 6000)
    keys = m.rows()
    n = len(keys)
    d_keys = m.dev_alloc(4 * n)
    assert m._lib.smatrix_list_rows(m._handle(), 0, d_keys, n) == n
    assert (_down(m, d_keys, keys) == keys).all()
    assert m._lib.smatrix_list_rows(m._handle(), 2, d_keys, 3) == int((keys >= 2).sum())
    assert (_down(m, d_keys, keys[:3]) == keys[keys >= 2][:3]).all()
    off, pairs = m.getrow_sorted_batch(keys)
    d_off, d_pairs = m.dev_alloc(8 * (n + 1)), m.dev_alloc(pairs.nbytes)
    d_keys = _dev(m, keys)
    total = m._lib.smatrix_getrow_sorted_batch(m._handle(), d_keys, n, d_off, d_pairs, len(pairs))
    assert total == len(pairs)
    assert (_down(m, d_off, off) == off).all() and (_down(m, d_pairs, pairs) == pairs).all()
    es.assert_rows_equal(off, pairs, ref, keys, "device arrays")
    a0 = m.stat("allocs")
    m._lib.smatrix_getrow_sorted_batch(m._handle(), d_keys, n, d_off, d_pairs, len(pairs))
    m._lib.smatrix_list_rows(m._handle(), 0, d_keys, n)
    assert m.stat("allocs") == a0
    for p in (d_keys, d_off, d_pairs):
        m.dev_free(p)
    m.close(); ref.close()


def test_checked_in_python(sim):
    m = SparseMatrix(_lib_path=sim)
    m.set(3, 4, 5)
    for bad in (-1, 1 << 32, 2.0, True, "0", None):
        with pytest.raises(ValueError):
            m.rows(bad)
        with pytest.raises(ValueError):
            m.iter_rows(bad)
    for bad in (0, -2, 1.5, True, "3"):
        with pytest.raises(ValueError):
            m.rows(0, bad)
        with pytest.raises(ValueError):
            m.iter_rows(0, bad)
    assert (m.rows(np.uint32(3), np.int64(1)) == [3]).all() and m.rows(4).shape == (0,)
    off, pairs = m.getrow_sorted_batch([])
    assert off.tolist() == [0] and pairs.shape == (0, 2)
    m.close()


def test_checked_in_c(sim):
    code = ("from libsmatrix_b200 import binding\n"
            f"lib = binding.load({sim!r}); h = lib.smatrix_open(None)\n"
            "lib.smatrix_getrow_sorted_batch(h, None, 0xFFFFFFFF, None, None, 0)\n")
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True,
                       cwd=os.path.dirname(HERE), timeout=120)
    assert r.returncode != 0 and "libsmatrix error: getrow_sorted_batch: too many rows in one call" in r.stdout, \
        (r.returncode, r.stdout)


class Recorder:
    """A stand-in handle that records the stream's batches, for the ranks to replay."""

    def __init__(self):
        self.batches = []

    def __getattr__(self, name):
        return lambda xs, ys, vs: self.batches.append((name[:-len("_batch")], xs, ys, vs))


def replay(m, batches, rank, world):
    """every batch as a collective one, each rank passing its slice"""
    sl = lambda a: a[rank * len(a) // world:(rank + 1) * len(a) // world]
    for op, xs, ys, vs in batches:
        getattr(m, op + "_batch")(sl(xs), sl(ys), sl(vs))


def _rank_main(sim, name, rank, world, errors, device_arrays, batches, want_keys, mine, ref_rows):
    try:
        from libsmatrix_b200.sharded import ShardedSparseMatrix
        m = ShardedSparseMatrix(rank, world, 0, name=name, _lib_path=sim)
        replay(m, batches, rank, world)
        assert (m.rows() == want_keys).all(), "rows()"
        for per in (1, 7, 1000):
            pages, start = [], 0
            while True:
                p = m.rows(start, per)
                pages.append(p)
                if len(p) < per or p[-1] == es.TOP:
                    break
                start = int(p[-1]) + 1
            assert (np.concatenate(pages) == want_keys).all(), f"pages of {per}"
        assert (m.rows(es.TOP) == want_keys[-1:]).all() and (m.rows(2, 3) == want_keys[want_keys >= 2][:3]).all()
        if device_arrays:
            loc, n = m.local, len(mine)
            d_keys = loc.dev_alloc(4 * len(want_keys))
            assert m._lib.smatrix_b200_shard_list_rows(m._handle(), 0, d_keys, len(want_keys)) == len(want_keys)
            assert (_down(loc, d_keys, want_keys) == want_keys).all()
            d_xs = _dev(loc, mine)
            total = m._lib.smatrix_b200_shard_getrow_sorted_batch(m._handle(), d_xs, n, None, None, 0)
            d_off, d_pairs = loc.dev_alloc(8 * (n + 1)), loc.dev_alloc(8 * max(total, 1))
            assert m._lib.smatrix_b200_shard_getrow_sorted_batch(m._handle(), d_xs, n, d_off, d_pairs,
                                                                 max(total, 1)) == total
            off = _down(loc, d_off, np.zeros(n + 1, np.uint64))
            pairs = _down(loc, d_pairs, np.zeros((total, 2), U32))
            for p in (d_keys, d_xs, d_off, d_pairs):
                loc.dev_free(p)
        else:
            off, pairs = m.getrow_sorted_batch(mine)
        assert len(off) == len(mine) + 1
        for i, x in enumerate(mine):
            got = pairs[off[i]:off[i + 1]]
            assert got.shape == ref_rows[int(x)].shape and (got == ref_rows[int(x)]).all(), f"row {int(x)}"
        m.close()
    except BaseException as e:                           # noqa: BLE001 - reported by the main thread
        import traceback
        errors.append(f"rank {rank}: {e!r}\n{traceback.format_exc()}")


@pytest.mark.parametrize("device_arrays", [False, True], ids=["host-arrays", "device-arrays"])
@pytest.mark.parametrize("world", [2, 3])
def test_router_ranks_as_threads(sim, world, device_arrays, monkeypatch):
    """The C router with ranks as threads: rows() is the single handle's on every rank, paged too, and every rank's
    sorted rows equal the checker's; the last rank passes no rows."""
    monkeypatch.setenv("SMATRIX_DIR_LOG2", "8")
    monkeypatch.setenv("SMATRIX_SHARD_INBOX", "1024")
    monkeypatch.setenv("SMATRIX_SHARD_TIMEOUT", "60")
    single, ref, rec = SparseMatrix(_lib_path=sim), es.port(), Recorder()
    st = es.Stream([single, rec], ref)
    es.build_shapes(st, 256, 4096, 6000)
    want_keys = es.oracle_rows(ref)
    assert (single.rows() == want_keys).all()
    single.close()
    ref_rows = {int(x): es.want_pairs(ref, x) for x in want_keys}
    ref.close()
    mine = [want_keys[r::world - 1] for r in range(world - 1)] + [np.zeros(0, U32)]
    name = f"smxexp_{os.getpid()}_{world}_{int(device_arrays)}"
    errors: list = []
    th = [threading.Thread(target=_rank_main, args=(sim, name, r, world, errors, device_arrays, rec.batches, want_keys,
                                                    mine[r], ref_rows))
          for r in range(world)]
    for x in th:
        x.start()
    for x in th:
        x.join(timeout=280)
    assert not errors, "\n".join(errors)
    assert not any(x.is_alive() for x in th), "a rank hangs"


# ------------------------------------------------------------------ GPU: full size
@pytest.mark.gpu
def test_shapes(monkeypatch):
    make = lambda: SparseMatrix()
    st = es.scenario_shapes(make, 256, 4096, 10**6, make_pieces=_pieces(make, monkeypatch, 2 * 4096 + 400))
    assert st["n_big"] >= 6 and st["sort_big_pieces"] == st["n_big"]


@pytest.mark.gpu
def test_follows_writes(monkeypatch, tmp_path):
    monkeypatch.setenv("SMATRIX_DIR_LOG2", "8")
    es.scenario_follows_writes(lambda fname=None: SparseMatrix(fname), tmp_path, big=20000)


@pytest.mark.gpu
def test_sort_rows():
    m = SparseMatrix()
    es.scenario_sort_rows(m, 256, 4096, _dev, _down)
    m.close()


@pytest.mark.gpu
def test_torch_in_out():
    import torch
    m, ref = SparseMatrix(), es.port()
    st = es.Stream([m], ref)
    es.build_shapes(st, 256, 4096, 20000)
    keys = m.rows()
    d_keys = m.rows(device=True)
    assert d_keys.is_cuda and d_keys.dtype == torch.int32
    assert (d_keys.cpu().numpy().view(U32) == keys).all()
    off, pairs = m.getrow_sorted_batch(d_keys)
    assert off.is_cuda and pairs.is_cuda and off.dtype == torch.int64 and pairs.shape[1] == 2
    es.assert_rows_equal(off.cpu().numpy(), pairs.cpu().numpy(), ref, keys, "torch")
    a0, h0 = m.stat("allocs"), m.stat("d2h_bytes")
    m.rows(device=True); m.getrow_sorted_batch(d_keys)          # again: no cudaMalloc, nothing through the host
    assert m.stat("allocs") == a0 and m.stat("d2h_bytes") - h0 < 8192
    pages = list(m.iter_rows(0, 7, device=True))
    assert (torch.cat([k for k, _, _ in pages]).cpu().numpy().view(U32) == keys).all()
    for k, o, p in pages:
        es.assert_rows_equal(o.cpu().numpy(), p.cpu().numpy(), ref, k.cpu().numpy().view(U32), "torch pages")
    m.close(); ref.close()


@pytest.mark.gpu
def test_config3_hot_item():
    """The config-3 table at bench size: the hottest items' rows (item 1 holds over 10^6 pairs) sorted on the device
    equal the unsorted rows sorted on the host."""
    from test_cf_topk import build_c3
    m = SparseMatrix(arena_gib=40)
    build_c3(m)
    items = np.arange(1, 2001, dtype=U32)
    assert m.rowlen(1) > 10**6
    b0 = m.stat("sort_big")
    off, pairs = m.getrow_sorted_batch(items)
    assert m.stat("sort_big") > b0
    uoff, upairs = m.getrow_batch(items)
    assert (off == uoff).all()
    for i in range(len(items)):
        seg, useg = pairs[off[i]:off[i + 1]], upairs[uoff[i]:uoff[i + 1]]
        assert (seg == useg[np.argsort(useg[:, 0], kind="stable")]).all(), int(items[i])
    m.close()


def build_c4(m, R=13_000_000, kmax=1_000_000, seed=5):
    """The config-4 table at bench size (bench.py run_c4), built on the device."""
    import torch
    from libsmatrix_b200.workloads import zipf_thresholds
    d_thr = torch.from_numpy(zipf_thresholds(kmax, 1.7).view(np.int64)).cuda()
    lens = torch.empty(R, dtype=torch.int32, device="cuda")
    m.gen_c4_lens(seed, 0, R, d_thr.data_ptr(), kmax, lens.data_ptr())
    m.sync()
    offs = torch.zeros(R + 1, dtype=torch.int64, device="cuda")
    torch.cumsum(lens.to(torch.int64), 0, out=offs[1:])
    nnz = int(offs[-1].item())
    B = 1 << 26
    bx, by, bv = (torch.empty(B, dtype=torch.int32, device="cuda") for _ in range(3))
    for first in range(0, nnz, B):
        cnt = min(B, nnz - first)
        m.gen_c4_ops(seed, first, cnt, offs.data_ptr(), R, bx.data_ptr(), by.data_ptr(), bv.data_ptr())
        m.incr_batch(bx[:cnt], by[:cnt], bv[:cnt])
    return nnz


@pytest.mark.gpu
def test_config4_export():
    """The config-4 table at bench size, exported page by page on the device, against invariants the export does not
    compute itself: rows, nnz and value sum of the table's own stats, strictly ascending columns, and 10^4 sampled rows
    equal to the unsorted getrow_batch sorted on the host."""
    import torch
    m = SparseMatrix(arena_gib=48)
    nnz = build_c4(m)
    assert m.stat("nnz") == nnz
    rows, value_sum = m.stat("rows"), m.stat("value_sum")
    n_rows = n_pairs = vsum = 0
    last = -1
    rng = np.random.default_rng(4)
    sample = []
    for keys, off, pairs in m.iter_rows(0, 1 << 21, device=True):
        k64 = keys.to(torch.int64) & 0xFFFFFFFF
        assert int(k64[0]) > last and bool((k64[1:] > k64[:-1]).all())
        last = int(k64[-1])
        n_rows += keys.numel()
        n_pairs += pairs.shape[0]
        assert int(off[-1]) == pairs.shape[0]
        vsum += int((pairs[:, 1].to(torch.int64) & 0xFFFFFFFF).sum())
        cols = pairs[:, 0].to(torch.int64) & 0xFFFFFFFF
        seg = torch.repeat_interleave(torch.arange(keys.numel(), device="cuda"), off[1:] - off[:-1])
        same = seg[1:] == seg[:-1]
        assert bool((cols[1:][same] > cols[:-1][same]).all()), "columns not strictly ascending"
        pick = rng.choice(keys.numel(), min(keys.numel(), 2000), replace=False)   # >= 5 pages of 2^21 rows
        for i in pick[:10_000 - len(sample)].tolist():
            sample.append((int(k64[i]), pairs[int(off[i]):int(off[i + 1])].cpu().numpy().view(U32)))
        del keys, off, pairs, cols, seg, same
    assert n_rows == rows and n_pairs == nnz
    assert vsum % (1 << 64) == value_sum
    assert len(sample) == 10_000
    xs = np.array([x for x, _ in sample], U32)
    uoff, upairs = m.getrow_batch(xs)
    for i, (x, seg) in enumerate(sample):
        useg = upairs[uoff[i]:uoff[i + 1]]
        assert (seg == useg[np.argsort(useg[:, 0], kind="stable")]).all(), x
    m.close()


@pytest.mark.gpu
def test_world2():
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    env = dict(os.environ, WORLD_SIZE="2", SMX_EXPORT_NAME=f"smxexp_{os.getpid()}")
    procs = [subprocess.Popen([sys.executable, os.path.join(HERE, "export_gpu_worker.py")],
                              env=dict(env, RANK=str(r)), stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
             for r in range(2)]
    outs = [p.communicate(timeout=600)[0] for p in procs]
    for r, (p, o) in enumerate(zip(procs, outs)):
        assert p.returncode == 0, f"rank {r} failed:\n{o[-3000:]}"
        assert f"rank {r} ok" in o
