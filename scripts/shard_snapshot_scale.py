"""File mode of the sharded matrix at scale: a config-2-shaped table per GPU (13 M rows x 256 columns, 2 G ops,
times `fraction`), saved to one .smx file in `dir` (every rank writes its part) and reloaded (every rank reads a
share of the directory and expands its row blocks on its GPU), at N = 1 (sharded world 1, and the single-GPU
SparseMatrix on the same table beside it) and at every N = 2, 4, 8 the box has.  Ranks are threads of this
process.  One JSON line per run.  usage: shard_snapshot_scale.py [fraction per GPU] [dir]"""
import json, os, subprocess, sys, threading, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from libsmatrix_b200 import SparseMatrix
from libsmatrix_b200.sharded import ShardedSparseMatrix

frac = float(sys.argv[1]) if len(sys.argv) > 1 else 0.25
where = sys.argv[2] if len(sys.argv) > 2 else "/dev/shm"
rows_per, ops_per, B = int(13_000_000 * frac), int(2_000_000_000 * frac), 1 << 26
arena = (max(4, int(56 * frac) + 2)) << 30
path = os.path.join(where, "smx_shard_snapshot_scale.smx")
ngpu = torch.cuda.device_count()
smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                     capture_output=True, text=True).stdout.strip().splitlines()
KEYS = ("rows", "nnz", "value_sum")


def build(m, dev, rank, world):
    """ops [rank * ops_per, (rank + 1) * ops_per) of one C2 stream over world * rows_per rows (order-free incr)"""
    xs = torch.empty(B, dtype=torch.int32, device=dev)
    ys = torch.empty(B, dtype=torch.int32, device=dev)
    for first in range(rank * ops_per, (rank + 1) * ops_per, B):
        cnt = min(B, (rank + 1) * ops_per - first)
        m.gen_c2_ops(2, first, cnt, world * rows_per, 256, xs.data_ptr(), ys.data_ptr())
        torch.cuda.synchronize(dev)
        if isinstance(m, ShardedSparseMatrix):
            m.incr_batch(xs[:cnt], ys[:cnt], None, ordered=False)
        else:
            m.incr_batch(xs[:cnt], ys[:cnt], None)


def sharded(world):
    if os.path.exists(path):
        os.remove(path)
    name, out = f"smx_scale_{os.getpid()}_{world}", {}

    def rank_main(r):
        dev = torch.device("cuda", r)
        torch.cuda.set_device(dev)
        m = ShardedSparseMatrix(r, world, r, name=name, arena_gib=arena / (1 << 30), fname=path)
        build(m, dev, r, world)
        before = [m.sum(m.stat(k)) % 2**64 for k in KEYS]
        m.barrier(); t0 = time.perf_counter()
        assert m.snapshot() == 0
        m.barrier(); save_s = time.perf_counter() - t0
        m.close()                                   # (writes the same table again, untimed)
        t0 = time.perf_counter()
        m2 = ShardedSparseMatrix(r, world, r, name=name + "_re", arena_gib=arena / (1 << 30), fname=path)
        m2.barrier(); load_s = time.perf_counter() - t0
        after = [m2.sum(m2.stat(k)) % 2**64 for k in KEYS]
        if r == 0:
            out.update(save_s=save_s, load_s=load_s, before=before, after=after)
        m2.close()
    ts = [threading.Thread(target=rank_main, args=(r,)) for r in range(world)]
    [t.start() for t in ts]; [t.join() for t in ts]
    size = os.path.getsize(path)
    os.remove(path)
    return size, out


def line(kind, world, size, save_s, load_s, before, after):
    print(json.dumps({"kind": kind, "gpus": world, "fraction_per_gpu": frac, "rows_per_gpu": rows_per,
                      "ops_per_gpu": ops_per, "dir": where, "file_bytes": size,
                      "save_s": round(save_s, 3), "save_gbs": round(size / save_s / 1e9, 3),
                      "load_s": round(load_s, 3), "load_gbs": round(size / load_s / 1e9, 3),
                      "before": before, "after": after, "identical": before == after, "gpu": smi[:world]}), flush=True)


# N = 1 on one GPU: the single-GPU handle, then sharded world 1
if os.path.exists(path):
    os.remove(path)
m = SparseMatrix(file_path=path, device=0, arena_gib=arena / (1 << 30))
build(m, torch.device("cuda", 0), 0, 1)
before = [m.stat(k) for k in KEYS]
t0 = time.perf_counter(); m.close(); save_s = time.perf_counter() - t0
size = os.path.getsize(path)
t0 = time.perf_counter(); m2 = SparseMatrix(file_path=path, device=0, arena_gib=arena / (1 << 30)); load_s = time.perf_counter() - t0
line("single", 1, size, save_s, load_s, before, [m2.stat(k) for k in KEYS])
m2.close()
os.remove(path)
for world in [1] + [w for w in (2, 4, 8) if w <= ngpu]:
    size, o = sharded(world)
    line("sharded", world, size, o["save_s"], o["load_s"], o["before"], o["after"])
