"""Multi-GPU parity (BASELINE config 5 shape at test scale): rows hash-partitioned over the GPUs of
one box, ops routed to their owners by the C router (peer-memory stores from the partition kernel,
shared-memory rendezvous) — every rank updating only its own shard, bit-exact against the reference
fed the whole stream, incl. getrow, batch_out and CF across ranks; "c-sliced" runs the same with every
shard on its slice-ordered paths.  Needs >= 2 GPUs."""
import os
import subprocess
import sys

import pytest

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))


def _ngpu():
    try:
        import torch
        return torch.cuda.device_count()
    except Exception:
        return 0


KINDS = ["c", "c-sliced"]


@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("world", [2, 4, 8])
def test_row_sharding(world, kind):
    if _ngpu() < world:
        pytest.skip(f"needs {world} GPUs")
    port = 29600 + world + 10 * KINDS.index(kind)
    env = dict(os.environ, MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port),
               WORLD_SIZE=str(world), SMX_SHARD_KIND=kind)
    if kind == "c-sliced":      # the C router with every owner ordering its inbox by directory slice: writes (256 slices
        # for the order-free batch without column 0) and the runs of queries it answers for the asking ranks
        env.update(SMATRIX_PARTITION_MIN="4096", SMATRIX_SLICE_LOG2="8", SMATRIX_GET_SLICE_MIN="1024")
    procs = [subprocess.Popen([sys.executable, os.path.join(HERE, "sharded_gpu_worker.py")],
                              env=dict(env, RANK=str(r), LOCAL_RANK=str(r)), stdout=subprocess.PIPE,
                              stderr=subprocess.STDOUT, text=True) for r in range(world)]
    outs = [p.communicate(timeout=600)[0] for p in procs]
    for r, (p, o) in enumerate(zip(procs, outs)):
        assert p.returncode == 0, f"rank {r} failed:\n{o[-3000:]}"
        assert f"rank {r} ok" in o
