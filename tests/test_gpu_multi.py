"""GPU parity of the multi-GPU search path: ShardedEmbeddingStore over NCCL (one process per GPU,
row-sharded store, ONE all-gather of packed (score, index) records + merge; query-sharded all-pairs
graph with the store rotated through all-gathers) equals the unsharded search and the oracle, and
every stage runs on a non-current device.  Needs at least two visible GPUs; skipped otherwise — the gather / merge
plumbing itself is covered on CPU with gloo in tests/test_cpu_host.py."""

from __future__ import annotations

import os
import socket
import subprocess
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

_WORKER = r"""
import os, sys
import numpy as np, torch, torch.distributed as dist
sys.path.insert(0, os.environ["ISX_REPO"])
sys.path.insert(0, os.path.join(os.environ["ISX_REPO"], "tests"))
rank, world = int(os.environ["ISX_RANK"]), int(os.environ["ISX_WORLD"])
torch.cuda.set_device(rank)
dist.init_process_group("nccl", init_method=f"tcp://127.0.0.1:{os.environ['ISX_PORT']}", rank=rank, world_size=world,
                        device_id=torch.device("cuda", rank))
from imagescry_b200.search import EmbeddingStore, ShardedEmbeddingStore, shard_range
from oracle import oracle as O
from test_gpu_knn import check
rng = np.random.default_rng(0)
n, q, d = 30011, 300, 128
store = O.bf16_round(rng.standard_normal((n, d)).astype(np.float32))
store[7] = store[29000]  # a tie across shards: the lower index must win
queries = O.bf16_round(rng.standard_normal((q, d)).astype(np.float32))
queries[0] = store[7]
b, e = shard_range(n, world, rank)
sharded = ShardedEmbeddingStore(torch.from_numpy(store[b:e]).cuda(), total_rows=n)
qd = torch.from_numpy(queries).cuda()
for k in (10, 100):
    s, i = sharded.search(qd, k)   # local fused search -> ONE all-gather of packed records -> merge
    fs, fi = EmbeddingStore(torch.from_numpy(store).cuda()).search(qd, k)
    assert torch.equal(i, fi) and torch.allclose(s, fs, atol=1e-6), (rank, k)
    check(store, queries, k, s, i)   # every index mismatch justified by a sub-tolerance score gap
    assert i[0, :2].tolist() == [7, 29000]
# the gather over peer memory (finalise + scatter in one kernel, symmetric-memory barrier) and the NCCL
# all-gather of packed records give the same answer
print("gather path:", sharded.gather_path, flush=True)
os.environ["ISX_PEER_GATHER"] = "0"
nccl_sharded = ShardedEmbeddingStore(torch.from_numpy(store[b:e]).cuda(), total_rows=n)
for k in (10, 100):
    for rep in range(3):   # both parities of the peer buffers
        s1, i1 = sharded.search_raw(qd, k)
        s2, i2 = nccl_sharded.search_raw(qd, k)
        assert torch.equal(i1, i2) and torch.equal(s1, s2), (rank, k, rep)
assert nccl_sharded.gather_path == "nccl"
del os.environ["ISX_PEER_GATHER"]
# streamed host batches (H2D / D2H on a copy stream around the sharded search) == the direct search
from imagescry_b200.search import search_host_batches
host_batches = [torch.from_numpy(queries[:128]).pin_memory(), torch.from_numpy(queries[128:131]).pin_memory(),
                torch.from_numpy(queries[131:]).pin_memory()]
got = [(s.clone(), i.clone()) for s, i in search_host_batches(sharded, host_batches, 10)]
ws, wi = sharded.search_raw(qd, 10)
assert torch.equal(torch.cat([g[1] for g in got]), wi.cpu()) and torch.equal(torch.cat([g[0] for g in got]), ws.cpu()), rank
# all-pairs graph over the sharded store (config 5): queries sharded, store rotated through the
# all-gather, running lists kept in the kernel workspace == the single-GPU graph == the oracle
gn = 5003
gstore = O.bf16_round(rng.standard_normal((gn, 64)).astype(np.float32))
gstore[11] = gstore[4000]
gb, ge = shard_range(gn, world, rank)
gsh = ShardedEmbeddingStore(torch.from_numpy(gstore[gb:ge]).cuda(), total_rows=gn)
fs, fi = EmbeddingStore(torch.from_numpy(gstore).cuda()).knn_graph(10)
for budget in (2 << 30, 64 * 700 * 2 * world):   # one all-gather / several chunked steps (KNN_CONTINUE)
    gs, gi = gsh.knn_graph(10, budget_bytes=budget)
    assert torch.equal(gi, fi) and torch.allclose(gs, fs, atol=1e-6), (rank, budget, gsh._last_graph_calls)
    ls, li = gsh.knn_graph(10, gather=False, budget_bytes=budget)
    assert torch.equal(li, fi[gb:ge]) and torch.allclose(ls, fs[gb:ge], atol=1e-6), (rank, budget)
assert len(gsh._last_graph_calls) > world, gsh._last_graph_calls
check(gstore, None, 10, gs, gi, graph=True)
assert not (gi == torch.arange(gn, device=gi.device).reshape(-1, 1)).any()
assert int(gi[11, 0]) == 4000 and int(gi[4000, 0]) == 11
# every stage on THIS rank's device while another device is current (the C ABI launches on the
# current device: the wrappers must switch to the operands' device)
other = (rank + 1) % world
mine = torch.device("cuda", rank)
from imagescry_b200.image.transforms import preprocess_tiles, resize
from imagescry_b200.models.embedding import l2_normalize_cells
tiles = torch.randint(0, 256, (4, 3, 64, 64), dtype=torch.uint8, device=mine)
st_mine = EmbeddingStore(torch.from_numpy(store[:4000]).to(mine))
want = (preprocess_tiles(tiles, output_hw=(32, 32), min_value=-3, max_value=3), resize(tiles, 48),
        l2_normalize_cells(tiles.float()), st_mine.search(qd, 10))
with torch.cuda.device(other):
    got = (preprocess_tiles(tiles, output_hw=(32, 32), min_value=-3, max_value=3), resize(tiles, 48),
           l2_normalize_cells(tiles.float()), st_mine.search(qd, 10))
    torch.cuda.synchronize(mine)
assert torch.equal(want[0], got[0]) and torch.equal(want[1], got[1]) and torch.equal(want[2], got[2])
assert torch.equal(want[3][1], got[3][1]) and got[0].device == mine
try:
    st_mine.search(qd.to(torch.device("cuda", other)), 10)
    raise SystemExit("operands on different devices were accepted")
except ValueError:
    pass
dist.barrier()
dist.destroy_process_group()
print("OK", rank)
"""


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_sharded_store_nccl_equals_single_gpu(tmp_path):
    world = min(torch.cuda.device_count(), 4)
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    script = tmp_path / "worker.py"
    script.write_text(_WORKER)
    procs = []
    for r in range(world):
        env = dict(os.environ, ISX_REPO=REPO, ISX_PORT=str(port), ISX_RANK=str(r), ISX_WORLD=str(world))
        procs.append(subprocess.Popen([sys.executable, str(script)], env=env, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True))
    outs = [p.communicate(timeout=600)[0] for p in procs]
    for r, (p, o) in enumerate(zip(procs, outs)):
        assert p.returncode == 0 and f"OK {r}" in o, o[-3000:]
