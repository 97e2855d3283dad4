"""CPU checks of the range search's host logic: threshold validation, the capacity and retry rule,
the numpy reference, and the padded all-gather of the sharded form over gloo (world size 2)."""

from __future__ import annotations

import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import range_oracle as R
from conftest import REPO
from imagescry_b200 import search as S
from oracle import oracle as O


def test_threshold_validation():
    assert S.range_threshold(0.5) == 0.5
    assert S.range_threshold(1) == 1.0
    assert S.range_threshold(torch.tensor(0.25)) == 0.25
    assert S.range_threshold(0.1) == float(np.float32(0.1))  # compared in float32
    assert S.range_threshold(np.float32(0.3)) == float(np.float32(0.3))  # numpy scalars are numbers too
    assert S.range_threshold(np.float64(-0.5)) == -0.5 and S.range_threshold(np.int64(1)) == 1.0
    for bad in (float("nan"), float("inf"), -float("inf"), 1e39, np.float32("nan"), True, np.bool_(True), "0.5", None,
                torch.tensor([0.1, 0.2]), torch.tensor(1)):
        with pytest.raises(ValueError):
            S.range_threshold(bad)


def test_capacity_and_retry_rule():
    assert S.range_capacity(S.RANGE_HITS_PER_QUERY, 1) == S.RANGE_MIN_CAPACITY
    assert S.range_capacity(64, 10_000) == 800_000  # the expected hits plus a quarter
    assert S.range_capacity(0.5, 10_000) == 6_250  # follows a strict call down, to the floor
    assert S.range_capacity(0.0, 1_000_000) == S.RANGE_MIN_CAPACITY
    assert S.range_retry_capacity(100, 4096) is None
    assert S.range_retry_capacity(4096, 4096) is None
    assert S.range_retry_capacity(4097, 4096) == 4097


def test_empty_result_and_sort_validation():
    off, idx, sc = S.range_empty(3, "cpu")
    assert off.tolist() == [0, 0, 0, 0] and idx.dtype == torch.int64 and sc.dtype == torch.float32 and idx.numel() == 0
    with pytest.raises(ValueError):
        S.range_sort(torch.zeros((4, 2), dtype=torch.int32), 2, 0)
    with pytest.raises(ValueError):
        S.range_sort(torch.zeros((4, 3), dtype=torch.int64), 2, 0)
    with pytest.raises(RuntimeError):  # the ordering pass runs on the GPU only
        S.range_sort(torch.zeros((4, 3), dtype=torch.int32), 2, 0)


def test_oracle_range_against_brute_force():
    rng = np.random.default_rng(1)
    store = O.bf16_round(rng.standard_normal((300, 16)).astype(np.float32))
    store[7] = store[2]
    queries = np.concatenate([store[[2]], O.bf16_round(rng.standard_normal((4, 16)).astype(np.float32))])
    off, idx, sc = R.cosine_range(store, queries, 0.3, index_base=10)
    ex = R.exact_scores(store, queries)
    for r in range(5):
        i = idx[off[r]:off[r + 1]] - 10
        s = sc[off[r]:off[r + 1]]
        assert set(np.nonzero(ex[r] >= 0.301)[0]) <= set(i.tolist()) <= set(np.nonzero(ex[r] >= 0.299)[0])
        assert np.array_equal(np.lexsort((i, -s)), np.arange(len(i)))
    assert idx[0] == 12 and idx[1] == 17  # a tie at the top is ordered by row
    off, idx, _ = R.cosine_range(store, store, 0.99, exclude_self=True)
    assert idx[off[2]:off[3]].tolist() == [7] and idx[off[7]:off[8]].tolist() == [2]


_WORKER = r"""
import os, sys
import torch, torch.distributed as dist
sys.path.insert(0, os.environ["ISX_REPO"])
from imagescry_b200.search import gather_range_records
dist.init_process_group("gloo", init_method=f"tcp://127.0.0.1:{os.environ['ISX_PORT']}",
                        rank=int(os.environ["ISX_RANK"]), world_size=2)
rank = dist.get_rank()
counts = [5, 2]
# a record buffer longer than its hit count: only the first `count` records are real
rec = torch.arange(30, dtype=torch.int32).view(10, 3) + 100 * rank
out, total = gather_range_records(rec, counts[rank])
assert total == 7 and out.shape == (10, 3), (total, out.shape)
real = out[out[:, 1] >= 0]
want = torch.cat([torch.arange(30, dtype=torch.int32).view(10, 3)[:5], torch.arange(30, dtype=torch.int32).view(10, 3)[:2] + 100])
assert torch.equal(real, want), real
assert bool((out[out[:, 1] < 0] == -1).all())
out, total = gather_range_records(rec[:0], 0) if rank else gather_range_records(rec, 3)
assert total == 3 and out.shape == (6, 3) and int((out[:, 1] >= 0).sum()) == 3
dist.barrier()
dist.destroy_process_group()
print("OK", rank)
"""


def test_sharded_range_gather_gloo_world2(tmp_path):
    import socket

    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    script = tmp_path / "worker.py"
    script.write_text(_WORKER)
    procs = []
    for r in range(2):
        env = dict(os.environ, ISX_REPO=REPO, ISX_PORT=str(port), ISX_RANK=str(r), OMP_NUM_THREADS="1")
        procs.append(subprocess.Popen([sys.executable, str(script)], env=env, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True))
    outs = [p.communicate(timeout=180)[0] for p in procs]
    for r, (p, o) in enumerate(zip(procs, outs)):
        assert p.returncode == 0 and f"OK {r}" in o, o
