"""Image-level (grouped) search on the host: the oracle's semantics, the `groups` layouts a store
accepts, and the sharded plumbing (local grouped lists → one all-gather of int32 records → grouped
merge) over gloo with the oracle standing in for the kernel."""

from __future__ import annotations

import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from conftest import REPO
import grouped_oracle as G
from oracle import oracle as O


def _brute(scores_row, groups, k):
    """Straight restatement: best score per group, representative = lowest row among the group's best."""
    best = {}
    for r, (s, g) in enumerate(zip(scores_row, groups)):
        if g not in best or s > best[g][0]:
            best[g] = (s, r)
    ranked = sorted(best.items(), key=lambda kv: (-kv[1][0], kv[1][1]))[:k]
    return [v[0] for _, v in ranked], [v[1] for _, v in ranked], [g for g, _ in ranked]


def test_oracle_groups_against_brute_force_and_ties():
    rng = np.random.default_rng(0)
    store = O.bf16_round(rng.standard_normal((60, 16)).astype(np.float32))
    queries = O.bf16_round(rng.standard_normal((4, 16)).astype(np.float32))
    store[7] = store[3]           # tie inside a group (rows 3 and 7 are both group 0 below)
    store[50] = 2 * store[3]      # tie across groups: same cosine, higher row
    queries[0] = store[3]
    groups = np.zeros(60, np.int64)
    groups[:10] = 0
    groups[10:] = 1 + (np.arange(50) % 9)  # non-contiguous ids
    s, i, g = G.cosine_knn_groups(store, queries, 5, groups, index_base=100)
    full = np.concatenate([sc for _, sc in O.cosine_scores(store, queries)], axis=1)
    for r in range(4):
        bs, bi, bg = _brute(full[r], groups, 5)
        assert np.array_equal(s[r], np.array(bs, np.float32))
        assert i[r].tolist() == [b + 100 for b in bi] and g[r].tolist() == bg
    # query 0: group 0 via row 3 (the lower of the tied rows 3 and 7), then the group of row 50
    assert i[0, :2].tolist() == [103, 150] and g[0, :2].tolist() == [0, groups[50]]
    assert s[0, 0] == s[0, 1]


def test_oracle_groups_padding_single_group_and_merge():
    rng = np.random.default_rng(1)
    store = O.bf16_round(rng.standard_normal((12, 8)).astype(np.float32))
    queries = O.bf16_round(rng.standard_normal((3, 8)).astype(np.float32))
    s, i, g = G.cosine_knn_groups(store, queries, 6, np.arange(12) // 4)  # 3 groups < k
    assert (g[:, :3] >= 0).all() and (g[:, 3:] == -1).all() and (i[:, 3:] == -1).all() and np.isneginf(s[:, 3:]).all()
    s1, i1, g1 = G.cosine_knn_groups(store, queries, 3, np.zeros(12, np.int64))  # one group
    rs, ri = O.cosine_knn(store, queries, 1)
    assert np.array_equal(i1[:, 0], ri[:, 0]) and (g1[:, 0] == 0).all() and (i1[:, 1:] == -1).all()
    # c = 1: grouped search is the row search
    sc, ic, gc = G.cosine_knn_groups(store, queries, 5, np.arange(12))
    rs, ri = O.cosine_knn(store, queries, 5)
    assert np.array_equal(ic, ri) and np.array_equal(sc, rs) and np.array_equal(gc, ri)
    # merging two row blocks whose cut splits a group equals one search
    groups = np.arange(12) // 5
    a = G.cosine_knn_groups(store[:7], queries, 3, groups[:7])
    b = G.cosine_knn_groups(store[7:], queries, 3, groups[7:], index_base=7)
    ms, mi, mg = G.topk_merge_groups(*(np.stack(x) for x in zip(a, b)), 3)
    ws, wi, wg = G.cosine_knn_groups(store, queries, 3, groups)
    assert np.array_equal(mi, wi) and np.array_equal(mg, wg) and np.array_equal(ms, ws)


def test_group_layout_validation():
    from imagescry_b200.search import group_offsets, image_cells, row_groups

    assert group_offsets(4, 12).tolist() == [0, 4, 8, 12]
    assert group_offsets(torch.tensor([0, 3, 3, 7]), 7).tolist() == [0, 3, 3, 7]
    assert row_groups(group_offsets(torch.tensor([0, 3, 3, 7]), 7), 2, 7).tolist() == [0, 2, 2, 2, 2]
    for bad in (5, 0, -1, True, 2.0, torch.tensor([0, 3, 11]), torch.tensor([1, 12]), torch.tensor([0, 8, 4, 12]),
                torch.tensor([[0, 12]]), torch.tensor([0.0, 12.0])):
        with pytest.raises(ValueError):
            group_offsets(bad, 12)
    cells = image_cells(torch.tensor([[5, 9, -1]]), torch.tensor([[1, 2, -1]]), torch.tensor([0, 4, 8]))
    assert cells.tolist() == [[1, 1, -1]]


def test_search_images_needs_groups_and_binding():
    from imagescry_b200 import _lib, search

    assert "isx_knn_search_grouped" in _lib.SIGNATURES and "isx_topk_merge_grouped" in _lib.SIGNATURES
    st = search.EmbeddingStore.__new__(search.EmbeddingStore)
    st.row_group = None
    with pytest.raises(ValueError):
        st.search_images_raw(torch.zeros((1, 8)), 3)


_WORKER = r"""
import os, sys
import numpy as np, torch, torch.distributed as dist
sys.path.insert(0, os.environ["ISX_REPO"])
sys.path.insert(0, os.path.join(os.environ["ISX_REPO"], "tests"))
import grouped_oracle as G
from imagescry_b200.search import gather_group_records, group_offsets, image_cells, pack_group_records, row_groups, shard_range
from oracle import oracle as O
dist.init_process_group("gloo", init_method=f"tcp://127.0.0.1:{os.environ['ISX_PORT']}",
                        rank=int(os.environ["ISX_RANK"]), world_size=2)
rank = dist.get_rank()
rng = np.random.default_rng(0)
n, c = 1001, 7                       # 143 images; the shard cut (row 501) falls inside image 71
base = rng.standard_normal((n // c, 32)).astype(np.float32)
store = O.bf16_round(np.repeat(base, c, axis=0) + 0.1 * rng.standard_normal((n, 32)).astype(np.float32))
queries = O.bf16_round(store[[3, 500, 502, 990]] + 0.05 * rng.standard_normal((4, 32)).astype(np.float32))
offsets = group_offsets(c, n)
b, e = shard_range(n, 2, rank)
groups = row_groups(offsets, b, e).numpy()
# the local grouped search is the CUDA kernel's job on a GPU box; the oracle stands in for it here
ls, li, lg = G.cosine_knn_groups(store[b:e], queries, 6, groups, index_base=b)
rec = gather_group_records(pack_group_records(torch.from_numpy(ls), torch.from_numpy(li), torch.from_numpy(lg)))
assert rec.shape == (2, 4, 6, 3) and rec.dtype == torch.int32
ms, mi, mg = G.topk_merge_groups(rec[..., 0].contiguous().view(torch.float32).numpy(), rec[..., 1].numpy(), rec[..., 2].numpy(), 6)
ws, wi, wg = G.cosine_knn_groups(store, queries, 6, np.arange(n) // c)
assert np.array_equal(mi, wi) and np.array_equal(mg, wg) and np.array_equal(ms, ws), rank
assert len(set(mg[1].tolist())) == 6 and 71 in mg[1].tolist()   # the image cut by the shard boundary: once
cells = image_cells(torch.from_numpy(mi), torch.from_numpy(mg), offsets[:-1])
assert torch.equal(cells, torch.from_numpy(wi - (np.arange(n) // c * c)[wi]))
dist.barrier()
dist.destroy_process_group()
print("OK", rank)
"""


def test_sharded_grouped_plumbing_gloo_world2(tmp_path):
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
