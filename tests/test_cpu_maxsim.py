"""CPU checks of multi-vector (maxsim) image search: the numpy reference, the image-aligned block plan,
the combine of columns of images cut by shard boundaries, and argument checks that need no device."""

from __future__ import annotations

import numpy as np
import pytest
import torch

import maxsim_oracle as M
from imagescry_b200 import search as S
from oracle import oracle as O


def _data(n, q, d, seed):
    rng = np.random.default_rng(seed)
    return O.bf16_round(rng.standard_normal((n, d)).astype(np.float32)), O.bf16_round(rng.standard_normal((q, d)).astype(np.float32))


def test_cell_image_max_is_the_best_cosine_of_each_image():
    store, queries = _data(300, 9, 16, 0)
    groups = np.random.default_rng(1).integers(0, 40, 300)
    groups[groups == 7] = 8  # group 7 has no row
    cm = M.cell_image_max(store, queries, groups, 40)
    full = np.concatenate([sc for _, sc in O.cosine_scores(store, queries)], axis=1)
    for g in range(40):
        want = full[:, groups == g].max(axis=1) if (groups == g).any() else np.full(9, -np.inf, np.float32)
        assert np.array_equal(cm[:, g], want)
    # a window of ids: the rest is ignored
    part = M.cell_image_max(store, queries, groups, 10, group_base=20)
    assert np.array_equal(part, cm[:, 20:30])


def test_set_scores_and_topk():
    store, queries = _data(512, 12, 8, 2)
    groups = np.arange(512) // 32
    off = [0, 1, 5, 5, 12]  # one cell, four cells, empty, seven cells
    cm = M.cell_image_max(store, queries, groups, 16)
    f64 = M.set_scores_fp64(cm, off)
    f32 = M.set_scores_fp32(cm, off)
    assert np.array_equal(f32[0], cm[0])  # a set of one cell scores its cell's maxima exactly
    assert np.all(np.isneginf(f64[2])) and np.all(np.isneginf(f32[2]))
    assert np.abs(f32[[0, 1, 3]] - f64[[0, 1, 3]]).max() < 1e-6
    # the fp32 sum is taken in row order: a hand-rolled loop agrees bit for bit
    acc = np.float32(0)
    for c in range(5, 12):
        acc = np.float32(acc + cm[c, 3])
    assert f32[3, 3] == np.float32(acc / np.float32(7))
    s, i = M.topk_images(f32, 20)  # more than the 16 images
    assert np.all(i[[0, 1, 3], 16:] == -1) and np.all(np.isneginf(s[:, 16:])) and np.all(i[2] == -1)
    for r in (0, 1, 3):
        assert np.array_equal(np.lexsort((i[r, :16], -s[r, :16])), np.arange(16))
        assert sorted(i[r, :16].tolist()) == list(range(16))
    ws, wi, full = M.maxsim_search(store, queries, off, groups, 16, 5)
    assert np.array_equal(full, f64) and np.array_equal(wi[1], np.argsort(-f64[1], kind="stable")[:5])


def test_block_plan():
    off = torch.tensor([0, 4, 4, 10, 11, 20, 30])  # 6 images, one empty
    assert S.maxsim_block_plan(off, 10, 1 << 30) == [(0, 6)]
    assert S.maxsim_block_plan(off, 10, 2 * 10 * 4) == [(0, 2), (2, 4), (4, 6)]
    assert S.maxsim_block_plan(off, 10, 3 * 10 * 4 + 39) == [(0, 3), (3, 6)]
    # one image's column alone is larger than the budget: one image per block
    assert S.maxsim_block_plan(off, 1000, 100) == [(i, i + 1) for i in range(6)]
    assert S.maxsim_block_plan(torch.tensor([0]), 10, 1 << 20) == []
    for plan in (S.maxsim_block_plan(off, q, b) for q in (1, 7, 100) for b in (1, 50, 4096)):
        assert plan[0][0] == 0 and plan[-1][1] == 6 and all(a < b for a, b in plan)
        assert all(plan[j][1] == plan[j + 1][0] for j in range(len(plan) - 1))
    for bad in (0, -1, 1.5, True, None):
        with pytest.raises(ValueError):
            S.maxsim_block_plan(off, 10, bad)


def test_combine_cut_columns():
    ids = torch.tensor([-1, 5, 5, 9, -1, 5])
    cols = torch.tensor([[9.0, 9.0], [0.5, -2.0], [0.25, -1.0], [7.0, 7.0], [8.0, 8.0], [-float("inf"), -3.0]])
    assert torch.equal(S.combine_cut_columns(ids, cols, 5), torch.tensor([0.5, -1.0]))
    assert torch.equal(S.combine_cut_columns(ids, cols, 9), torch.tensor([7.0, 7.0]))
    with pytest.raises(ValueError):
        S.combine_cut_columns(ids, cols, 4)
    with pytest.raises(ValueError):
        S.combine_cut_columns(ids[:3], cols, 5)


def test_set_validation_without_a_device():
    # sets are validated with the store's group-layout rule before any launch
    assert S.group_offsets(4, 12).tolist() == [0, 4, 8, 12]
    assert S.group_offsets(torch.tensor([0, 0, 3, 12]), 12).tolist() == [0, 0, 3, 12]
    for bad in (5, 0, True, torch.tensor([0, 3]), torch.tensor([0, 5, 3, 12]), torch.tensor([0.0, 12.0])):
        with pytest.raises(ValueError):
            S.group_offsets(bad, 12)
    with pytest.raises(RuntimeError):
        S.EmbeddingStore(torch.zeros(8, 16), groups=4)  # the store lives on the GPU only
