"""CPU reference of multi-vector (maxsim) image search: plain numpy restatements that the maxsim tests
compare the CUDA path against.  Cosine scores are those of `oracle.cosine_scores` (the ones
`oracle.cosine_knn` ranks)."""

from __future__ import annotations

import numpy as np

from oracle.oracle import cosine_scores


def cell_image_max(store: np.ndarray, queries: np.ndarray, row_group, num_groups: int, group_base: int = 0) -> np.ndarray:
    """Q × num_groups float32: for query row c and group g = group_base + j, the largest cosine score of
    c with a row of g; -inf where g has no row.  Rows whose group lies outside the range are ignored."""
    g = np.asarray(row_group, dtype=np.int64) - group_base
    out = np.full((queries.shape[0], num_groups), -np.inf, np.float32)
    for s, sc in cosine_scores(store, queries):
        gb = g[s:s + sc.shape[1]]
        keep = (gb >= 0) & (gb < num_groups)
        gs, cols = gb[keep], sc[:, keep]
        if not gs.size:
            continue
        order = np.argsort(gs, kind="stable")
        gs, cols = gs[order], cols[:, order]
        starts = np.flatnonzero(np.r_[True, gs[1:] != gs[:-1]])
        out[:, gs[starts]] = np.maximum(out[:, gs[starts]], np.maximum.reduceat(cols, starts, axis=1))
    return out


def set_scores_fp64(cell_max: np.ndarray, set_offsets) -> np.ndarray:
    """S × images float64: the mean of the set's per-cell maxima."""
    off = np.asarray(set_offsets, dtype=np.int64)
    out = np.full((len(off) - 1, cell_max.shape[1]), -np.inf)
    for s in range(len(off) - 1):
        if off[s + 1] > off[s]:
            out[s] = cell_max[off[s]:off[s + 1]].astype(np.float64).mean(axis=0)
    return out


def set_scores_fp32(values: np.ndarray, set_offsets) -> np.ndarray:
    """S × images float32: the library's rounding — fp32 sum of the set's per-cell values in ascending
    row order, then one correctly rounded division by the set's size."""
    off = np.asarray(set_offsets, dtype=np.int64)
    out = np.full((len(off) - 1, values.shape[1]), -np.inf, np.float32)
    for s in range(len(off) - 1):
        if off[s + 1] > off[s]:
            acc = np.zeros(values.shape[1], np.float32)
            for c in range(off[s], off[s + 1]):
                acc = (acc + values[c].astype(np.float32)).astype(np.float32)
            out[s] = (acc / np.float32(off[s + 1] - off[s])).astype(np.float32)
    return out


def topk_images(scores: np.ndarray, k: int):
    """Best k images of every set by (score desc, image asc); images scoring -inf are not results;
    padded with (-inf, -1).  Returns (scores S×k float, images S×k int64)."""
    S = scores.shape[0]
    out_s = np.full((S, k), -np.inf, scores.dtype)
    out_i = np.full((S, k), -1, np.int64)
    for s in range(S):
        ids = np.flatnonzero(scores[s] > -np.inf)
        order = ids[np.lexsort((ids, -scores[s][ids]))][:k]
        out_s[s, :len(order)], out_i[s, :len(order)] = scores[s][order], order
    return out_s, out_i


def maxsim_search(store: np.ndarray, queries: np.ndarray, set_offsets, row_group, num_groups: int, k: int):
    """The whole search in fp64 set scores: (scores S×k float64, images S×k int64, fp64 S×images)."""
    full = set_scores_fp64(cell_image_max(store, queries, row_group, num_groups), set_offsets)
    s, i = topk_images(full, k)
    return s, i, full
