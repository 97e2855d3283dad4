"""CPU reference of the image-level (grouped) search: plain numpy restatements that the grouped
tests compare the CUDA path against.  Scores are the cosine scores of `oracle.cosine_scores` (the
ones `oracle.cosine_knn` ranks); the grouping uses no pre-selection shortcut."""

from __future__ import annotations

import numpy as np

from oracle.oracle import cosine_scores


def _first_per_group(s: np.ndarray, i: np.ndarray, g: np.ndarray, k: int):
    """One query: the k best groups of the entries (s, i, g), each by its first entry in (score desc,
    index asc) order; padded with (-inf, -1, -1)."""
    order = np.lexsort((i, -s))
    _, first = np.unique(g[order], return_index=True)
    pick = order[np.sort(first)][:k]
    out_s = np.full(k, -np.inf, np.float32)
    out_i = np.full(k, -1, np.int64)
    out_g = np.full(k, -1, np.int64)
    out_s[: len(pick)], out_i[: len(pick)], out_g[: len(pick)] = s[pick], i[pick], g[pick]
    return out_s, out_i, out_g


def cosine_knn_groups(store: np.ndarray, queries: np.ndarray, k: int, row_group, index_base: int = 0):
    """Image-level (grouped) cosine search.  Store row r belongs to group `row_group[r]` (>= 0, any
    order).  A group's score is the best cosine score of its rows (the scores of `cosine_knn`), its
    representative the first of its rows in (score desc, index asc) order; the result is the k groups
    whose representatives come first in that order: (scores Q×k float32, indices Q×k int64 =
    index_base + representative row, groups Q×k int64), padded with (-inf, -1, -1)."""
    row_group = np.asarray(row_group, dtype=np.int64)
    n = store.shape[0]
    assert row_group.shape == (n,)
    Q = queries.shape[0]
    full = np.concatenate([sc for _, sc in cosine_scores(store, queries)], axis=1) if n else np.zeros((Q, 0), np.float32)
    rows = np.arange(n, dtype=np.int64) + index_base
    out = [np.empty((Q, k), np.float32), np.empty((Q, k), np.int64), np.empty((Q, k), np.int64)]
    for r in range(Q):
        for o, v in zip(out, _first_per_group(full[r], rows, row_group, k)):
            o[r] = v
    return tuple(out)


def topk_merge_groups(scores: np.ndarray, idx: np.ndarray, groups: np.ndarray, k: int):
    """Merge G grouped partial results (G×Q×k each; index < 0 = padding) into the k best groups per
    query, each group once with its first entry in (score desc, index asc) order."""
    G, Q, kk = scores.shape
    s = np.transpose(scores, (1, 0, 2)).reshape(Q, G * kk).astype(np.float32)
    i = np.transpose(idx, (1, 0, 2)).reshape(Q, G * kk).astype(np.int64)
    g = np.transpose(groups, (1, 0, 2)).reshape(Q, G * kk).astype(np.int64)
    out = [np.empty((Q, k), np.float32), np.empty((Q, k), np.int64), np.empty((Q, k), np.int64)]
    for r in range(Q):
        keep = i[r] >= 0
        for o, v in zip(out, _first_per_group(s[r][keep], i[r][keep], g[r][keep], k)):
            o[r] = v
    return tuple(out)


