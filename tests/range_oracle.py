"""Plain numpy reference of the range search (EmbeddingStore.search_range): every store row whose
cosine score with a query is >= a threshold, as CSR ordered by (score desc, row asc).  Scores are the
oracle's `cosine_scores` (fp32) or exact fp64 ones; neither is bit-identical to the kernel's, so a
comparison allows a band around the threshold."""

from __future__ import annotations

import numpy as np

from oracle import oracle as O


def exact_scores(store: np.ndarray, queries: np.ndarray, eps: float = 1e-12) -> np.ndarray:
    """fp64 Q×N cosine scores with F.normalize's eps."""
    s = store.astype(np.float64)
    q = queries.astype(np.float64)
    sn = s / np.maximum(np.linalg.norm(s, axis=1), eps)[:, None]
    qn = q / np.maximum(np.linalg.norm(q, axis=1), eps)[:, None]
    return qn @ sn.T


def cosine_range(store: np.ndarray, queries: np.ndarray, threshold: float, *, index_base: int = 0,
                 exclude_self: bool = False):
    """(offsets int64 Q + 1, indices int64, scores fp32) from the oracle's fp32 cosine scores."""
    per_q_idx = [[] for _ in range(queries.shape[0])]
    per_q_s = [[] for _ in range(queries.shape[0])]
    for s0, sc in O.cosine_scores(store, queries):
        if exclude_self:
            r = np.arange(queries.shape[0])
            inside = (r >= s0) & (r < s0 + sc.shape[1])
            sc[r[inside], r[inside] - s0] = -np.inf
        qi, cj = np.nonzero(sc >= np.float32(threshold))
        for a, b in zip(qi.tolist(), cj.tolist()):
            per_q_idx[a].append(s0 + b + index_base)
            per_q_s[a].append(sc[a, b])
    offsets = np.zeros(queries.shape[0] + 1, np.int64)
    idx, scores = [], []
    for a in range(queries.shape[0]):
        i = np.asarray(per_q_idx[a], np.int64)
        s = np.asarray(per_q_s[a], np.float32)
        order = np.lexsort((i, -s))
        idx.append(i[order])
        scores.append(s[order])
        offsets[a + 1] = offsets[a] + len(i)
    return offsets, np.concatenate(idx) if idx else np.zeros(0, np.int64), np.concatenate(scores) if scores else np.zeros(0, np.float32)
