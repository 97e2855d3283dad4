"""CPU reference of the fp8 search: plain numpy / torch restatements that the fp8 tests compare the CUDA
path against.

quantize   every row scaled by the power of two that puts its largest |x| in (224, 448] (computed from
           the exponent of the maximum, not from a rounded log2), then torch's CPU cast to
           float8_e4m3fn (round to nearest even), zero-padded to d16 bytes;
scan       `oracle.cosine_knn` over the dequantized rows;
re-score   fp64 cosine of the bf16 rows."""

from __future__ import annotations

import numpy as np
import torch

from oracle.oracle import cosine_knn, row_rnorm


def fp8_width(d: int) -> int:
    return (d + 15) // 16 * 16


def row_exponent(m: np.ndarray) -> np.ndarray:
    """e with 224 < m * 2^e <= 448 for every finite m > 0; 0 for m == 0."""
    m = np.asarray(m, dtype=np.float64)
    f, ex = np.frexp(m)  # m = f * 2^ex, f in [0.5, 1)
    e = np.where(f > 0.875, 8 - ex, 9 - ex)
    return np.where(m > 0, e, 0).astype(np.int64)


def quantize(x: np.ndarray) -> tuple[np.ndarray, np.ndarray]:
    """bf16-valued float32 rows N×d → (uint8 N×d16 E4M3 bit patterns, fp32 rnorm of the E4M3 values)."""
    x = np.asarray(x, dtype=np.float32)
    n, d = x.shape
    e = row_exponent(np.abs(x).max(axis=1) if d else np.zeros(n))
    scaled = (x.astype(np.float64) * np.exp2(e.astype(np.float64))[:, None]).astype(np.float32)
    q = torch.from_numpy(scaled).to(torch.float8_e4m3fn)
    out = np.zeros((n, fp8_width(d)), np.uint8)
    out[:, :d] = q.view(torch.uint8).numpy()
    return out, row_rnorm(dequantize(out))


def dequantize(b: np.ndarray) -> np.ndarray:
    """uint8 E4M3 bit patterns → float32 values."""
    return torch.from_numpy(np.ascontiguousarray(b)).view(torch.float8_e4m3fn).float().numpy()


def scan(store: np.ndarray, queries: np.ndarray, k: int, *, index_base: int = 0):
    """Top-k by the cosine of the quantized rows: (scores Q×k float32, indices Q×k int64)."""
    return cosine_knn(dequantize(quantize(store)[0]), dequantize(quantize(queries)[0]), k, index_base=index_base)


def rescore(store: np.ndarray, queries: np.ndarray, cand: np.ndarray, k: int, *, index_base: int = 0):
    """fp64 cosine of every candidate (global rows; < 0 or outside the store = none; duplicates once),
    best k by (score desc, index asc), padded with (-inf, -1): (scores Q×k float64, indices Q×k int64)."""
    s64 = store.astype(np.float64)
    q64 = queries.astype(np.float64)
    sn = np.maximum(np.linalg.norm(s64, axis=1), 1e-12)
    qn = np.maximum(np.linalg.norm(q64, axis=1), 1e-12)
    Q = queries.shape[0]
    out_s = np.full((Q, k), -np.inf)
    out_i = np.full((Q, k), -1, np.int64)
    for r in range(Q):
        rows = np.unique([int(c) for c in cand[r] if 0 <= c - index_base < store.shape[0]]).astype(np.int64)
        sc = (s64[rows - index_base] @ q64[r]) / (sn[rows - index_base] * qn[r]) if len(rows) else np.zeros(0)
        order = np.lexsort((rows, -sc))[:k]
        out_s[r, : len(order)], out_i[r, : len(order)] = sc[order], rows[order]
    return out_s, out_i
