"""Embedding-store format bridge (SURVEY.md §8f.1): the reference's `embeddings.embedding_data` BLOBs
↔ the device-resident bf16 search store.

The reference stores every embedding map as the raw bytes of a float32, C-order `C×H×W` array
(`storage/models.py:94-129`: `Embedding.create` = `tensor.numpy().tobytes()`, `embedding_tensor` =
`np.frombuffer(...).reshape(C, H, W)`), and reads them back in bulk as `N×C×H×W`
(`storage/operations.py:108-144`).  This module decodes/encodes exactly that wire format on the
host and turns stacks of maps into search rows on the GPU (`isx_maps_to_rows_bf16`):

    pool=None    one row per feature-map cell, in `EmbeddingBatch.get_flat_vectors` order
                 (`data.py:112-118`): row = image * H*W + cell
    pool="mean"  one row per image (spatial mean)

SQLite access itself (DatabaseManager, sessions) stays the reference's code and is out of scope.
"""

from __future__ import annotations

from collections.abc import Iterable, Sequence

import numpy as np
import torch
from torch import Tensor

from imagescry_b200 import _lib
from imagescry_b200.search import EmbeddingStore


def decode_embedding_blob(data: bytes, dim: int, height: int, width: int) -> Tensor:
    """`Embedding.embedding_tensor` (`storage/models.py:94-102`): bytes → float32 `C×H×W` tensor."""
    expected = dim * height * width * 4
    if len(data) != expected:
        raise ValueError(f"embedding BLOB has {len(data)} bytes, expected {expected} for {dim}x{height}x{width} float32")
    return torch.from_numpy(np.frombuffer(data, dtype=np.float32).reshape(dim, height, width).copy())


def encode_embedding_blob(embedding: Tensor) -> tuple[bytes, int, int, int]:
    """`Embedding.create` (`storage/models.py:104-129`): float32 `C×H×W` tensor → (bytes, C, H, W)."""
    if embedding.ndim != 3:
        raise ValueError(f"embedding must be C×H×W, got shape {tuple(embedding.shape)}")
    t = embedding.detach().to(device="cpu", dtype=torch.float32).contiguous()
    c, h, w = t.shape
    return t.numpy().tobytes(), c, h, w


def stack_blobs(records: Iterable[tuple[bytes, int, int, int]]) -> Tensor:
    """Bulk read (`storage/operations.py:108-144`): equal-shaped BLOB records → pinned float32
    `N×C×H×W` host tensor ready for one H2D copy."""
    maps = [decode_embedding_blob(*r) for r in records]
    if not maps:
        raise ValueError("no embedding records")
    shape = maps[0].shape
    if any(m.shape != shape for m in maps):
        raise ValueError("all embedding maps must share one C×H×W shape (pad or group them first)")
    out = torch.stack(maps, dim=0)
    return out.pin_memory() if torch.cuda.is_available() else out


def maps_to_rows(maps: Tensor, *, pool: str | None = None) -> Tensor:
    """float32 `N×C×H×W` maps on a CUDA device → bf16 search rows (`(N·H·W)×C`, or `N×C` pooled)."""
    _lib.require_cuda(maps, "maps")
    if maps.ndim != 4:
        raise ValueError(f"maps must be N×C×H×W, got shape {tuple(maps.shape)}")
    if pool not in (None, "mean"):
        raise ValueError(f"Invalid pool: {pool}")
    x = maps.to(torch.float32).contiguous()
    n, c, h, w = x.shape
    rows = torch.empty((n if pool else n * h * w, c), dtype=torch.bfloat16, device=x.device)
    if n:
        with _lib.on_device(x) as stream:
            rc = _lib.load().isx_maps_to_rows_bf16(x.data_ptr(), n, c, h * w, int(pool is not None), rows.data_ptr(), stream)
        _lib.check(rc, "isx_maps_to_rows_bf16")
    return rows


def store_from_maps(maps: Tensor, *, pool: str | None = None, index_base: int = 0, device=None) -> EmbeddingStore:
    """Build a search store from a stack of embedding maps (host or device).  The store knows its
    images (`groups` = H·W rows per image, or 1 when pooled), so `search_images` works on it."""
    if not maps.is_cuda:
        maps = maps.to(device or "cuda", non_blocking=True)
    cells = 1 if pool else maps.shape[2] * maps.shape[3]
    return EmbeddingStore(maps_to_rows(maps, pool=pool), index_base=index_base, groups=cells)


def store_from_blobs(records: Iterable[tuple[bytes, int, int, int]], *, pool: str | None = None, index_base: int = 0, device=None) -> EmbeddingStore:
    """BLOB records (embedding_data, embedding_dim, embedding_height, embedding_width) → store."""
    return store_from_maps(stack_blobs(records), pool=pool, index_base=index_base, device=device)


def store_from_mixed_blobs(
    records: Iterable[tuple[bytes, int, int, int]], *, pool: str | None = None, index_base: int = 0, device=None
) -> tuple[EmbeddingStore, Tensor]:
    """BLOB records whose maps differ in H×W (same channel count) → one search store.

    A real imagescry database holds one embedding map per image and images differ in size.  The
    reference's reader pads every map with zero cells to the largest H×W (`StoredEmbeddingsDataset`,
    `data.py:378-399`); zero cells are not embeddings, so here nothing is padded: records are grouped by
    shape (`SimilarShapeBatcher`'s rule), every group is converted on the GPU, and the rows of image i
    occupy `[row_offsets[i], row_offsets[i + 1])` of the store in the records' order (one row per
    cell in `get_flat_vectors` order, or one pooled row).  Returns `(store, row_offsets)`, `row_offsets`
    an int64 CPU tensor of length `n + 1`; `rows_to_image_cell(rows, row_offsets)` maps hits back."""
    from imagescry_b200.ingest import similar_shape_batches

    recs = list(records)
    if not recs:
        raise ValueError("no embedding records")
    dims = {r[1] for r in recs}
    if len(dims) != 1:
        raise ValueError(f"all embedding maps must share one channel count, got {sorted(dims)}")
    (c,) = dims
    per_image = [1 if pool else r[2] * r[3] for r in recs]
    row_offsets = torch.zeros(len(recs) + 1, dtype=torch.int64)
    row_offsets[1:] = torch.cumsum(torch.tensor(per_image, dtype=torch.int64), dim=0)
    dev = torch.device(device or "cuda")
    rows = torch.empty((int(row_offsets[-1]), c), dtype=torch.bfloat16, device=dev)
    for batch in similar_shape_batches([(r[2], r[3]) for r in recs], 4096):
        maps = stack_blobs([recs[i] for i in batch]).to(dev, non_blocking=True)
        part = maps_to_rows(maps, pool=pool)
        n_rows = per_image[batch[0]]
        dst = torch.cat([torch.arange(int(row_offsets[i]), int(row_offsets[i]) + n_rows) for i in batch]).to(dev)
        rows.index_copy_(0, dst, part)
    return EmbeddingStore(rows, index_base=index_base, groups=row_offsets), row_offsets


def rows_to_image_cell(rows: Tensor | Sequence[int], cells_per_image: int | Tensor) -> tuple[Tensor, Tensor]:
    """Search result rows of a per-cell store → (image position in the stack, cell index y*W + x).
    `cells_per_image`: the common cell count, or the `row_offsets` of `store_from_mixed_blobs`."""
    r = torch.as_tensor(rows)
    if isinstance(cells_per_image, Tensor):
        offsets = cells_per_image.to(r.device)
        img = torch.searchsorted(offsets, r, right=True) - 1
        return img, r - offsets[img]
    return torch.div(r, cells_per_image, rounding_mode="floor"), r % cells_per_image
