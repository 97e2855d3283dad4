"""ROI masks on the feature-map grid and ROI query vectors (SURVEY.md §8f-4).

Mirror of `imagescry/geometry.py:14-65` `create_roi_mask` — same name, arguments, return type
(`Int64[Tensor, "H W"]`) and class-index convention — computed by `isx_roi_rasterize` on the GPU,
plus the step the reference leaves to its annotator app: pooling the embedding cells an ROI covers
into one query vector for the cosine search (`isx_masked_pool`).

The reference rasterises with `rasterio.features.rasterize(..., all_touched=True)`; rasterio and
shapely are not installed here and are not needed: a polygon is anything with shapely's
`.exterior.coords` / `.interiors`, a `{"exterior": [...], "interiors": [[...], ...]}` dict, or a
plain sequence of `(x, y)` vertices in image coordinates.  The rule is "a cell is burned when its
rectangle shares positive area with the polygon" (DESIGN.md §8f-4 states how that relates to GDAL).
"""

from __future__ import annotations

from collections.abc import Sequence

import numpy as np
import torch
from torch import Tensor

from imagescry_b200 import _lib


def _rings(poly) -> list[np.ndarray]:
    if hasattr(poly, "exterior"):
        rings = [np.asarray(poly.exterior.coords, dtype=np.float64)]
        rings += [np.asarray(r.coords, dtype=np.float64) for r in poly.interiors]
    elif isinstance(poly, dict):
        rings = [np.asarray(poly["exterior"], dtype=np.float64)]
        rings += [np.asarray(r, dtype=np.float64) for r in poly.get("interiors", [])]
    else:
        rings = [np.asarray(poly, dtype=np.float64)]
    out = []
    for r in rings:
        if r.ndim != 2 or r.shape[1] != 2 or r.shape[0] < 3:
            raise ValueError(f"a polygon ring needs at least three (x, y) vertices, got an array of shape {r.shape}")
        if np.array_equal(r[0], r[-1]):
            r = r[:-1]
        out.append(r)
    return out


def _is_single_polygon(roi) -> bool:
    if hasattr(roi, "exterior") or isinstance(roi, dict):
        return True
    try:
        first = roi[0]
    except (TypeError, IndexError, KeyError):
        return True
    if hasattr(first, "exterior") or isinstance(first, dict):
        return False
    # a vertex sequence: its first element is an (x, y) pair of numbers
    return np.ndim(first) == 1 and len(first) == 2 and np.ndim(first[0]) == 0


def polygon_edges(roi) -> tuple[np.ndarray, np.ndarray]:
    """Flatten polygon(s) into the C ABI's edge list: fp32 `[n_edges][4]` (x0, y0, x1, y1) and int32
    `poly_offsets[n_poly + 1]`."""
    polys = [roi] if _is_single_polygon(roi) else list(roi)
    edges, offsets = [], [0]
    for poly in polys:
        for ring in _rings(poly):
            nxt = np.roll(ring, -1, axis=0)
            edges.append(np.concatenate([ring, nxt], axis=1))
        offsets.append(offsets[-1] + sum(len(r) for r in _rings(poly)))
    e = np.concatenate(edges, axis=0).astype(np.float32) if edges else np.zeros((0, 4), dtype=np.float32)
    return np.ascontiguousarray(e), np.asarray(offsets, dtype=np.int32)


def create_roi_mask(
    roi,
    original_image_shape: tuple[int, int] | torch.Size,
    feature_map_shape: tuple[int, int] | torch.Size,
    class_index: int = 1,
    *,
    device: torch.device | str | int | None = None,
) -> Tensor:
    """Mask of the region(s) of interest on the feature map (`geometry.py:14-65`).

    Args:
        roi: polygon or list of polygons on the original image (see the module docstring).
        original_image_shape: (height, width) of the image the ROI is defined on.
        feature_map_shape: (height, width) of the feature map to rasterise onto.
        class_index: value the covered cells are filled with.
        device: CUDA device of the result (default: the current one).

    Returns:
        Int64 tensor `H x W` on the device: `class_index` in covered cells, 0 elsewhere.

    Example (the reference's docstring example, `geometry.py:33-43`):
        >>> create_roi_mask([(0, 0), (4, 0), (4, 3), (0, 3)], (6, 8), (3, 4)).tolist()
        [[1, 1, 0, 0], [1, 1, 0, 0], [0, 0, 0, 0]]
    """
    h, w = (int(v) for v in original_image_shape)
    hf, wf = (int(v) for v in feature_map_shape)
    if min(h, w, hf, wf) <= 0:
        raise ValueError(f"shapes must be positive, got image {h}x{w} and feature map {hf}x{wf}")
    lib = _lib.load()
    dev = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
    if dev.type != "cuda":
        raise RuntimeError(f"create_roi_mask runs on the GPU only (got device {dev}); there is no CPU fallback")
    edges, offsets = polygon_edges(roi)
    with torch.cuda.device(dev):
        d_edges = torch.from_numpy(edges).to(dev)
        d_off = torch.from_numpy(offsets).to(dev)
        mask = torch.empty((hf, wf), dtype=torch.int64, device=dev)
        rc = lib.isx_roi_rasterize(d_edges.data_ptr(), d_off.data_ptr(), len(offsets) - 1, h, w, hf, wf, int(class_index),
                                   mask.data_ptr(), _lib.stream_ptr(dev))
    _lib.check(rc, "isx_roi_rasterize")
    return mask


def roi_query(embeddings: Tensor, mask: Tensor, class_index: int = 1) -> Tensor:
    """Query vector(s) of an ROI: the mean of the embedding cells whose mask value is `class_index`.

    embeddings: float32 `B x E x h x w` (what `predict_step` returns, `models/embedding.py:57-76`) or
    `E x h x w`; mask: int64 `h x w` (one ROI for every image) or `B x h x w`.  Returns float32
    `B x E` (or `E`), zero for an image whose mask has no such cell; feed it to
    `EmbeddingStore.search`."""
    _lib.require_cuda(embeddings, "embeddings")
    _lib.require_cuda(mask, "mask")
    squeeze = embeddings.ndim == 3
    emb = embeddings.unsqueeze(0) if squeeze else embeddings
    if emb.ndim != 4 or emb.dtype != torch.float32:
        raise ValueError(f"embeddings must be float32 B x E x h x w, got {embeddings.dtype} {tuple(embeddings.shape)}")
    b, e, h, w = emb.shape
    if mask.dtype != torch.int64 or tuple(mask.shape) not in ((h, w), (b, h, w)):
        raise ValueError(f"mask must be int64 {h}x{w} or {b}x{h}x{w}, got {mask.dtype} {tuple(mask.shape)}")
    if mask.device != emb.device:
        raise ValueError(f"embeddings and mask are on different devices ({emb.device}, {mask.device})")
    emb = emb.contiguous()
    mask = mask.contiguous()
    out = torch.empty((b, e), dtype=torch.float32, device=emb.device)
    with torch.cuda.device(emb.device):
        rc = _lib.load().isx_masked_pool(emb.data_ptr(), b, e, h, w, mask.data_ptr(), int(mask.ndim == 3), int(class_index),
                                         out.data_ptr(), _lib.stream_ptr(emb.device))
    _lib.check(rc, "isx_masked_pool")
    return out[0] if squeeze else out


def roi_cells(embeddings: Tensor, mask: Tensor, class_index: int = 1) -> tuple[Tensor, Tensor]:
    """The ROI's cells as a multi-vector query: the multi-vector counterpart of `roi_query`.

    embeddings: float32 `B x E x h x w` (or `E x h x w`); mask: int64 `h x w` (one ROI for every image)
    or `B x h x w`.  Returns (cells bf16 `M x E`, sets int64 `B + 1`): the rows of `maps_to_rows` whose
    cell's mask value is `class_index`, image by image in row-major cell order, and the offsets of each
    image's rows (an image without such a cell gives an empty set).  Pass them as `queries, sets` to
    `EmbeddingStore.search_images_maxsim`."""
    from imagescry_b200.store_format import maps_to_rows

    _lib.require_cuda(embeddings, "embeddings")
    _lib.require_cuda(mask, "mask")
    emb = embeddings.unsqueeze(0) if embeddings.ndim == 3 else embeddings
    if emb.ndim != 4 or emb.dtype != torch.float32:
        raise ValueError(f"embeddings must be float32 B x E x h x w, got {embeddings.dtype} {tuple(embeddings.shape)}")
    b, e, h, w = emb.shape
    if mask.dtype != torch.int64 or tuple(mask.shape) not in ((h, w), (b, h, w)):
        raise ValueError(f"mask must be int64 {h}x{w} or {b}x{h}x{w}, got {mask.dtype} {tuple(mask.shape)}")
    if mask.device != emb.device:
        raise ValueError(f"embeddings and mask are on different devices ({emb.device}, {mask.device})")
    covered = (mask == class_index).expand(b, h, w).reshape(b, h * w)
    cells = maps_to_rows(emb)[covered.reshape(-1)]
    sets = torch.zeros(b + 1, dtype=torch.int64, device=emb.device)
    sets[1:] = covered.sum(dim=1).cumsum(0)
    return cells, sets


__all__: Sequence[str] = ("create_roi_mask", "polygon_edges", "roi_cells", "roi_query")
