"""Exhaustive cosine k-NN over a bf16 embedding store (stage 3 of the sift path).

The reference has no search entry point (SURVEY.md §3.5); this module adds one on top of what its
store holds (`storage/models.py:94-129`: float32 C×H×W BLOBs → rows of a bf16 matrix).  Semantics:
`normalize(q) @ normalize(e).T` with `F.normalize`'s eps (`models/embedding.py:74`), top-k ordered by
(score descending, index ascending).

Single GPU:   EmbeddingStore(embeddings).search(queries, k)
Several GPUs: ShardedEmbeddingStore — rows are split contiguously over the ranks of a
              `torch.distributed` group (one process per GPU); every rank searches its shard with the
              fused tcgen05 kernel, whose finalising pass stores the rank's packed (score, index)
              records into every rank's gather buffer over NVLink (peer-mapped symmetric memory; ONE
              NCCL all-gather of the same records as the fallback); every rank merges its buffer.
              All-pairs graphs shard the queries and rotate the store through all-gathers while the
              running top-k lists stay in the kernel's workspace.  Preprocessing and projection
              shard by batch and need no collective.
"""

from __future__ import annotations

import math
import numbers

import torch
from torch import Tensor

from imagescry_b200 import _lib

MAX_K = 128
# fp8 search: candidates the E4M3 scan passes to the exact re-score by default, the most the scan's
# fast selection (k <= 16) keeps
FP8_CANDIDATES = 16
# range search: a store's first call sizes its record buffer for RANGE_HITS_PER_QUERY hits per query,
# later calls for the hits per query of the store's previous call of the same kind (search or graph)
# plus RANGE_HEADROOM, never below RANGE_MIN_CAPACITY records; a call that overflows reruns once at its
# exact count
RANGE_HITS_PER_QUERY = 16
RANGE_HEADROOM = 1.25
RANGE_MIN_CAPACITY = 4096


def shard_range(num_rows: int, world_size: int, rank: int) -> tuple[int, int]:
    """Contiguous row range [begin, end) owned by `rank`: sizes differ by at most one row."""
    if world_size < 1 or not (0 <= rank < world_size):
        raise ValueError(f"invalid rank {rank} for world size {world_size}")
    base, rem = divmod(num_rows, world_size)
    begin = rank * base + min(rank, rem)
    return begin, begin + base + (1 if rank < rem else 0)


def row_rnorm(x: Tensor, eps: float = 1e-12) -> Tensor:
    """fp32 `1 / max(||row||, eps)` of a bf16 matrix (the denominator of `F.normalize`)."""
    _lib.require_cuda(x, "x")
    if x.dtype != torch.bfloat16 or x.ndim != 2 or not x.is_contiguous():
        raise ValueError("row_rnorm expects a contiguous 2-D bfloat16 tensor")
    n, d = x.shape
    out = torch.empty(n, dtype=torch.float32, device=x.device)
    if n:
        with _lib.on_device(x) as stream:
            rc = _lib.load().isx_row_rnorm_bf16(x.data_ptr(), n, d, eps, out.data_ptr(), stream)
        _lib.check(rc, "isx_row_rnorm_bf16")
    return out


def fp8_width(d: int) -> int:
    """Row width in bytes of the E4M3 copy of d-wide rows: d rounded up to 16 (16-byte TMA rows)."""
    return (d + 15) // 16 * 16


def quantize_e4m3(x: Tensor) -> tuple[Tensor, Tensor]:
    """E4M3 copy of a bf16 matrix for the fp8 scan (`isx_quantize_rows_e4m3`): every row scaled by the
    power of two that puts its largest |x| in (224, 448], rounded to nearest even and zero-padded to
    `fp8_width(d)` bytes.  Returns (uint8 N×d16 E4M3 bit patterns, fp32 `1 / max(‖row‖, eps)` of the
    E4M3 values)."""
    _lib.require_cuda(x, "x")
    if x.dtype != torch.bfloat16 or x.ndim != 2 or not x.is_contiguous():
        raise ValueError("quantize_e4m3 expects a contiguous 2-D bfloat16 tensor")
    n, d = x.shape
    d16 = fp8_width(d)
    out = torch.empty((n, d16), dtype=torch.uint8, device=x.device)
    rn = torch.empty(n, dtype=torch.float32, device=x.device)
    if n:
        with _lib.on_device(x, out, rn) as stream:
            rc = _lib.load().isx_quantize_rows_e4m3(x.data_ptr(), n, d, d16, out.data_ptr(), rn.data_ptr(), stream)
        _lib.check(rc, "isx_quantize_rows_e4m3")
    return out, rn


def merge_topk(scores: Tensor, indices: Tensor, k: int | None = None) -> tuple[Tensor, Tensor]:
    """Merge G partial results (G×Q×k fp32 scores, G×Q×k int32 indices; index < 0 = padding) into
    Q×k, ordered by (score desc, index asc)."""
    _lib.require_cuda(scores, "scores")
    if scores.shape != indices.shape or scores.ndim != 3:
        raise ValueError("scores and indices must both be G×Q×k")
    g, q, kk = scores.shape
    k = kk if k is None else k
    if k != kk:
        raise ValueError(f"k={k} does not match the partial lists' width {kk}")
    s = scores.contiguous().float()
    i = indices.contiguous().to(torch.int32)
    out_s = torch.empty((q, k), dtype=torch.float32, device=s.device)
    out_i = torch.empty((q, k), dtype=torch.int32, device=s.device)
    if q:
        with _lib.on_device(s, i) as stream:
            rc = _lib.load().isx_topk_merge(s.data_ptr(), i.data_ptr(), g, q, k, out_s.data_ptr(), out_i.data_ptr(), stream)
        _lib.check(rc, "isx_topk_merge")
    return out_s, out_i


def merge_topk_packed(records: Tensor, k: int | None = None) -> tuple[Tensor, Tensor]:
    """Merge G partial results held as packed records (G×Q×k int64: low word = fp32 score bits, high
    word = int32 index, what `EmbeddingStore.search_packed` writes and ONE all-gather moves) into
    (scores fp32 Q×k, indices int32 Q×k), ordered by (score desc, index asc)."""
    _lib.require_cuda(records, "records")
    if records.ndim != 3 or records.dtype != torch.int64:
        raise ValueError("records must be a G×Q×k int64 tensor")
    g, q, kk = records.shape
    k = kk if k is None else k
    if k != kk:
        raise ValueError(f"k={k} does not match the partial lists' width {kk}")
    r = records.contiguous()
    out_s = torch.empty((q, k), dtype=torch.float32, device=r.device)
    out_i = torch.empty((q, k), dtype=torch.int32, device=r.device)
    if q:
        with _lib.on_device(r) as stream:
            rc = _lib.load().isx_topk_merge_packed(r.data_ptr(), g, q, k, out_s.data_ptr(), out_i.data_ptr(), stream)
        _lib.check(rc, "isx_topk_merge_packed")
    return out_s, out_i


def pack_records(scores: Tensor, indices: Tensor) -> Tensor:
    """(fp32 score, int32 index) → int64 records, little-endian {score bits, index} like the kernel's
    8-byte records (host-side helper for tests and CPU plumbing; not on the search path)."""
    words = torch.stack([scores.contiguous().float().view(torch.int32), indices.to(torch.int32)], dim=-1)
    return words.contiguous().view(torch.int64).squeeze(-1)


def unpack_records(records: Tensor) -> tuple[Tensor, Tensor]:
    """int64 records → (fp32 scores, int32 indices); inverse of `pack_records`."""
    words = records.contiguous().view(torch.int32).view(*records.shape, 2)
    return words[..., 0].contiguous().view(torch.float32), words[..., 1].contiguous()


def group_offsets(groups, num_rows: int) -> Tensor:
    """Validate a store's image layout and return it as `row_offsets` (int64 CPU, images + 1 entries):
    image i owns rows [offsets[i], offsets[i + 1]).  `groups` is an int `c` (every image has c
    consecutive rows; num_rows % c == 0) or a 1-D integer tensor of row offsets from 0 to num_rows,
    non-decreasing (`store_from_mixed_blobs`)."""
    if isinstance(groups, bool):
        raise ValueError("groups must be an int (rows per image) or a 1-D tensor of row offsets")
    if isinstance(groups, int):
        if groups < 1 or num_rows % groups:
            raise ValueError(f"groups={groups} rows per image must be >= 1 and divide the store's {num_rows} rows")
        return torch.arange(0, num_rows + 1, groups, dtype=torch.int64)
    if not isinstance(groups, Tensor) or groups.ndim != 1 or groups.dtype.is_floating_point or groups.dtype == torch.bool:
        raise ValueError("groups must be an int (rows per image) or a 1-D integer tensor of row offsets")
    off = groups.detach().to(device="cpu", dtype=torch.int64)
    if off.numel() < 1 or int(off[0]) != 0 or int(off[-1]) != num_rows:
        raise ValueError(f"row offsets must run from 0 to the store's {num_rows} rows")
    if bool((off[1:] < off[:-1]).any()):
        raise ValueError("row offsets must be non-decreasing")
    if off.numel() - 1 >= 2**31:
        raise ValueError("at most 2^31 - 1 images")
    return off


def row_groups(offsets: Tensor, begin: int, end: int) -> Tensor:
    """int32 image id of every row in [begin, end) under `offsets` (CPU)."""
    rows = torch.arange(begin, end, dtype=torch.int64)
    return (torch.searchsorted(offsets, rows, right=True) - 1).to(torch.int32)


def image_cells(rows: Tensor, images: Tensor, first_row: Tensor) -> Tensor:
    """Cell of every hit inside its image: representative row - the image's first row (int64;
    -1 where images < 0, i.e. padding).  `first_row[i]` is image i's first row in the rows' numbering."""
    rows = rows.to(torch.int64)
    img = images.to(torch.int64)
    valid = img >= 0
    cells = rows - first_row.to(rows.device)[img.clamp(min=0)]
    return torch.where(valid, cells, torch.full_like(cells, -1))


def merge_topk_groups(records: Tensor, k: int | None = None) -> tuple[Tensor, Tensor, Tensor]:
    """Merge G grouped partial results held as G×Q×k×3 int32 records {fp32 score bits, row, group}
    (row < 0 = padding) into the k best groups per query: (scores fp32 Q×k, rows int32 Q×k, groups
    int32 Q×k), each group once, ordered by (score desc, row asc)."""
    _lib.require_cuda(records, "records")
    if records.ndim != 4 or records.shape[3] != 3 or records.dtype != torch.int32:
        raise ValueError("records must be a G×Q×k×3 int32 tensor")
    g, q, kk, _ = records.shape
    k = kk if k is None else k
    if k != kk:
        raise ValueError(f"k={k} does not match the partial lists' width {kk}")
    r = records.contiguous()
    out_s = torch.empty((q, k), dtype=torch.float32, device=r.device)
    out_r = torch.empty((q, k), dtype=torch.int32, device=r.device)
    out_g = torch.empty((q, k), dtype=torch.int32, device=r.device)
    if q:
        with _lib.on_device(r) as stream:
            rc = _lib.load().isx_topk_merge_grouped(r.data_ptr(), g, q, k, out_s.data_ptr(), out_r.data_ptr(),
                                                    out_g.data_ptr(), stream)
        _lib.check(rc, "isx_topk_merge_grouped")
    return out_s, out_r, out_g


def pack_group_records(scores: Tensor, rows: Tensor, groups: Tensor) -> Tensor:
    """(fp32 score, int32 row, int32 group) Q×k → Q×k×3 int32 records, the form one all-gather moves."""
    return torch.stack([scores.contiguous().float().view(torch.int32), rows.to(torch.int32), groups.to(torch.int32)], dim=-1)


def gather_group_records(records: Tensor, group=None) -> Tensor:
    """All-gather every rank's Q×k×3 grouped records: returns G×Q×k×3 (one collective)."""
    import torch.distributed as dist

    world = dist.get_world_size(group)
    q, k, three = records.shape
    out = torch.empty((world * q, k, three), dtype=records.dtype, device=records.device)
    dist.all_gather_into_tensor(out, records.contiguous(), group=group)
    return out.view(world, q, k, three)


def maxsim_block_plan(offsets: Tensor, num_queries: int, budget_bytes: int) -> list[tuple[int, int]]:
    """Image-aligned blocks of a multi-vector search (`search_images_maxsim`): `offsets` (images + 1
    row offsets) → [(first image, end image)) in order, covering every image, each block's Q × images
    fp32 cell-max matrix within `budget_bytes` and at least one image per block (an image whose column
    alone exceeds the budget gets a block of its own)."""
    if isinstance(budget_bytes, bool) or not isinstance(budget_bytes, int) or budget_bytes < 1:
        raise ValueError(f"budget_bytes must be a positive int, got {budget_bytes!r}")
    images = len(offsets) - 1
    per = max(1, budget_bytes // max(1, 4 * num_queries))
    return [(i, min(images, i + per)) for i in range(0, images, per)]


def combine_cut_columns(ids: Tensor, columns: Tensor, image: int) -> Tensor:
    """Cell-max column of an image cut by shard boundaries: the element-wise max of every gathered
    column (`columns` R×Q fp32) whose id (`ids` R) is `image`.  A max of maxima is exact, so the result
    is the column the unsharded store computes."""
    if ids.ndim != 1 or columns.ndim != 2 or columns.shape[0] != ids.shape[0]:
        raise ValueError("ids must be R and columns R×Q")
    pick = ids == image
    if not bool(pick.any()):
        raise ValueError(f"no column of image {image}")
    return columns[pick].amax(dim=0)


def range_threshold(threshold) -> float:
    """The range search's threshold as the fp32 value the kernel compares against (a finite float)."""
    if isinstance(threshold, Tensor):
        ok = threshold.numel() == 1 and threshold.dtype.is_floating_point
    else:  # Python and numpy numbers; bool is a number to Python, not a threshold
        ok = isinstance(threshold, numbers.Real) and not isinstance(threshold, bool)
    if not ok:
        raise ValueError(f"threshold must be a real number, got {threshold!r}")
    t = float(torch.tensor(float(threshold), dtype=torch.float32))
    if not math.isfinite(t):
        raise ValueError(f"threshold must be finite in float32, got {threshold!r}")
    return t


def range_capacity(hits_per_query: float, num_queries: int) -> int:
    """Record capacity of a range search's first run, from the expected hits per query."""
    return max(RANGE_MIN_CAPACITY, math.ceil(hits_per_query * RANGE_HEADROOM * num_queries))


def range_retry_capacity(count: int, capacity: int) -> int | None:
    """The capacity of the one rerun a range search needs, or None: the hit set is deterministic, so a
    rerun at exactly `count` records holds every hit."""
    return count if count > capacity else None


def range_empty(num_queries: int, device) -> tuple[Tensor, Tensor, Tensor]:
    """CSR of a range search without hits: (offsets int64 Q + 1, indices int64 [0], scores fp32 [0])."""
    return (torch.zeros(num_queries + 1, dtype=torch.int64, device=device), torch.empty(0, dtype=torch.int64, device=device),
            torch.empty(0, dtype=torch.float32, device=device))


def range_sort(records: Tensor, num_queries: int, hits: int) -> tuple[Tensor, Tensor, Tensor]:
    """Ordering pass of a range search (`isx_knn_range_sort`): N×3 int32 records {query, row, score
    bits} (row < 0 = padding) holding `hits` real records → CSR (offsets int64 Q + 1, indices int64,
    scores fp32), each query's hits ordered by (score desc, row asc)."""
    if records.ndim != 2 or records.shape[1] != 3 or records.dtype != torch.int32:
        raise ValueError("records must be an N×3 int32 tensor")
    _lib.require_cuda(records, "records")
    dev = records.device
    if num_queries == 0:
        return range_empty(0, dev)
    r = records.contiguous()
    offsets = torch.empty(num_queries + 1, dtype=torch.int64, device=dev)
    rows = torch.empty(hits, dtype=torch.int32, device=dev)
    scores = torch.empty(hits, dtype=torch.float32, device=dev)
    lib = _lib.load()
    with torch.cuda.device(dev):
        ws = torch.empty(max(int(lib.isx_knn_range_sort_workspace_bytes(r.shape[0], num_queries)), 256),
                         dtype=torch.uint8, device=dev)
    with _lib.on_device(r, offsets, ws) as stream:
        rc = lib.isx_knn_range_sort(r.data_ptr(), r.shape[0], num_queries, offsets.data_ptr(), rows.data_ptr(),
                                    scores.data_ptr(), ws.data_ptr(), ws.numel(), stream)
    _lib.check(rc, "isx_knn_range_sort")
    return offsets, rows.to(torch.int64), scores


def gather_range_records(records: Tensor, count: int, group=None) -> tuple[Tensor, int]:
    """All-gather every rank's first `count` range records (N×3 int32): one all-gather of the counts,
    one of the records padded to the largest count with row = -1.  Returns (world·max×3, total hits)."""
    import torch.distributed as dist

    world = dist.get_world_size(group)
    counts = torch.empty(world, dtype=torch.int64, device=records.device)
    dist.all_gather_into_tensor(counts, torch.tensor([count], dtype=torch.int64, device=records.device), group=group)
    counts = counts.tolist()
    width = max(counts)
    padded = torch.full((width, 3), -1, dtype=torch.int32, device=records.device)
    padded[:count] = records[:count]
    out = torch.empty((world * width, 3), dtype=torch.int32, device=records.device)
    dist.all_gather_into_tensor(out, padded, group=group)
    return out, sum(counts)


def _as_bf16_matrix(x: Tensor, name: str) -> Tensor:
    """bf16, contiguous, and — the kernel's TMA rows are 16-byte units — zero-padded to a multiple of
    8 features.  Zero features change neither dot products nor norms, so cosine scores are unchanged
    (the reference's PCA picks `num_components` from `min_explained_variance`: widths like 37 are
    normal, `decomposition.py:128-137`)."""
    _lib.require_cuda(x, name)
    if x.ndim != 2:
        raise ValueError(f"{name} must be 2-D (rows × features), got shape {tuple(x.shape)}")
    if not x.dtype.is_floating_point:
        raise ValueError(f"{name} must be a floating-point tensor, got {x.dtype}")
    d = x.shape[1]
    if d % 8:
        out = torch.zeros((x.shape[0], (d + 7) // 8 * 8), dtype=torch.bfloat16, device=x.device)
        out[:, :d] = x
        return out
    return x.to(torch.bfloat16).contiguous()


class EmbeddingStore:
    """A device-resident N×d bf16 embedding matrix with its inverse row norms.

    Vectors are kept as given (not re-rounded after normalisation): the kernel multiplies bf16×bf16
    products exactly, accumulates in fp32 and applies both inverse norms in the epilogue.

    A store may be searched from several CUDA streams: the scratch workspace (running top-k lists,
    per-query locks and bounds) is cached per stream.

    `groups` describes which rows belong to one image (a per-cell store has one row per feature-map
    cell): an int `c` (rows [i·c, (i+1)·c) are image i) or a 1-D int64 tensor of `row_offsets`
    (image i owns rows [offsets[i], offsets[i + 1])).  It enables `search_images`.

    `fp8=True` also keeps an E4M3 copy of the rows (`embeddings_e4m3`, N × `fp8_width(dim)` bytes, with
    its inverse norms `rnorm_e4m3`), built once here: N·d16 + 4N more bytes of device memory.  It
    enables `search_fp8`."""

    def __init__(self, embeddings: Tensor, *, index_base: int = 0, groups: int | Tensor | None = None,
                 fp8: bool = False) -> None:
        if embeddings.ndim != 2:
            raise ValueError(f"embeddings must be 2-D (rows × features), got shape {tuple(embeddings.shape)}")
        offsets = None if groups is None else group_offsets(groups, embeddings.shape[0])
        self.num_features = embeddings.shape[1]
        self.embeddings = _as_bf16_matrix(embeddings, "embeddings")
        self.index_base = int(index_base)
        self.rnorm = row_rnorm(self.embeddings)
        self._workspaces: dict[int, Tensor] = {}
        self.row_group: Tensor | None = None
        if offsets is not None:
            self._set_groups(offsets, 0, self.index_base)
        self.embeddings_e4m3: Tensor | None = None
        self.rnorm_e4m3: Tensor | None = None
        if fp8:
            self.embeddings_e4m3, self.rnorm_e4m3 = quantize_e4m3(self.embeddings)

    def _set_groups(self, offsets: Tensor, begin: int, row0: int) -> None:
        """Rows of this store are rows [begin, begin + len) of the layout `offsets`; a hit's row in
        the results is row0 + its layout row."""
        self.row_group = row_groups(offsets, begin, begin + len(self)).to(self.device)
        self.group_first_row = (offsets[:-1] + row0).to(self.device)
        self._layout = (offsets, begin)

    def __len__(self) -> int:
        return self.embeddings.shape[0]

    @property
    def dim(self) -> int:
        """Row width in memory (`num_features` rounded up to a multiple of 8)."""
        return self.embeddings.shape[1]

    @property
    def device(self) -> torch.device:
        return self.embeddings.device

    def _ws(self, nbytes: int) -> Tensor:
        key = torch.cuda.current_stream(self.device).cuda_stream
        ws = self._workspaces.get(key)
        if ws is None or ws.numel() < nbytes:
            ws = torch.empty(nbytes, dtype=torch.uint8, device=self.device)
            self._workspaces[key] = ws
        return ws

    def _queries(self, queries: Tensor) -> Tensor:
        if queries.ndim != 2:
            raise ValueError(f"queries must be 2-D (rows × features), got shape {tuple(queries.shape)}")
        if queries.shape[1] != self.num_features and queries.shape[1] != self.dim:
            raise ValueError(f"queries have {queries.shape[1]} features, the store has {self.num_features}")
        q = _as_bf16_matrix(queries, "queries")
        if q.device != self.device:
            raise ValueError(f"queries are on {q.device}, the store is on {self.device}")
        return q

    def search_block(
        self, rows: Tensor, rows_rnorm: Tensor, index_base: int, q: Tensor, q_rnorm: Tensor, k: int, *, flags: int = 0,
        query_index_base: int = 0, out_a: Tensor | None = None, out_b: Tensor | None = None,
    ) -> None:
        """One `isx_knn_search_ex` call: search the bf16 block `rows` (global indices from `index_base`)
        for the prepared queries `q`, on this store's per-stream workspace.  With `KNN_CONTINUE` the
        block is added to the running lists of the previous call (same q and k)."""
        lib = _lib.load()
        nq = q.shape[0]
        with torch.cuda.device(self.device):  # the size depends on the device's SM count
            ws_bytes = max(int(lib.isx_knn_workspace_bytes(max(rows.shape[0], 1), nq, q.shape[1], k)), 256)
            ws = self._ws(ws_bytes)
        with _lib.on_device(rows, rows_rnorm, q, q_rnorm, out_a, out_b, ws) as stream:
            rc = lib.isx_knn_search_ex(
                rows.data_ptr(), rows_rnorm.data_ptr(), rows.shape[0], q.data_ptr(), q_rnorm.data_ptr(), nq, q.shape[1], k,
                int(index_base), int(query_index_base), int(flags), None if out_a is None else out_a.data_ptr(),
                None if out_b is None else out_b.data_ptr(), ws.data_ptr(), ws.numel(), stream,
            )
        _lib.check(rc, "isx_knn_search_ex")

    def _check_k(self, k: int) -> None:
        if not (1 <= k <= MAX_K):
            raise ValueError(f"k must be between 1 and {MAX_K}, got {k}")

    def search_raw(self, queries: Tensor, k: int, *, query_rnorm: Tensor | None = None) -> tuple[Tensor, Tensor]:
        """Local top-k: fp32 scores Q×k and int32 global indices Q×k (padding: -inf / -1)."""
        q = self._queries(queries)
        self._check_k(k)
        nq = q.shape[0]
        scores = torch.empty((nq, k), dtype=torch.float32, device=self.device)
        idx = torch.empty((nq, k), dtype=torch.int32, device=self.device)
        if nq == 0:
            return scores, idx
        qr = row_rnorm(q) if query_rnorm is None else query_rnorm
        self.search_block(self.embeddings, self.rnorm, self.index_base, q, qr, k, out_a=scores, out_b=idx)
        return scores, idx

    def search_packed(self, queries: Tensor, k: int, *, query_rnorm: Tensor | None = None, out: Tensor | None = None) -> Tensor:
        """Local top-k as Q×k packed int64 records {fp32 score, int32 global index}: the form a
        row-sharded search all-gathers in ONE collective (`merge_topk_packed` consumes it)."""
        q = self._queries(queries)
        self._check_k(k)
        nq = q.shape[0]
        rec = torch.empty((nq, k), dtype=torch.int64, device=self.device) if out is None else out
        if nq == 0:
            return rec
        qr = row_rnorm(q) if query_rnorm is None else query_rnorm
        self.search_block(self.embeddings, self.rnorm, self.index_base, q, qr, k, flags=_lib.KNN_PACKED, out_a=rec)
        return rec

    def search(self, queries: Tensor, k: int) -> tuple[Tensor, Tensor]:
        """Cosine top-k of every query row: (scores fp32 Q×k, indices int64 Q×k)."""
        scores, idx = self.search_raw(queries, k)
        return scores, idx.to(torch.int64)

    def search_images_raw(self, queries: Tensor, k: int) -> tuple[Tensor, Tensor, Tensor]:
        """Local image-level top-k: (scores fp32 Q×k, representative rows int32 Q×k in the store's
        global numbering, images int32 Q×k); padding (-inf, -1, -1)."""
        if self.row_group is None:
            raise ValueError("search_images needs a store built with groups= (rows per image or row offsets)")
        q = self._queries(queries)
        self._check_k(k)
        nq = q.shape[0]
        scores = torch.empty((nq, k), dtype=torch.float32, device=self.device)
        rows = torch.empty((nq, k), dtype=torch.int32, device=self.device)
        images = torch.empty((nq, k), dtype=torch.int32, device=self.device)
        if nq == 0:
            return scores, rows, images
        qr = row_rnorm(q)
        lib = _lib.load()
        with torch.cuda.device(self.device):
            ws = self._ws(max(int(lib.isx_knn_workspace_bytes(max(len(self), 1), nq, q.shape[1], k)), 256))
        with _lib.on_device(self.embeddings, q, qr, ws, self.row_group) as stream:
            rc = lib.isx_knn_search_grouped(
                self.embeddings.data_ptr(), self.rnorm.data_ptr(), self.row_group.data_ptr(), len(self), q.data_ptr(),
                qr.data_ptr(), nq, q.shape[1], k, self.index_base, scores.data_ptr(), rows.data_ptr(), images.data_ptr(),
                ws.data_ptr(), ws.numel(), stream,
            )
        _lib.check(rc, "isx_knn_search_grouped")
        return scores, rows, images

    def search_images(self, queries: Tensor, k: int) -> tuple[Tensor, Tensor, Tensor]:
        """The k most similar IMAGES of every query row: (scores fp32 Q×k, images int64 Q×k, cells
        int64 Q×k).  An image scores its best cell (the cosine of `search`); `cells` is that cell's
        position in the image (its row - the image's first row; the lowest such row on ties).  Ordered
        by (score desc, row asc); if the store has fewer than k images the tail is (-inf, -1, -1)."""
        scores, rows, images = self.search_images_raw(queries, k)
        return scores, images.to(torch.int64), image_cells(rows, images, self.group_first_row)

    def _maxsim_prepare(self, queries: Tensor, sets, k: int):
        """Checks of a multi-vector search: (prepared queries, set offsets int64 CPU)."""
        if self.row_group is None:
            raise ValueError("search_images_maxsim needs a store built with groups= (rows per image or row offsets)")
        self._check_k(k)
        q = self._queries(queries)
        return q, group_offsets(sets, q.shape[0])

    def _maxsim_records(self, q: Tensor, qr: Tensor, set_off: Tensor, k: int, budget_bytes: int, *,
                        shard: bool = False) -> tuple[list[Tensor], list[tuple[int, Tensor]]]:
        """Per image-aligned block of this store's rows: one `isx_knn_maxsim` and one
        `isx_maxsim_sets_topk`.  Returns the blocks' S×k packed records and, with `shard`, the
        (image, cell-max column) of the store's first and last image when a shard boundary cuts them;
        those images are left out of the records."""
        offsets, begin = self._layout
        n, nq, num_sets = len(self), q.shape[0], len(set_off) - 1
        if n == 0:
            return [], []
        end = begin + n
        lo = int(torch.searchsorted(offsets, torch.tensor([begin]), right=True)[0]) - 1
        hi = int(torch.searchsorted(offsets, torch.tensor([end - 1]), right=True)[0])  # one past the last image
        local = offsets[lo:hi + 1].clamp(begin, end) - begin
        cut_first = shard and int(offsets[lo]) < begin
        cut_last = shard and int(offsets[hi]) > end
        plan = maxsim_block_plan(local, nq, budget_bytes)
        lib = _lib.load()
        with torch.cuda.device(self.device):
            ws = self._ws(_lib.KNN_RANGE_WORKSPACE_BYTES)
        cell = torch.empty(nq * max(b - a for a, b in plan), dtype=torch.float32, device=self.device)
        sets_dev = set_off.to(self.device)
        records, edges = [], []
        for a, b in plan:
            r0, r1, ng = int(local[a]), int(local[b]), b - a
            cm = cell[: nq * ng].view(nq, ng)
            rows = self.embeddings[r0:r1]
            with _lib.on_device(rows, q, qr, cm, ws, self.row_group) as stream:
                rc = lib.isx_knn_maxsim(
                    rows.data_ptr(), self.rnorm[r0:].data_ptr(), self.row_group[r0:].data_ptr(), r1 - r0, q.data_ptr(),
                    qr.data_ptr(), nq, q.shape[1], lo + a, ng, cm.data_ptr(), ws.data_ptr(), ws.numel(), stream,
                )
            _lib.check(rc, "isx_knn_maxsim")
            first, last = cut_first and a == 0, cut_last and b == len(local) - 1
            c0 = 1 if first else 0
            c1 = max(c0, ng - 1 if last else ng)
            if first:
                edges.append((lo, cm[:, 0].clone()))
            if last:
                edges.append((hi - 1, cm[:, ng - 1].clone()))
            records.append(self._maxsim_sets_topk(cm, qr, c0, c1, lo + a, sets_dev, num_sets, k))
        return records, edges

    def _maxsim_sets_topk(self, cm: Tensor, qr: Tensor, c0: int, c1: int, group_base: int, sets_dev: Tensor,
                          num_sets: int, k: int) -> Tensor:
        """One `isx_maxsim_sets_topk` over columns [c0, c1) of the cell-max matrix `cm`: S×k records."""
        rec = torch.empty((num_sets, k), dtype=torch.int64, device=self.device)
        nq, ng = cm.shape
        with _lib.on_device(cm, qr, sets_dev, rec) as stream:
            rc = _lib.load().isx_maxsim_sets_topk(cm.data_ptr(), qr.data_ptr(), nq, ng, c0, c1, sets_dev.data_ptr(), num_sets,
                                                  k, group_base, rec.data_ptr(), stream)
        _lib.check(rc, "isx_maxsim_sets_topk")
        return rec

    def search_images_maxsim(self, queries: Tensor, sets, k: int, *, budget_bytes: int = 1 << 30) -> tuple[Tensor, Tensor]:
        """Multi-vector image search (late interaction, "MaxSim"): the k best images for every query SET.

        `sets` says which query rows form one set: an int m (consecutive sets of m rows; Q % m == 0) or a
        1-D offsets tensor from 0 to Q (set s = rows [offsets[s], offsets[s + 1]); sets may be empty).
        Image I scores, for the set S,

            score(S, I) = (1 / |S|) · Σ_{c ∈ S} max_{r ∈ I} cos(q_c, e_r)

        where the cosine of (c, r) is bit for bit the fp32 score `search` reports, so each term is the
        `search_images` score of image I for row c.  The terms are summed in fp32 in ascending row order
        and the sum is divided (correctly rounded) by |S|: the result does not depend on the store's
        blocks or tiles.  Returns (scores fp32 S×k, images int64 S×k), ordered by (score desc, image
        asc) and padded with (-inf, -1) when there are fewer than k images; an empty set gets padding
        only.  Needs a store built with `groups=`.

        The per-(row, image) maxima are formed in the search kernel's epilogue (`isx_knn_maxsim`): the
        Q × N score matrix never exists, only Q × images fp32 maxima, in image-aligned blocks of at most
        `budget_bytes` each (at least one image per block)."""
        q, set_off = self._maxsim_prepare(queries, sets, k)
        num_sets = len(set_off) - 1
        nq = q.shape[0]
        if nq == 0 or len(self) == 0:
            return (torch.full((num_sets, k), float("-inf"), dtype=torch.float32, device=self.device),
                    torch.full((num_sets, k), -1, dtype=torch.int64, device=self.device))
        records, _ = self._maxsim_records(q, row_rnorm(q), set_off, k, budget_bytes)
        scores, images = merge_topk_packed(torch.stack(records), k)
        return scores, images.to(torch.int64)

    def scan_fp8(self, queries: Tensor, k: int) -> tuple[Tensor, Tensor]:
        """The fp8 scan alone (`isx_knn_search_fp8`): the top-k of the E4M3 copies of the queries and
        the store by their cosine, (scores fp32 Q×k, int32 global indices Q×k), padding (-inf, -1).
        These are candidates; the scores are those of the quantized rows."""
        if self.embeddings_e4m3 is None:
            raise ValueError("search_fp8 needs a store built with fp8=True")
        q = self._queries(queries)
        self._check_k(k)
        nq = q.shape[0]
        scores = torch.empty((nq, k), dtype=torch.float32, device=self.device)
        idx = torch.empty((nq, k), dtype=torch.int32, device=self.device)
        if nq == 0:
            return scores, idx
        q8, qr8 = quantize_e4m3(q)
        lib = _lib.load()
        d16 = q8.shape[1]
        with torch.cuda.device(self.device):
            ws = self._ws(max(int(lib.isx_knn_workspace_bytes(max(len(self), 1), nq, d16, k)), 256))
        with _lib.on_device(self.embeddings_e4m3, q8, qr8, scores, idx, ws) as stream:
            rc = lib.isx_knn_search_fp8(
                self.embeddings_e4m3.data_ptr(), self.rnorm_e4m3.data_ptr(), len(self), q8.data_ptr(), qr8.data_ptr(), nq,
                d16, k, self.index_base, scores.data_ptr(), idx.data_ptr(), ws.data_ptr(), ws.numel(), stream,
            )
        _lib.check(rc, "isx_knn_search_fp8")
        return scores, idx

    def rescore(self, queries: Tensor, candidates: Tensor, k: int, *, query_rnorm: Tensor | None = None) -> tuple[Tensor, Tensor]:
        """Exact re-score of candidate lists (`isx_knn_rescore`): `candidates` Q×kc global rows (any order,
        -1 = none, 1 <= kc <= 128) → the best k by the bf16 cosine `search` computes, (scores fp32 Q×k,
        int32 global indices Q×k) ordered by (score desc, index asc), padding (-inf, -1)."""
        q = self._queries(queries)
        self._check_k(k)
        if candidates.ndim != 2 or candidates.shape[0] != q.shape[0] or not (1 <= candidates.shape[1] <= MAX_K):
            raise ValueError(f"candidates must be Q×kc with 1 <= kc <= {MAX_K}, got shape {tuple(candidates.shape)}")
        if candidates.dtype.is_floating_point or candidates.dtype == torch.bool:
            raise ValueError("candidates must be an integer tensor of global rows")
        nq, kc = candidates.shape
        cand = candidates.to(device=self.device, dtype=torch.int32).contiguous()
        scores = torch.empty((nq, k), dtype=torch.float32, device=self.device)
        idx = torch.empty((nq, k), dtype=torch.int32, device=self.device)
        if nq == 0:
            return scores, idx
        qr = row_rnorm(q) if query_rnorm is None else query_rnorm
        with _lib.on_device(self.embeddings, q, qr, cand, scores, idx) as stream:
            rc = _lib.load().isx_knn_rescore(
                self.embeddings.data_ptr(), self.rnorm.data_ptr(), len(self), q.data_ptr(), qr.data_ptr(), nq, q.shape[1],
                cand.data_ptr(), kc, self.index_base, k, scores.data_ptr(), idx.data_ptr(), stream,
            )
        _lib.check(rc, "isx_knn_rescore")
        return scores, idx

    def search_fp8_raw(self, queries: Tensor, k: int, *, candidates: int = FP8_CANDIDATES) -> tuple[Tensor, Tensor]:
        """`search_fp8` with int32 global indices."""
        if self.embeddings_e4m3 is None:
            raise ValueError("search_fp8 needs a store built with fp8=True")
        if isinstance(k, bool) or isinstance(candidates, bool) or not (1 <= k <= candidates <= MAX_K):
            raise ValueError(f"search_fp8 needs 1 <= k <= candidates <= {MAX_K}, got k={k} candidates={candidates}")
        q = self._queries(queries)
        nq = q.shape[0]
        if nq == 0 or len(self) == 0:
            return (torch.full((nq, k), float("-inf"), dtype=torch.float32, device=self.device),
                    torch.full((nq, k), -1, dtype=torch.int32, device=self.device))
        _, cand = self.scan_fp8(q, candidates)
        return self.rescore(q, cand, k)

    def search_fp8(self, queries: Tensor, k: int, *, candidates: int = FP8_CANDIDATES) -> tuple[Tensor, Tensor]:
        """Cosine top-k through the fp8 tensor-core path: (scores fp32 Q×k, indices int64 Q×k).

        An E4M3 scan of the store picks the `candidates` best rows of every query by the cosine of the
        quantized rows; those are re-scored exactly from the bf16 rows and the best k returned, ordered
        by (score desc, index asc).  Every returned score is the fp32 cosine `search` computes for the
        pair (up to its fp32 summation order); only recall is approximate: a row of the exact top-k is
        missed when quantization moves it out of the candidates.  More candidates, more recall; 16 is
        the most the scan's fast selection keeps.  Needs a store built with `fp8=True`."""
        scores, idx = self.search_fp8_raw(queries, k, candidates=candidates)
        return scores, idx.to(torch.int64)

    def range_records(
        self, q: Tensor, q_rnorm: Tensor, threshold: float, *, flags: int = 0, query_index_base: int = 0,
        _capacity: int | None = None,
    ) -> tuple[Tensor, int]:
        """Unordered hits of a range search over this store for the prepared queries `q`: (N×3 int32
        records {query, global row, score bits}, N).  The buffer is sized from the hits per query of
        the store's previous call with the same flags; if the hits do not fit, the search runs once
        more with exactly as many records."""
        lib = _lib.load()
        nq = q.shape[0]
        hints = self.__dict__.setdefault("_range_hints", {})
        cap = range_capacity(hints.get(flags, RANGE_HITS_PER_QUERY), nq) if _capacity is None else _capacity
        count = torch.zeros(1, dtype=torch.int64, device=self.device)
        with torch.cuda.device(self.device):
            ws = self._ws(_lib.KNN_RANGE_WORKSPACE_BYTES)
        while True:
            records = torch.empty((cap, 3), dtype=torch.int32, device=self.device)
            with _lib.on_device(self.embeddings, q, q_rnorm, records, count, ws) as stream:
                rc = lib.isx_knn_range(
                    self.embeddings.data_ptr(), self.rnorm.data_ptr(), len(self), q.data_ptr(), q_rnorm.data_ptr(), nq,
                    q.shape[1], threshold, self.index_base, int(query_index_base), int(flags), records.data_ptr(), cap,
                    count.data_ptr(), ws.data_ptr(), ws.numel(), stream,
                )
            _lib.check(rc, "isx_knn_range")
            hits = int(count.item())
            retry = range_retry_capacity(hits, cap)
            if retry is None:
                break
            cap = retry
        if nq:
            hints[flags] = hits / nq
        if cap > 2 * hits + RANGE_MIN_CAPACITY:
            # a buffer sized for many more hits would stay allocated through the ordering pass
            return records[:hits].clone(), hits
        return records[:hits], hits

    def search_range(self, queries: Tensor, threshold: float) -> tuple[Tensor, Tensor, Tensor]:
        """Every store row whose cosine score with a query is >= `threshold` (rounded to float32), as CSR:
        (offsets int64 Q + 1, indices int64 M, scores fp32 M).  Query i's hits are
        indices[offsets[i]:offsets[i + 1]], ordered by (score desc, index asc); a score is bit for bit
        what `search` reports for the pair, so the hits are the prefix of a long enough `search`
        result whose scores are >= threshold."""
        t = range_threshold(threshold)
        q = self._queries(queries)
        nq = q.shape[0]
        if nq == 0 or len(self) == 0:
            return range_empty(nq, self.device)
        records, hits = self.range_records(q, row_rnorm(q), t)
        return range_sort(records, nq, hits)

    def range_graph(self, threshold: float) -> tuple[Tensor, Tensor, Tensor]:
        """ε-graph of the store: every OTHER row whose cosine score with a row is >= `threshold`, as the
        CSR of `search_range` with the store's own rows as queries (a row is never its own hit).  The
        counterpart of `knn_graph` for a fixed similarity instead of a fixed count."""
        t = range_threshold(threshold)
        n = len(self)
        if n == 0:
            return range_empty(0, self.device)
        records, hits = self.range_records(self.embeddings, self.rnorm, t, flags=_lib.KNN_EXCLUDE_SELF,
                                           query_index_base=self.index_base)
        return range_sort(records, n, hits)

    def knn_graph(self, k: int) -> tuple[Tensor, Tensor]:
        """All-pairs similarity graph (BASELINE.json config 5): the k nearest OTHER rows of every row,
        (scores N×k fp32, indices N×k int64).  One fused search with the store's own rows as queries;
        a row's own entry is skipped inside the kernel's selection (no k + 1 search, no post-filter)."""
        self._check_k(k)
        n = len(self)
        scores = torch.empty((n, k), dtype=torch.float32, device=self.device)
        idx = torch.empty((n, k), dtype=torch.int32, device=self.device)
        if n:
            self.search_block(
                self.embeddings, self.rnorm, self.index_base, self.embeddings, self.rnorm, k,
                flags=_lib.KNN_EXCLUDE_SELF, query_index_base=self.index_base, out_a=scores, out_b=idx,
            )
        return scores, idx.to(torch.int64)


def knn_graph(store: "EmbeddingStore", k: int) -> tuple[Tensor, Tensor]:
    """All-pairs similarity graph over a store: see `EmbeddingStore.knn_graph`."""
    return store.knn_graph(k)


def knn_search(embeddings: Tensor, queries: Tensor, k: int) -> tuple[Tensor, Tensor]:
    """One-shot convenience: build an `EmbeddingStore` and search it."""
    return EmbeddingStore(embeddings).search(queries, k)


def gather_records(records: Tensor, group=None) -> Tensor:
    """All-gather every rank's packed local top-k (Q×k int64): returns G×Q×k.  The ONE collective of
    a sharded search; backend-agnostic (NCCL over NVLink on GPUs, gloo in CPU tests)."""
    import torch.distributed as dist

    world = dist.get_world_size(group)
    q, k = records.shape
    # concatenation along dim 0 is the one output form every backend (NCCL, gloo) accepts
    out = torch.empty((world * q, k), dtype=records.dtype, device=records.device)
    dist.all_gather_into_tensor(out, records.contiguous(), group=group)
    return out.view(world, q, k)


def gather_partials(scores: Tensor, idx: Tensor, group=None) -> tuple[Tensor, Tensor]:
    """Two-array form of `gather_records` (kept for callers that hold separate score / index
    tensors): returns (G×Q×k scores, G×Q×k indices)."""
    import torch.distributed as dist

    world = dist.get_world_size(group)
    q, k = scores.shape
    all_s = torch.empty((world * q, k), dtype=scores.dtype, device=scores.device)
    all_i = torch.empty((world * q, k), dtype=idx.dtype, device=idx.device)
    dist.all_gather_into_tensor(all_s, scores.contiguous(), group=group)
    dist.all_gather_into_tensor(all_i, idx.contiguous(), group=group)
    return all_s.view(world, q, k), all_i.view(world, q, k)


def graph_chunk_plan(sizes: list[int], dim: int, budget_bytes: int) -> tuple[int, int]:
    """Chunking of the store rotation in `ShardedEmbeddingStore.knn_graph`: every step all-gathers
    rows [c, c + chunk) of every rank's shard.  Returns (chunk rows per rank, number of steps) such
    that the gathered buffer (world × chunk × dim bf16) stays within `budget_bytes`."""
    per = max(sizes)
    world = len(sizes)
    chunk = max(1, min(per, budget_bytes // max(1, world * dim * 2)))
    return chunk, (per + chunk - 1) // chunk if per else 0


class ShardedEmbeddingStore:
    """Row-sharded store over the ranks of a process group (one process per GPU).

    `local_embeddings` are this rank's rows; their global indices start at `index_base` (by default
    the contiguous partition of `shard_range`).  Queries are replicated on every rank.  `groups`
    (rows per image, or row offsets) describes the GLOBAL rows, as for `EmbeddingStore`; an image may
    be cut by a shard boundary."""

    def __init__(self, local_embeddings: Tensor, *, total_rows: int | None = None, index_base: int | None = None, group=None,
                 groups: int | Tensor | None = None, fp8: bool = False) -> None:
        import torch.distributed as dist

        self.group = group
        self.world_size = dist.get_world_size(group)
        self.rank = dist.get_rank(group)
        if index_base is None:
            if total_rows is None:
                raise ValueError("give either index_base or total_rows")
            begin, end = shard_range(total_rows, self.world_size, self.rank)
            if end - begin != local_embeddings.shape[0]:
                raise ValueError(
                    f"rank {self.rank} should hold rows [{begin}, {end}) but got {local_embeddings.shape[0]} rows"
                )
            index_base = begin
        self.total_rows = total_rows
        self.local = EmbeddingStore(local_embeddings, index_base=index_base, fp8=fp8)
        if groups is not None:
            if isinstance(groups, int) and not isinstance(groups, bool) and total_rows is None:
                raise ValueError("groups given as rows per image need total_rows")
            total = total_rows if total_rows is not None else int(torch.as_tensor(groups)[-1])
            offsets = group_offsets(groups, total)
            if index_base + len(self.local) > total:
                raise ValueError(f"rows [{index_base}, {index_base + len(self.local)}) exceed the layout's {total} rows")
            self.local._set_groups(offsets, index_base, 0)

    def search_images(self, queries: Tensor, k: int) -> tuple[Tensor, Tensor, Tensor]:
        """`EmbeddingStore.search_images` over the sharded store: local grouped search, ONE all-gather of
        the Q×k×3 int32 records {score, row, image}, grouped merge (an image cut by a shard boundary
        comes out once, with its best cell)."""
        s, r, g = self.local.search_images_raw(queries, k)
        merged_s, merged_r, merged_g = merge_topk_groups(gather_group_records(pack_group_records(s, r, g), self.group), k)
        return merged_s, merged_g.to(torch.int64), image_cells(merged_r, merged_g, self.local.group_first_row)

    def search_images_maxsim(self, queries: Tensor, sets, k: int, *, budget_bytes: int = 1 << 30) -> tuple[Tensor, Tensor]:
        """`EmbeddingStore.search_images_maxsim` over the sharded store, bit for bit the unsharded result.

        Every rank scores the images whose rows it holds entirely.  An image cut by a shard boundary is
        scored by the rank that holds its first row: every rank keeps the cell-max columns (Q floats)
        of its first and last image when a boundary cuts them, one all-gather moves those columns and
        their image ids, and the owner combines them by max (`combine_cut_columns`, exact) and scores
        the image with the same set-reduce kernel.  Then one all-gather of the S×k packed records and
        one merge."""
        import torch.distributed as dist

        st = self.local
        q, set_off = st._maxsim_prepare(queries, sets, k)
        num_sets, nq, dev = len(set_off) - 1, q.shape[0], st.device
        if nq == 0 or num_sets == 0:
            return (torch.full((num_sets, k), float("-inf"), dtype=torch.float32, device=dev),
                    torch.full((num_sets, k), -1, dtype=torch.int64, device=dev))
        qr = row_rnorm(q)
        records, edges = st._maxsim_records(q, qr, set_off, k, budget_bytes, shard=True)
        # rows of the edge exchange: int32 [image id or -1, Q fp32 bit patterns], first and last image
        send = torch.zeros((2, nq + 1), dtype=torch.int32, device=dev)
        send[:, 0] = -1
        for j, (image, col) in enumerate(edges[:2]):
            send[j, 0] = image
            send[j, 1:] = col.view(torch.int32)
        got = torch.empty((self.world_size * 2, nq + 1), dtype=torch.int32, device=dev)
        dist.all_gather_into_tensor(got, send, group=self.group)
        offsets, begin = st._layout
        for image, _ in edges:
            # the last image of this shard, cut at its end and starting here: this rank owns it
            if int(offsets[image]) >= begin and int(offsets[image + 1]) > begin + len(st):
                col = combine_cut_columns(got[:, 0], got[:, 1:].contiguous().view(torch.float32), image)
                records.append(st._maxsim_sets_topk(col.view(nq, 1), qr, 0, 1, image, set_off.to(dev), num_sets, k))
        if records:
            s, i = merge_topk_packed(torch.stack(records), k)
            mine = pack_records(s, i)
        else:
            mine = pack_records(torch.full((num_sets, k), float("-inf"), device=dev),
                                torch.full((num_sets, k), -1, dtype=torch.int32, device=dev))
        scores, images = merge_topk_packed(gather_records(mine, self.group), k)
        return scores, images.to(torch.int64)

    def search_fp8(self, queries: Tensor, k: int, *, candidates: int = FP8_CANDIDATES) -> tuple[Tensor, Tensor]:
        """`EmbeddingStore.search_fp8` over the sharded store (built with `fp8=True`): local fp8 scan and
        exact re-score, ONE all-gather of the packed records, merge.  The ranks merge exact scores: a
        returned score is bit for bit the one the unsharded store computes for the pair.  Each rank keeps
        its own `candidates`, a superset of the unsharded candidates (the scan's scores do not depend on
        the shard), so the result is the exact top-k of more candidates: never a worse row, sometimes a
        better one than the unsharded `search_fp8`."""
        s, i = self.local.search_fp8_raw(queries, k, candidates=candidates)
        merged_s, merged_i = merge_topk_packed(gather_records(pack_records(s, i), self.group), k)
        return merged_s, merged_i.to(torch.int64)

    def search_range(self, queries: Tensor, threshold: float) -> tuple[Tensor, Tensor, Tensor]:
        """`EmbeddingStore.search_range` over the sharded store: local range search with global rows, one
        all-gather of the per-rank hit counts, one of the records padded to the largest count, one
        ordering pass.  Every rank returns the same CSR."""
        t = range_threshold(threshold)
        q = self.local._queries(queries)
        nq = q.shape[0]
        if nq == 0:
            return range_empty(0, self.local.device)
        if len(self.local):
            records, hits = self.local.range_records(q, row_rnorm(q), t)
        else:
            records, hits = torch.empty((0, 3), dtype=torch.int32, device=self.local.device), 0
        gathered, total = gather_range_records(records, hits, self.group)
        return range_sort(gathered, nq, total)

    # ------------------------------------------------------------------ gather over peer memory
    def _peer_buffers(self, nq: int, k: int):
        """Symmetric (peer-mapped) gather buffers for Q×k results: [2 parities][G][Q][k] packed records
        on every rank, exchanged once through torch's symmetric-memory rendezvous.  With them the
        search's finalising pass stores this rank's records straight into every peer's buffer over
        NVLink (`isx_knn_search_scatter`): finalise + all-gather is ONE kernel of ours, followed by a
        device-side barrier.  Returns None when peer mapping is unavailable (gloo / no NVLink P2P /
        ISX_PEER_GATHER=0): the NCCL all-gather of `gather_records` is used instead."""
        import os

        import torch.distributed as dist

        key = (nq, k)
        cache = self.__dict__.setdefault("_peer_cache", {})
        if key in cache:
            return cache[key]
        entry = None
        if os.environ.get("ISX_PEER_GATHER", "1") != "0" and self.world_size <= 16 and self.local.device.type == "cuda":
            try:
                import torch.distributed._symmetric_memory as symm_mem

                group = self.group if self.group is not None else dist.group.WORLD
                buf = symm_mem.empty((2, self.world_size, nq, k), dtype=torch.int64, device=self.local.device)
                hdl = symm_mem.rendezvous(buf, group)
                ptrs = [int(p) for p in hdl.buffer_ptrs]
                if len(ptrs) == self.world_size and all(ptrs):
                    entry = {"buf": buf, "hdl": hdl, "ptrs": ptrs, "step": 0}
            except Exception as ex:  # no peer mapping on this system: NCCL carries the gather
                import sys

                print(f"imagescry_b200: symmetric-memory gather unavailable ({ex!r}); using the NCCL all-gather", file=sys.stderr)
        # every rank must take the same path
        flag = torch.tensor([1 if entry is not None else 0], dtype=torch.int32, device=self.local.device)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN, group=self.group)
        if int(flag.item()) == 0:
            entry = None
        cache[key] = entry
        return entry

    @property
    def gather_path(self) -> str:
        """"peer-store" once a search has used the symmetric-memory path, else "nccl"."""
        return "peer-store" if any(v is not None for v in self.__dict__.get("_peer_cache", {}).values()) else "nccl"

    def search_raw(self, queries: Tensor, k: int) -> tuple[Tensor, Tensor]:
        """(scores fp32 Q×k, GLOBAL indices int32 Q×k): local fused search whose finalising pass stores
        the packed (score, index) records into every rank's gather buffer over NVLink, a device-side
        barrier, merge.  Without peer-mapped memory: local search → ONE NCCL all-gather of the packed
        records → merge."""
        import ctypes

        q = self.local._queries(queries)
        self.local._check_k(k)
        nq = q.shape[0]
        peer = self._peer_buffers(nq, k) if nq else None
        if peer is None:
            sink = self.__dict__.get("_event_sink")
            if sink is not None:
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                qr0 = row_rnorm(q)
                e0.record()
                rec = self.local.search_packed(q, k, query_rnorm=qr0)
                e1.record()
                sink.append((e0, e1))
            else:
                rec = self.local.search_packed(q, k)
            return merge_topk_packed(gather_records(rec, self.group), k)
        lib = _lib.load()
        st = self.local
        qr = row_rnorm(q)
        parity = peer["step"] & 1
        peer["step"] += 1
        stride = self.world_size * nq * k * 8  # bytes of one parity's [G][Q][k] block
        arr = (ctypes.c_void_p * self.world_size)(*[p + parity * stride for p in peer["ptrs"]])
        with torch.cuda.device(st.device):
            ws_bytes = max(int(lib.isx_knn_workspace_bytes(max(len(st), 1), nq, st.dim, k)), 256)
            ws = st._ws(ws_bytes)
        sink = self.__dict__.get("_event_sink")
        with _lib.on_device(st.embeddings, q, qr, ws) as stream:
            if sink is not None:  # bench.py times the fused search + scatter kernel with CUDA events
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
            rc = lib.isx_knn_search_scatter(
                st.embeddings.data_ptr(), st.rnorm.data_ptr(), len(st), q.data_ptr(), qr.data_ptr(), nq, st.dim, k,
                st.index_base, 0, 0, arr, self.world_size, self.rank, ws.data_ptr(), ws.numel(), stream,
            )
            _lib.check(rc, "isx_knn_search_scatter")
            if sink is not None:
                e1.record()
                sink.append((e0, e1))
            # every rank's stores have landed once all ranks passed this barrier; the buffer of this
            # parity is rewritten two searches later, after every rank has passed the NEXT barrier,
            # i.e. after its merge of this one (stream order)
            peer["hdl"].barrier(channel=parity)
        return merge_topk_packed(peer["buf"][parity], k)

    def search(self, queries: Tensor, k: int) -> tuple[Tensor, Tensor]:
        s, i = self.search_raw(queries, k)
        return s, i.to(torch.int64)

    def knn_graph(self, k: int, *, gather: bool = True, budget_bytes: int = 2 << 30) -> tuple[Tensor, Tensor]:
        """All-pairs similarity graph over the sharded store (BASELINE.json config 5).

        The QUERIES are sharded — rank r answers for its own rows — and the STORE rotates: step by
        step every rank contributes the next chunk of its shard to one all-gather over NVLink and
        searches the gathered rows with `KNN_CONTINUE`, so the running top-k lists of its queries
        persist across all store blocks inside the search kernel's workspace.  No partial result is
        ever gathered or merged, and a row's own entry is skipped inside the kernel.

        gather=True  every rank returns the full graph (scores N×k fp32, indices N×k int64): one
                     final all-gather of the finished lists;
        gather=False a rank returns the lists of its own rows only (rows `shard_range(total, G, r)`)."""
        import torch.distributed as dist

        if self.total_rows is None:
            raise ValueError("knn_graph needs a store built with total_rows (the contiguous partition)")
        self.local._check_k(k)
        G, r = self.world_size, self.rank
        ranges = [shard_range(self.total_rows, G, g) for g in range(G)]
        sizes = [e - b for b, e in ranges]
        local, d, dev = self.local.embeddings, self.local.dim, self.local.device
        n_local = local.shape[0]
        chunk, steps = graph_chunk_plan(sizes, d, budget_bytes)
        scores = torch.empty((n_local, k), dtype=torch.float32, device=dev)
        idx = torch.empty((n_local, k), dtype=torch.int32, device=dev)
        uniform = all(sz == sizes[0] for sz in sizes)
        calls = []  # (rows, index_base) in search order
        first = True
        for step in range(steps):
            c0 = step * chunk
            cr = min(chunk, max(sizes) - c0)
            if n_local >= c0 + cr:
                send = local[c0:c0 + cr]
            else:  # shards differ by one row: pad the short ones
                send = torch.zeros((cr, d), dtype=local.dtype, device=dev)
                if n_local > c0:
                    send[: n_local - c0] = local[c0:]
            gathered = torch.empty((G * cr, d), dtype=local.dtype, device=dev)
            dist.all_gather_into_tensor(gathered, send.contiguous(), group=self.group)
            rn = row_rnorm(gathered)
            if uniform and steps == 1:
                blocks = [(0, G * cr, 0)]  # the gathered buffer IS the store in global row order
            else:
                blocks = [(g * cr, min(cr, max(0, sizes[g] - c0)), ranges[g][0] + c0) for g in range(G)]
                blocks = [b for b in blocks if b[1] > 0]
            for bi, (off, rows, base) in enumerate(blocks):
                last = step == steps - 1 and bi == len(blocks) - 1
                flags = _lib.KNN_EXCLUDE_SELF | (0 if first else _lib.KNN_CONTINUE) | (0 if last else _lib.KNN_NO_FINALIZE)
                if n_local:
                    self.local.search_block(
                        gathered[off:off + rows], rn[off:off + rows], base, local, self.local.rnorm, k, flags=flags,
                        query_index_base=ranges[r][0], out_a=scores if last else None, out_b=idx if last else None,
                    )
                first = False
                calls.append((rows, base))
        self._last_graph_calls = calls
        if not gather:
            return scores, idx.to(torch.int64)
        per = max(sizes)
        if not uniform:
            ps = torch.full((per, k), float("-inf"), dtype=torch.float32, device=dev)
            pi = torch.full((per, k), -1, dtype=torch.int32, device=dev)
            ps[:n_local], pi[:n_local] = scores, idx
            scores, idx = ps, pi
        all_s = torch.empty((G * per, k), dtype=torch.float32, device=dev)
        all_i = torch.empty((G * per, k), dtype=torch.int32, device=dev)
        dist.all_gather_into_tensor(all_s, scores, group=self.group)
        dist.all_gather_into_tensor(all_i, idx, group=self.group)
        if not uniform:
            keep = torch.cat([torch.arange(g * per, g * per + sizes[g], device=dev) for g in range(G)])
            all_s, all_i = all_s[keep], all_i[keep]
        return all_s, all_i.to(torch.int64)

    def replicate_queries(self, host_queries: Tensor) -> Tensor:
        """Replicated device copy of a (pinned) host query matrix without sending it over PCIe once
        per GPU: every rank uploads only its 1/G slice of the rows and one all-gather over NVLink
        completes the copy.  All ranks must pass the same `host_queries`; the returned tensor is a
        view of a staging buffer that the next call overwrites."""
        import torch.distributed as dist

        q, d = host_queries.shape
        per = (q + self.world_size - 1) // self.world_size
        dev = self.local.device
        staging = getattr(self, "_q_staging", None)
        if staging is None or staging.shape != (per * self.world_size, d) or staging.dtype != host_queries.dtype:
            staging = torch.empty((per * self.world_size, d), dtype=host_queries.dtype, device=dev)
            self._q_staging = staging
        b, e = min(q, self.rank * per), min(q, (self.rank + 1) * per)
        mine = staging[self.rank * per:self.rank * per + (e - b)]
        mine.copy_(host_queries[b:e], non_blocking=True)
        dist.all_gather_into_tensor(staging, staging[self.rank * per:(self.rank + 1) * per], group=self.group)
        return staging[:q]


class HostBatchSearch:
    """Streamed search of query batches that live in (pinned) HOST memory, for serving loops.

    `run(host_batches)` yields `(scores, indices)` per batch as PINNED HOST tensors (fp32 Q×k, int32
    Q×k global rows), in order.  The host→device copy of batch i + 1 and the device→host copy of
    batch i run on a copy stream (DMA engines, no SMs) while the neighbouring batch is searched on the
    caller's current stream, so the PCIe transfers cost no search time; with a row-sharded store every
    rank passes the same batches (each uploads them over its own PCIe link).  A yielded pair stays
    valid until the generator is advanced again.  The staging buffers (two device query buffers, two
    pinned result pairs) and the copy stream live as long as the object: keep it across calls.
    `store` is an `EmbeddingStore` or a `ShardedEmbeddingStore`."""

    def __init__(self, store, k: int) -> None:
        self.store = store
        local = store.local if isinstance(store, ShardedEmbeddingStore) else store
        self.device = local.device
        if self.device.type != "cuda":
            raise RuntimeError(f"HostBatchSearch needs a CUDA store (got {self.device}); there is no CPU path")
        local._check_k(k)
        self.k = k
        self._copy = torch.cuda.Stream(self.device)
        self._q_dev: list[Tensor | None] = [None, None]
        self._q_n = [0, 0]
        self._out_s: list[Tensor | None] = [None, None]
        self._out_i: list[Tensor | None] = [None, None]
        self._r_n = [0, 0]
        self._uploaded: list[torch.cuda.Event | None] = [None, None]    # H2D of the slot's queries finished
        self._searched: list[torch.cuda.Event | None] = [None, None]    # the search that read the slot finished
        self._downloaded: list[torch.cuda.Event | None] = [None, None]  # D2H of the slot's result finished
        self._keep: list[tuple | None] = [None, None]                    # device results until their D2H is done

    def _upload(self, slot: int, hb: Tensor) -> None:
        if hb.ndim != 2 or hb.device.type != "cpu":
            raise ValueError("host batches must be 2-D CPU tensors (pin them for asynchronous copies)")
        n = hb.shape[0]
        buf = self._q_dev[slot]
        if buf is None or buf.shape[0] < n or buf.shape[1] != hb.shape[1] or buf.dtype != hb.dtype:
            if self._searched[slot] is not None:
                self._searched[slot].synchronize()  # the old buffer is released: its last reader must be done
            self._q_dev[slot] = torch.empty((n, hb.shape[1]), dtype=hb.dtype, device=self.device)
        with torch.cuda.stream(self._copy):
            if self._searched[slot] is not None:
                self._copy.wait_event(self._searched[slot])  # the search that last read this device buffer
            self._q_dev[slot][:n].copy_(hb, non_blocking=True)
            ev = torch.cuda.Event()
            ev.record(self._copy)
        self._uploaded[slot] = ev
        self._q_n[slot] = n

    def _search(self, slot: int, compute) -> None:
        n, k = self._q_n[slot], self.k
        if self._out_s[slot] is None or self._out_s[slot].shape[0] < n:
            self._out_s[slot] = torch.empty((n, k), dtype=torch.float32).pin_memory()
            self._out_i[slot] = torch.empty((n, k), dtype=torch.int32).pin_memory()
        compute.wait_event(self._uploaded[slot])
        s, i = self.store.search_raw(self._q_dev[slot][:n], k)
        ev = torch.cuda.Event()
        ev.record(compute)
        self._searched[slot] = ev
        self._keep[slot] = (s, i)
        with torch.cuda.stream(self._copy):
            self._copy.wait_event(ev)
            self._out_s[slot][:n].copy_(s, non_blocking=True)
            self._out_i[slot][:n].copy_(i, non_blocking=True)
            done = torch.cuda.Event()
            done.record(self._copy)
        self._downloaded[slot] = done
        self._r_n[slot] = n

    def _collect(self, slot: int) -> tuple[Tensor, Tensor]:
        self._downloaded[slot].synchronize()
        self._keep[slot] = None
        return self._out_s[slot][: self._r_n[slot]], self._out_i[slot][: self._r_n[slot]]

    def run(self, host_batches):
        compute = torch.cuda.current_stream(self.device)
        it = iter(host_batches)
        try:
            current = next(it, None)
            if current is not None:
                self._upload(0, current)
            i = 0
            waiting = None  # the slot whose result has not been yielded yet
            while current is not None:
                slot = i & 1
                following = next(it, None)
                if following is not None:
                    self._upload(slot ^ 1, following)  # in flight while this batch is searched
                self._search(slot, compute)            # enqueued behind batch i - 1's search: no gap on the device
                if waiting is not None:
                    yield self._collect(waiting)       # batch i - 1: its host buffers are rewritten by batch i + 1
                waiting = slot
                current = following
                i += 1
            if waiting is not None:
                yield self._collect(waiting)
        finally:
            self._copy.synchronize()  # nothing of ours is in flight when the caller moves on


def search_host_batches(store, host_batches, k: int):
    """One-shot form of `HostBatchSearch(store, k).run(host_batches)`."""
    yield from HostBatchSearch(store, k).run(host_batches)
