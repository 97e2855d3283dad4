/*
 * imagescry_b200 — C ABI of the B200-native sift path (libimagescry_b200.so).
 *
 * The reference (libertininick/imagescry) is pure Python and has no FFI layer; its seams on this
 * path are Python callables (SURVEY.md §8b).  Each entry point below replaces the arithmetic behind
 * one of those seams and is what a ctypes binding in the reference would call (INTEGRATION.md shows
 * the stubs).  Citations are /root/reference/src/imagescry/<file>:<line>.
 *
 * Conventions
 *   - every pointer except `workspace`-free host out-params is a DEVICE pointer on the current device;
 *   - all functions are asynchronous on `stream` (a cudaStream_t passed as void*; NULL = legacy
 *     default stream), re-entrant, and own no device memory: the caller allocates outputs and
 *     workspaces (sizes from the *_workspace_bytes functions);
 *   - return value: ISX_OK, or a negative code with a per-thread message from isx_last_error();
 *   - no function reads or writes host copies of the data; there is no CPU fallback.
 */
#ifndef IMAGESCRY_B200_H_
#define IMAGESCRY_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ISX_ABI_VERSION 1

/* status codes */
#define ISX_OK 0
#define ISX_ERR_INVALID_ARG (-1)
#define ISX_ERR_CUDA (-2)
#define ISX_ERR_UNSUPPORTED (-3)
#define ISX_ERR_WORKSPACE (-4)

/* tile layouts */
#define ISX_LAYOUT_NCHW 0 /* planar: what ImageBatch.images holds (data.py:29-41)          */
#define ISX_LAYOUT_NHWC 1 /* interleaved: what a decoder / PIL hands over (image/io.py:41-52) */

/* element types */
#define ISX_DTYPE_U8 0
#define ISX_DTYPE_F32 1
#define ISX_DTYPE_BF16 2

typedef void* isx_stream_t;

/* ---- library ------------------------------------------------------------------------------ */
int isx_abi_version(void);
const char* isx_last_error(void);
/* SM count and compute capability of the current device (host out-params). */
int isx_device_info(int* sm_count, int* cc_major, int* cc_minor);

/* ---- stage 1: tile preprocessing ------------------------------------------------------------
 * Replaces image/transforms.py:78-126 `resize` (bilinear, align_corners=False, no antialias),
 * image/transforms.py:16-74 `normalize_per_channel` and their composition
 * models/embedding.py:150-165 `EfficientNetEmbedder.preprocess`, plus the HWC->CHW step of
 * image/io.py:52 / data.py:456-459 when layout == ISX_LAYOUT_NHWC.
 *
 * Geometry: input tiles B x C x H x W (or B x H x W x C), output B x C x outH x outW, always NCHW.
 * outH == H and outW == W means "no resize"; otherwise every output pixel is the bilinear sample
 * of the input, bit-identical to torch-CPU's upsample_bilinear2d, and is never materialised
 * between the statistics pass and the apply pass.
 */

/* Bytes of scratch isx_preprocess_stats needs for C channels. */
size_t isx_preprocess_stats_workspace_bytes(int C);

/* Per-channel batch mean and unbiased std over (batch, height, width) of the (resized) tiles,
 * transforms.py:62-65.  uint8 tiles without resize are reduced exactly in integers; every other
 * case accumulates in fp64.  Results are rounded once to fp32: mean[C], std[C]. */
int isx_preprocess_stats(const void* in, int in_dtype, int layout, int B, int C, int H, int W,
                         int outH, int outW, float* mean, float* std, void* workspace,
                         size_t workspace_bytes, isx_stream_t stream);

/* out = clip((resize(x) - mean) / (std + eps), lo, hi), transforms.py:68-72, fp32 arithmetic with
 * IEEE division (bit-identical to the reference given the same statistics).
 * mean/std hold stat_batch x C floats, stat_batch in {1, B} ("#B C 1 1" broadcasting).
 * out_dtype: ISX_DTYPE_F32 (reference behaviour) or ISX_DTYPE_BF16 (rounded from the fp32 value). */
int isx_preprocess_apply(const void* in, int in_dtype, int layout, int B, int C, int H, int W,
                         int outH, int outW, const float* mean, const float* std, int stat_batch,
                         float eps, int has_lo, float lo, int has_hi, float hi, void* out,
                         int out_dtype, isx_stream_t stream);

/* resize only (transforms.py:78-126): out fp32 NCHW = bilinear(in). */
int isx_resize_bilinear(const void* in, int in_dtype, int layout, int B, int C, int H, int W,
                        int outH, int outW, float* out, isx_stream_t stream);

/* Patch tiling (BASELINE.json north_star, stage 1: "with resize and patch tiling"; the reference has
 * no counterpart — its only "patches" are feature-map cells, SURVEY.md §8c — so the semantics are the
 * restatement oracle/oracle.py::preprocess_patches: cut every image into patch x patch windows at
 * `stride` (full windows only: ny = (img_h - patch) / stride + 1, likewise nx), treat the windows as the
 * tile batch of models/embedding.py:150-165 and preprocess them as above).  The windows are index
 * arithmetic inside both passes' reads: no patch tensor is materialised.
 * images: uint8, n_img x img_h x img_w x 3 (NHWC) or n_img x 3 x img_h x img_w (NCHW); C must be 3.
 * out: (n_img * ny * nx) x 3 x outH x outW, patches in (image, py, px) order; batch statistics are
 * over ALL patches (overlapping pixels count once per patch that holds them). */
int isx_preprocess_patches_stats(const void* images, int layout, int n_img, int C, int img_h, int img_w, int patch,
                                 int stride, int outH, int outW, float* mean, float* std, void* workspace,
                                 size_t workspace_bytes, isx_stream_t stream);
int isx_preprocess_patches_apply(const void* images, int layout, int n_img, int C, int img_h, int img_w, int patch,
                                 int stride, int outH, int outW, const float* mean, const float* std, float eps,
                                 int has_lo, float lo, int has_hi, float hi, void* out, int out_dtype,
                                 isx_stream_t stream);

/* ---- stage 2: L2-normalise (+ pool) + PCA projection ------------------------------------------
 * Replaces models/embedding.py:74 `F.normalize(x, p=2, dim=1)`, data.py:112-118
 * `get_flat_vectors`, models/decomposition.py:79-91 `PCA.forward` and the reshape/permute of
 * models/pipelines.py:82-84, fused: the B x E x h x w feature map is read once.
 */

/* Bytes of the packed projection operand for F features and k components. */
size_t isx_project_packed_bytes(int F, int k);

/* Pack PCA weights once per fitted model: component_vectors element (f, j) is read at
 * comps[f * ld_f + j * ld_k] (the reference stores a transposed view: ld_f = 1, ld_k = F),
 * feature_means is F floats.  Writes bf16 hi/lo splits (K-major, k x F each) and the fp32 bias
 * -(means . comps) into `packed`. */
int isx_project_pack(const float* feature_means, const float* comps, int F, int k, int64_t ld_f,
                     int64_t ld_k, void* packed, size_t packed_bytes, isx_stream_t stream);

size_t isx_l2norm_project_workspace_bytes(int B, int E, int h, int w, int k, int pool);

/* fmap: fp32 B x E x h x w (NCHW, contiguous).
 * pool == 0: out is fp32 (B*h*w) x k row-major, i.e. B x k x h x w viewed with NHWC strides —
 *            exactly the memory pipelines.py:82-84 returns.
 * pool == 1: spatial mean of the normalised cells, then the projection: out is fp32 B x k.
 * normalize == 0 skips the L2 step (plain PCA.transform of h*w == 1 rows: fmap is n x F). */
int isx_l2norm_project(const float* fmap, int B, int E, int h, int w, int pool, int normalize,
                       const void* packed, int k, float* out, void* workspace,
                       size_t workspace_bytes, isx_stream_t stream);

/* Same contract with ONE fp16 tensor pass instead of the three-pass bf16 split: feature values and
 * weights are rounded to fp16 (11-bit significand; |x| saturates at 65504), fp32 accumulation.
 * Error relative to a row's norm is ~1e-5 (bar: 1e-3); the kernel then runs at the HBM roofline
 * instead of the tensor one.  Shapes the staged kernel cannot take fall back to the exact kernels. */
int isx_l2norm_project_fp16(const float* fmap, int B, int E, int h, int w, int pool, int normalize,
                            const void* packed, int k, float* out, void* workspace,
                            size_t workspace_bytes, isx_stream_t stream);

/* Stand-alone per-cell L2 normalisation, models/embedding.py:74 `F.normalize(x, p=2, dim=1)` as
 * `EmbeddingModule.predict_step` (:57-76) returns it: out[b][e][c] = fmap[b][e][c] /
 * max(||fmap[b][:][c]||_2, eps), IEEE division.  fmap, out: fp32 B x E x h x w (NCHW, contiguous,
 * distinct buffers).  One pass: 4 bytes read + 4 written per element. */
int isx_l2norm_cells(const float* fmap, int B, int E, int h, int w, float eps, float* out, isx_stream_t stream);

/* ---- PCA.fit moments (models/decomposition.py:94-148) -------------------------------------------
 * mean[F] = column means of x (n x F fp32, row-major; :116) and cov[F x F] = Xc^T Xc / (n - 1) with
 * Xc = x - mean centred in fp32 as the reference does (:119).  The eigenvectors / eigenvalues of cov
 * are the right singular vectors / s^2 / (n - 1) the reference takes from its SVD (:122-125). */
size_t isx_pca_moments_workspace_bytes(int64_t n, int F);
int isx_pca_moments(const float* x, int64_t n, int F, float* mean, float* cov, void* workspace,
                    size_t workspace_bytes, isx_stream_t stream);

/* ---- stage 3: exhaustive cosine k-NN -----------------------------------------------------------
 * No reference counterpart (SURVEY.md §0.2); semantics are the composition of the reference's
 * idioms: normalize(q) . normalize(e) with F.normalize's eps (embedding.py:74) and a stable
 * (score descending, index ascending) top-k.
 */

/* rnorm[i] = 1 / max(||x_i||_2, eps) for the rows of a bf16 matrix n x d (fp32 accumulation). */
int isx_row_rnorm_bf16(const void* x, int64_t n, int d, float eps, float* rnorm, isx_stream_t stream);

/* Store build from the reference's embedding BLOBs (storage/models.py:94-129: float32, C-order
 * C x H x W; bulk read storage/operations.py:108-144).  maps: fp32 n x C x hw (hw = H*W).
 * pool == 0: rows = bf16 (n*hw) x C, one row per feature-map cell in data.py:112-118's
 *            get_flat_vectors order (row = image * hw + cell);
 * pool == 1: rows = bf16 n x C, the spatial mean of every map. */
int isx_maps_to_rows_bf16(const float* maps, int64_t n, int C, int hw, int pool, void* rows, isx_stream_t stream);

size_t isx_knn_workspace_bytes(int64_t n, int q, int d, int k);

/* store: bf16 n x d row-major; queries: bf16 q x d row-major; *_rnorm from isx_row_rnorm_bf16.
 * out_scores fp32 q x k, out_idx int32 q x k = index_base + local row.  Rows are ordered by
 * (score desc, index asc); if n < k the tail is (-inf, -1).  The q x n score matrix never exists
 * in memory: top-k selection is fused into the GEMM epilogue. */
int isx_knn_search(const void* store, const float* store_rnorm, int64_t n, const void* queries,
                   const float* query_rnorm, int q, int d, int k, int64_t index_base,
                   float* out_scores, int32_t* out_idx, void* workspace, size_t workspace_bytes,
                   isx_stream_t stream);

/* Extended form.  flags:
 *   ISX_KNN_CONTINUE      the workspace holds the running top-k lists of a previous call with the same
 *                         q and k (same queries): this call adds another block of store rows to them —
 *                         a store that arrives in pieces (ring / chunked all-gather) is searched
 *                         without ever gathering partial results;
 *   ISX_KNN_NO_FINALIZE   more blocks follow: outputs are not written (may be NULL);
 *   ISX_KNN_EXCLUDE_SELF  query row r IS store row query_index_base + r (all-pairs graph) and is never
 *                         its own neighbour;
 *   ISX_KNN_PACKED        out_scores receives q x k 8-byte records {fp32 score, int32 index} instead of
 *                         two arrays (out_idx unused): what ONE all-gather moves between shards.
 * isx_knn_workspace_bytes depends on (q, k) only, so one workspace serves every block. */
#define ISX_KNN_CONTINUE 1
#define ISX_KNN_NO_FINALIZE 2
#define ISX_KNN_EXCLUDE_SELF 4
#define ISX_KNN_PACKED 8
int isx_knn_search_ex(const void* store, const float* store_rnorm, int64_t n, const void* queries,
                      const float* query_rnorm, int q, int d, int k, int64_t index_base,
                      int64_t query_index_base, int flags, float* out_scores, int32_t* out_idx,
                      void* workspace, size_t workspace_bytes, isx_stream_t stream);

/* Row-sharded search whose finalising pass IS the gather: this rank's q x k packed records are stored
 * straight into slot `slot` of every rank's g x q x k gather buffer over NVLink.  peer_bufs is a HOST
 * array of n_peers device pointers (peer-mapped memory, e.g. torch symmetric memory / cuMem IPC; entry
 * `slot` is this rank's own buffer).  No collective library call is involved; the caller runs a
 * cross-rank barrier before isx_topk_merge_packed reads its buffer.  flags: ISX_KNN_CONTINUE and
 * ISX_KNN_EXCLUDE_SELF as above. */
int isx_knn_search_scatter(const void* store, const float* store_rnorm, int64_t n, const void* queries,
                           const float* query_rnorm, int q, int d, int k, int64_t index_base,
                           int64_t query_index_base, int flags, void* const* peer_bufs, int n_peers, int slot,
                           void* workspace, size_t workspace_bytes, isx_stream_t stream);

/* Merge g partial results (scores, idx: g x q x k, e.g. the NCCL all-gather of every shard's
 * local top-k) into q x k with the same ordering.  idx < 0 marks padding. */
int isx_topk_merge(const float* scores, const int32_t* idx, int g, int q, int k, float* out_scores,
                   int32_t* out_idx, isx_stream_t stream);
/* Same for packed records (g x q x k x {fp32 score, int32 index}, ISX_KNN_PACKED). */
int isx_topk_merge_packed(const void* records, int g, int q, int k, float* out_scores, int32_t* out_idx,
                          isx_stream_t stream);

/* Image-level (grouped) search: the k most similar GROUPS of rows, e.g. the images of a store with
 * one row per feature-map cell.  row_group: int32 n, the group id (>= 0) of every store row; groups
 * need not be contiguous or sorted.  A group's score is the best cosine score of its rows (the same
 * score isx_knn_search computes) and its representative is its first row in (score desc, index asc)
 * order.  out_scores fp32 q x k, out_rows int32 q x k (index_base + local row of the representative),
 * out_groups int32 q x k, ordered by the representatives' (score desc, index asc); if fewer than k
 * groups exist the tail is (-inf, -1, -1).  Selection is fused into the search kernel like the
 * row-level top-k; the workspace is sized by isx_knn_workspace_bytes. */
int isx_knn_search_grouped(const void* store, const float* store_rnorm, const int32_t* row_group, int64_t n,
                           const void* queries, const float* query_rnorm, int q, int d, int k, int64_t index_base,
                           float* out_scores, int32_t* out_rows, int32_t* out_groups,
                           void* workspace, size_t workspace_bytes, isx_stream_t stream);
/* Merge g grouped partial results (e.g. every shard's isx_knn_search_grouped output, gathered) into
 * the k best groups per query, ordered as above.  records: int32 g x q x k x 3
 * {fp32 score bits, global row, group}; row < 0 marks padding.  A group present in several partial
 * lists (an image cut by a shard boundary) comes out once, with its best row. */
int isx_topk_merge_grouped(const int32_t* records, int g, int q, int k, float* out_scores,
                           int32_t* out_rows, int32_t* out_groups, isx_stream_t stream);

/* ---- ROI masks on the feature-map grid (SURVEY.md 8f-4) ---------------------------------------
 * geometry.py:14-65 `create_roi_mask`: rasterio.features.rasterize(shapes, out_shape=(hf, wf),
 * transform=Affine.scale(w / wf, h / hf), fill=0, all_touched=True) * class_index.  rasterio / GDAL
 * are third-party and absent from the reference tree; the rule implemented is "a cell is burned when
 * its open rectangle shares positive area with a polygon" (cells that only touch a polygon along an
 * edge or corner stay 0), which reproduces tests/test_geometry.py:10-52 and the docstring example.
 *
 * edges: fp32 [n_edges][4] = (x0, y0, x1, y1) in IMAGE coordinates, the closed rings (exterior and
 * holes) of polygon p occupying edges [poly_offsets[p], poly_offsets[p + 1]).  mask: int64 fmap_h x
 * fmap_w, class_index where burned, else 0 (Int64[H W], geometry.py:19). */
int isx_roi_rasterize(const float* edges, const int32_t* poly_offsets, int n_poly, int image_h, int image_w,
                      int fmap_h, int fmap_w, int64_t class_index, int64_t* mask, isx_stream_t stream);

/* Masked pooling: out[b][e] = mean over the cells c with mask[c] == class_index of fmap[b][e][c]
 * (0 when no cell matches).  fmap: fp32 B x E x h x w, what predict_step returns
 * (models/embedding.py:57-76); mask: int64 h x w shared by all images (mask_per_image == 0) or
 * B x h x w.  The result is the ROI's query vector for isx_knn_search.  No reference code. */
int isx_masked_pool(const float* fmap, int B, int E, int h, int w, const int64_t* mask, int mask_per_image,
                    int64_t class_index, float* out, isx_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* IMAGESCRY_B200_H_ */
