// Stage 3 of the sift path: exhaustive cosine k-NN over a bf16 embedding store.
//
//   K0  row_rnorm_kernel   1 / max(||row||, eps) for the store and the queries (HBM-bound pass)
//   K4  knn_search_kernel  tcgen05 GEMM  S = Q . E^T  (bf16 operands from TMA-filled shared memory,
//                          fp32 accumulators in TMEM) with the per-query top-k fused into the
//                          epilogue: the Q x N score matrix never leaves the SM.
//   K5  topk_merge_kernel  finalises K4's running lists (scale by the queries' inverse norms, rebase
//                          the rows — as two arrays, packed records, or packed records stored into every
//                          peer's gather buffer over NVLink) and merges the partial lists of several GPUs.
//   fp8 search (isx_knn_search_fp8): K0q quantize_e4m3_kernel writes an E4M3 copy of the rows and its
//   inverse norms, K4 in its fp8 form (knn_search_fp8_kernel: the same body with kind::f8f6f4 MMAs
//   over 128-element k-blocks) picks candidates, K5r rescore_kernel re-scores them from the bf16 rows.
//
// There is no reference implementation of this stage (SURVEY.md §0.2); semantics follow
// oracle/oracle.py::cosine_knn: normalize(q) . normalize(e) with F.normalize's eps
// (/root/reference/src/imagescry/models/embedding.py:74), ordered by (score desc, index asc).
//
// K4 structure (one persistent CTA per SM; CTA pairs when there are at least two query blocks):
//   warp 0      TMA producer: query tile 128 x 64 and store tile 256 x 64 (bf16, 128B swizzle) per
//               k-block into a STAGES-deep shared-memory ring (short rows, d <= 256 and k <= 16: the
//               query tile stays resident for a whole item and the ring carries store tiles only)
//   warp 1      MMA issuer: one elected lane issues tcgen05.mma 128 x 256 x 16 (256 x 256 x 16 per
//               pair), accumulating a 128 x 256 fp32 tile in one of two TMEM accumulator stages
//   warp 2      TMEM allocation / deallocation
//   warps 4-7 (k <= 16: 4-11, two groups of four, each owning 128 of the tile's 256 columns)
//               epilogue: tcgen05.ld the finished tile 64 columns at a time (one query row per
//               thread), scale by the store rows' inverse norms (FMUL2), reject everything below the
//               row's running k-th best with one warp-uniform compare, append the rare survivors to a
//               per-row candidate buffer and prune that buffer warp-cooperatively (rank counting for
//               32 entries, bitonic sort for 256) when it is full.
// Work decomposition: items = (N-split, query block); a unit walks items in split-major order so
// that units running at the same time stream the same store rows and share them through L2.  At the
// end of an item every row's best k are merged (per-query lock, bitonic merge) into the query's
// running list in global memory, whose k-th best is the bound every later item starts from; a final
// pass scales the running lists by the queries' inverse norms.
// Diagnostics: -DISX_KNN_PROFILE (ISX_NVCC_EXTRA) makes every role count the cycles it waits.
#include "common.cuh"

#include <algorithm>
#include <cfloat>
#include <cmath>
#include <climits>
#include <cstdlib>

namespace isx {
namespace {

constexpr int BM = 128;  // queries per tile  (TMEM lanes)
constexpr int BN = 256;  // store rows per tile (TMEM columns)
constexpr int BK = 64;   // bf16 elements per k-block: 128 bytes = one swizzle row
constexpr int UMMA_K = 16;
constexpr int ACC_STAGES = 2;
constexpr int kEpilogueWarp0 = 4;
// Two groups of four epilogue warps: group g selects columns [128 g, 128 g + 128) of every tile with
// its own per-row thresholds and candidate buffers, i.e. it is a sub-split of the item and writes its
// own partial list.  Two warps per scheduler halve the epilogue time per tile and hide each other's
// TMEM / shared-memory latencies (d = 256: the epilogue, not the MMA, was the limiter with one group).
// Large k (256-entry candidate buffers in global memory, long sorts) keeps one group: there the
// second set of per-row lists costs more than the shorter fast path saves.  One group at small k
// measured slower (with the pipelined loads: d = 256 4.83 ms against 4.38, d = 64 4.57 against 3.64).
__host__ __device__ constexpr int epi_groups(int cap) { return cap <= 32 ? 2 : 1; }
__host__ __device__ constexpr int knn_threads(int cap) { return kEpilogueWarp0 * 32 + 128 * epi_groups(cap); }
constexpr int kMaxK = 128;
constexpr int kSmallK = 16;  // k <= kSmallK keeps candidate buffers in shared memory

constexpr uint32_t A_STAGE_BYTES = BM * BK * 2;  // 16 KB per CTA

struct KnnPlan {
  int mb;        // 128-query blocks
  long long nb;  // 256-row store blocks
  int splits;    // N-splits
  long long items;
  int grid;
};

// ncta = 2: CTA pairs (cta_group::2) — an M block is 256 queries and the schedulable units are SM pairs.
KnnPlan plan_knn(long long n, int q, int sms_total, int ncta) {
  KnnPlan p;
  const int sms = std::max(1, sms_total / ncta);
  p.mb = (q + BM * ncta - 1) / (BM * ncta);
  p.nb = (n + BN - 1) / BN;
  if (p.nb < 1) p.nb = 1;
  const long long max_s = std::max<long long>(1, std::min<long long>(p.nb, 4096));
  // Fewest splits whose item count fills whole waves of `sms` units to >= 97 %.  Items are kept
  // long: every item end costs a sort and a locked merge into the query's running list per row, and
  // (with the running lists) short items no longer buy better thresholds.
  int best_s = 1;
  double best_eff = -1.0;
  for (long long s = 1; s <= max_s; ++s) {
    const long long items = static_cast<long long>(p.mb) * s;
    const long long waves = (items + sms - 1) / sms;
    const double eff = static_cast<double>(items) / static_cast<double>(waves * sms);
    // keep items long enough to amortise the cold start of the running threshold
    const bool long_enough = (p.nb / s) >= 16 || s == 1;
    if (!long_enough) break;
    if (eff > best_eff + 1e-9) { best_eff = eff; best_s = static_cast<int>(s); }
    if (eff >= 0.97) break;
  }
  p.splits = best_s;
  p.items = static_cast<long long>(p.mb) * p.splits;
  p.grid = static_cast<int>(std::min<long long>(sms, p.items)) * ncta;
  return p;
}

// ------------------------------------------------------------------------------------------
// K0: inverse row norms
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
row_rnorm_kernel(const __nv_bfloat16* __restrict__ x, long long n, int d, float eps,
                 float* __restrict__ rnorm) {
  const int lane = threadIdx.x & 31;
  const long long warps = (static_cast<long long>(gridDim.x) * blockDim.x) >> 5;
  for (long long row = (static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5; row < n;
       row += warps) {
    const __nv_bfloat16* p = x + row * d;
    float ss = 0.f;
    if ((d & 7) == 0 && (reinterpret_cast<uintptr_t>(p) & 15u) == 0) {
      for (int i = lane * 8; i < d; i += 256) {
        const uint4 v = ld_nc_v4(p + i);
        const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const float lo = __uint_as_float(w[j] << 16), hi = __uint_as_float(w[j] & 0xFFFF0000u);
          ss = fmaf(lo, lo, ss);
          ss = fmaf(hi, hi, ss);
        }
      }
    } else {
      for (int i = lane; i < d; i += 32) {
        const float v = __bfloat162float(p[i]);
        ss = fmaf(v, v, ss);
      }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) ss += __shfl_xor_sync(kFullMask, ss, o);
    if (lane == 0) rnorm[row] = 1.0f / fmaxf(sqrtf(ss), eps);
  }
}

// ------------------------------------------------------------------------------------------
// K0q: E4M3 copy of bf16 rows for the fp8 scan.  One warp per row:
//   1. m = max |x|; the row is scaled by the power of two 2^e that puts m in (224, 448] (exact, and a
//      cosine does not see it), so every row uses the format's full range whatever its norm;
//   2. round to nearest even into E4M3 (cvt.rn.satfinite), zero-pad to d16 bytes (16-byte TMA rows);
//   3. rnorm = 1 / max(||q||, eps) of the E4M3 values q themselves.  Their squares are exact and their
//      sum is exact in fp64 (every q^2 is a multiple of 2^-18 below 2^18), so the norm is the correctly
//      rounded one, whatever the summation order.
// The fp8 scan therefore ranks by the exact cosine of the quantized rows, up to the fp32 accumulation
// of the tensor cores; rows that are power-of-two multiples of each other get identical bytes.  A zero
// row stays zero (e = 0) and gets 1 / eps, as in row_rnorm_kernel.
// ------------------------------------------------------------------------------------------
constexpr float kRnormEps = 1e-12f;  // F.normalize's eps, the value row_rnorm is called with

// exponent e with 224 < m * 2^e <= 448 for finite m > 0 (0 otherwise)
__device__ __forceinline__ int e4m3_row_exponent(float m) {
  if (!(m > 0.f) || isinf(m)) return 0;
  int ex;
  const float f = frexpf(m, &ex);  // m = f * 2^ex, f in [0.5, 1): 2f is m's significand
  return (f > 0.875f) ? 8 - ex : 9 - ex;
}

// value of a finite E4M3 byte (sign, 4 exponent bits with bias 7, 3 mantissa bits)
__device__ __forceinline__ float e4m3_to_f32(uint32_t b) {
  const uint32_t ex = (b >> 3) & 15u, man = b & 7u;
  const float mag = ex ? __uint_as_float(((ex + 120u) << 23) | (man << 20)) : static_cast<float>(man) * 0.001953125f;
  return (b & 0x80u) ? -mag : mag;
}

__global__ void __launch_bounds__(256)
quantize_e4m3_kernel(const __nv_bfloat16* __restrict__ x, long long n, int d, int d16, uint8_t* __restrict__ out,
                     float* __restrict__ rnorm) {
  const int lane = threadIdx.x & 31;
  const long long warps = (static_cast<long long>(gridDim.x) * blockDim.x) >> 5;
  const bool vec = (d & 7) == 0 && (reinterpret_cast<uintptr_t>(x) & 15u) == 0;
  for (long long row = (static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5; row < n;
       row += warps) {
    const __nv_bfloat16* p = x + row * d;
    uint8_t* o = out + row * d16;
    float m = 0.f;
    if (vec) {
      for (int i = lane * 8; i < d; i += 256) {
        const uint4 v = ld_nc_v4(p + i);
        const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
        for (int j = 0; j < 4; ++j) m = fmaxf(m, fmaxf(fabsf(__uint_as_float(w[j] << 16)), fabsf(__uint_as_float(w[j] & 0xFFFF0000u))));
      }
    } else {
      for (int i = lane; i < d; i += 32) m = fmaxf(m, fabsf(__bfloat162float(p[i])));
    }
#pragma unroll
    for (int o2 = 16; o2 > 0; o2 >>= 1) m = fmaxf(m, __shfl_xor_sync(kFullMask, m, o2));
    // 2^e in two factors (e reaches 157 for the smallest bf16 subnormals): each product is exact for
    // every element that does not end far below E4M3's smallest subnormal
    const int e = e4m3_row_exponent(m);
    const int e1 = e / 2;
    const float s1 = __int_as_float((127 + e1) << 23), s2 = __int_as_float((127 + e - e1) << 23);
    double ss = 0.0;
    auto quant2 = [&](float a, float b) -> uint16_t {
      const uint16_t r = cvt_e4m3x2(__fmul_rn(__fmul_rn(a, s1), s2), __fmul_rn(__fmul_rn(b, s1), s2));
      const double qa = e4m3_to_f32(r & 0xFFu), qb = e4m3_to_f32(r >> 8);
      ss = fma(qa, qa, ss);
      ss = fma(qb, qb, ss);
      return r;
    };
    if (vec) {
      // 8 elements (one 16-byte load, one 8-byte store) per lane and step; d % 8 == 0 and d16 % 16 == 0,
      // so a step is either all data or all padding
      for (int i = lane * 8; i < d16; i += 256) {
        uint4 v = make_uint4(0u, 0u, 0u, 0u);
        if (i < d) v = ld_nc_v4(p + i);
        const uint32_t w[4] = {v.x, v.y, v.z, v.w};
        uint32_t b[2];
#pragma unroll
        for (int j = 0; j < 2; ++j) {
          const uint16_t lo = quant2(__uint_as_float(w[2 * j] << 16), __uint_as_float(w[2 * j] & 0xFFFF0000u));
          const uint16_t hi = quant2(__uint_as_float(w[2 * j + 1] << 16), __uint_as_float(w[2 * j + 1] & 0xFFFF0000u));
          b[j] = static_cast<uint32_t>(lo) | (static_cast<uint32_t>(hi) << 16);
        }
        *reinterpret_cast<uint2*>(o + i) = make_uint2(b[0], b[1]);
      }
    } else {
      for (int i = lane * 2; i < d16; i += 64) {
        const float a = i < d ? __bfloat162float(p[i]) : 0.f;
        const float b = i + 1 < d ? __bfloat162float(p[i + 1]) : 0.f;
        *reinterpret_cast<uint16_t*>(o + i) = quant2(a, b);
      }
    }
#pragma unroll
    for (int o2 = 16; o2 > 0; o2 >>= 1) ss += __shfl_xor_sync(kFullMask, ss, o2);
    if (lane == 0) rnorm[row] = 1.0f / fmaxf(__double2float_rn(sqrt(ss)), kRnormEps);
  }
}

// ------------------------------------------------------------------------------------------
// Store build from the reference's embedding BLOB layout (storage/models.py:94-129: float32 C x H x W,
// C-order): maps N x C x hw  ->  bf16 rows.  pool == 0: one row per cell, (N * hw) x C, i.e. the
// get_flat_vectors order of data.py:112-118; pool == 1: the spatial mean, N x C.
// 32 x 32 tiles go through shared memory so that both the reads (along hw) and the writes (along C)
// are coalesced.
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
maps_to_rows_kernel(const float* __restrict__ maps, long long n, int C, int hw, __nv_bfloat16* __restrict__ rows) {
  __shared__ float tile[32][33];
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;  // 32 x 8
  const int ctiles = (C + 31) / 32, stiles = (hw + 31) / 32;
  const long long per_img = static_cast<long long>(ctiles) * stiles;
  const long long total = per_img * n;
  for (long long t = blockIdx.x; t < total; t += gridDim.x) {
    const long long img = t / per_img;
    const int rem = static_cast<int>(t - img * per_img);
    const int c0 = (rem / stiles) * 32, s0 = (rem % stiles) * 32;
    const float* src = maps + img * C * static_cast<long long>(hw);
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int c = c0 + ty + 8 * j, sidx = s0 + tx;
      tile[ty + 8 * j][tx] = (c < C && sidx < hw) ? src[static_cast<long long>(c) * hw + sidx] : 0.f;
    }
    __syncthreads();
    __nv_bfloat16* dst = rows + (img * hw) * C;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int sidx = s0 + ty + 8 * j, c = c0 + tx;
      if (sidx < hw && c < C) dst[static_cast<long long>(sidx) * C + c] = __float2bfloat16_rn(tile[tx][ty + 8 * j]);
    }
    __syncthreads();
  }
}

// one warp per (image, channel): fp32 sum over the cells in a fixed order, / hw, rounded to bf16
__global__ void __launch_bounds__(256)
maps_pool_rows_kernel(const float* __restrict__ maps, long long n, int C, int hw, __nv_bfloat16* __restrict__ rows) {
  const int lane = threadIdx.x & 31;
  const long long warps = (static_cast<long long>(gridDim.x) * blockDim.x) >> 5;
  const long long total = n * C;
  for (long long r = (static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5; r < total; r += warps) {
    const float* src = maps + r * hw;
    float acc = 0.f;
    for (int i = lane; i < hw; i += 32) acc += src[i];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(kFullMask, acc, o);
    if (lane == 0) rows[r] = __float2bfloat16_rn(acc / static_cast<float>(hw));
  }
}

// ------------------------------------------------------------------------------------------
// K4: search
// ------------------------------------------------------------------------------------------
struct KnnParams {
  int q, d, k;
  long long n;
  int mb, splits;
  long long nb, items;
  int index_base;   // added to a store row when it enters a candidate buffer: the lists hold GLOBAL rows
  int self_base;    // >= 0: query row r is store row self_base + r and never its own neighbour; -1: off
  const float* store_rnorm;
  const float* query_rnorm;
  float* run_scores;   // [q][k] running top-k of every query: raw scores (before the query's inverse norm)
  int32_t* run_idx;    // [q][k] global store rows (index_base + shard-local row), -1 = empty slot
  uint32_t* run_lock;  // [q]
  uint2* cand_global;  // [grid][BM][CAP] when k > kSmallK
  uint32_t* thr_shared;  // [q] per-query lower bound on the global k-th best (ordered-uint encoding)
  uint32_t throttle_window, throttle_every;
  uint32_t* progress;    // [units] tiles loaded so far by every scheduling unit (lockstep throttle)
  const int32_t* row_group;  // [n] group id of every store row (grouped search only)
  // range search only: every column with fl(raw * query_rnorm) >= range_tau is appended to
  // range_rec as {query, global row, fp32 score bits}; range_count counts past range_cap
  float range_tau;
  int32_t* range_rec;
  long long range_cap;
  unsigned long long* range_count;
  // maxsim only: cell_max[q][num_groups] (row-major, 64-bit index) receives, for every query row and
  // group g in [group_base, group_base + num_groups), the largest raw score of g's rows (atomic max)
  float* cell_max;
  int group_base, num_groups;
#ifdef ISX_KNN_PROFILE
  unsigned long long* prof;  // [16] wait-cycle counters (diagnostic build only: -DISX_KNN_PROFILE)
  int debug_skip_select;     // ISX_KNN_SKIP_SELECT=1: the epilogue only loads and releases (floor of the MMA pipeline)
#endif
};

// Diagnostic build (-DISX_KNN_PROFILE): every role accumulates the cycles it spends in each wait and
// adds them to p.prof at the end; the host prints them per CTA.  Compiled out otherwise.
#ifdef ISX_KNN_PROFILE
#define ISX_PROF_DECL unsigned long long prof_acc[24] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0}; long long prof_t0 = 0, prof_t1 = 0, prof_t2 = 0; (void)prof_t0; (void)prof_t1; (void)prof_t2
#define ISX_PROF_COUNT(slot, v) prof_acc[slot] += (v)
#define ISX_PROF_BEGIN1() prof_t1 = clock64()
#define ISX_PROF_END1(slot) prof_acc[slot] += static_cast<unsigned long long>(clock64() - prof_t1)
#define ISX_PROF_BEGIN2() prof_t2 = clock64()
#define ISX_PROF_END2(slot) prof_acc[slot] += static_cast<unsigned long long>(clock64() - prof_t2)
#define ISX_PROF_BEGIN() prof_t0 = clock64()
#define ISX_PROF_END(slot) prof_acc[slot] += static_cast<unsigned long long>(clock64() - prof_t0)
#define ISX_PROF_FLUSH(slot) atomicAdd(p.prof + (slot), prof_acc[slot])
#else
#define ISX_PROF_DECL
#define ISX_PROF_COUNT(slot, v)
#define ISX_PROF_BEGIN1()
#define ISX_PROF_END1(slot)
#define ISX_PROF_BEGIN2()
#define ISX_PROF_END2(slot)
#define ISX_PROF_BEGIN()
#define ISX_PROF_END(slot)
#define ISX_PROF_FLUSH(slot)
#endif

// Shared-memory plan.  k <= kSmallK: 32-entry per-row candidate buffers live in shared memory next to
// a 4-stage operand ring (the buffers are XOR-swizzled by row so that 32 rows appending at the same
// depth hit different banks).  Larger k: 256-entry buffers in the global workspace.  Range search
// (RANGE) has no candidate buffers: it is the CAP = 32 plan without them; MAXSIM likewise, plus the
// tile's group ids.
template <int CAP, int NCTA, bool RES_ = false, bool GROUPED = false, bool RANGE = false, bool MAXSIM = false>
struct KnnSmem {
  // RES: the query tile (all k-blocks, at most kResKb = 4, i.e. d <= 256) stays resident in shared
  // memory for a whole item and the ring holds store tiles only: half the operand traffic per tile.
  static constexpr bool RES = RES_;
  static constexpr int kResKb = 4;
  static constexpr uint32_t B_STAGE_BYTES = (BN / NCTA) * BK * 2;  // 32 KB, or 16 KB per CTA of a pair
  static constexpr int G = epi_groups(CAP);
  static constexpr int STAGES = RES ? 6 : (NCTA == 2) ? (CAP <= 32 ? 5 : 6) : (CAP <= 32 ? 3 : 4);
  static constexpr bool kSmemCand = (CAP <= 32);
  static constexpr int CHUNK = kSmemCand ? 16 : 32;  // accumulator columns per selection window
  static constexpr uint32_t kCandBytes = (kSmemCand && !RANGE && !MAXSIM) ? G * BM * CAP * 8 : 0;
  static constexpr uint32_t kAOff = 0;
  static constexpr uint32_t kBOff = kAOff + (RES ? kResKb : STAGES) * A_STAGE_BYTES;
  static constexpr uint32_t kCandOff = kBOff + STAGES * B_STAGE_BYTES;
  static constexpr uint32_t kRnormOff = kCandOff + kCandBytes;            // [ACC_STAGES][BN] floats
  static constexpr uint32_t kBarOff = kRnormOff + ACC_STAGES * BN * 4;    // mbarriers
  static constexpr uint32_t kNumBars = 2 * STAGES + 2 * ACC_STAGES + 2;  // + resident-query full / empty
  static constexpr uint32_t kTmemPtrOff = kBarOff + kNumBars * 8;
  // grouped search and maxsim: [ACC_STAGES][BN / 32] flags, 1 where all 32 store rows of a chunk are one group
  static constexpr uint32_t kChunkUniOff = kTmemPtrOff + 16;
  // maxsim: [ACC_STAGES][BN] group ids of the tile's store rows (-1 past the store's end)
  static constexpr uint32_t kGroupIdOff = kChunkUniOff + ((GROUPED || MAXSIM) ? ACC_STAGES * (BN / 32) * 4 : 0);
  static constexpr uint32_t kTotal = kGroupIdOff + (MAXSIM ? ACC_STAGES * BN * 4 : 0);
  // the operand tiles need 1024-byte alignment; the dynamic window normally starts aligned, so only
  // as much slack as the 227 KB limit leaves is requested and the kernel checks that it suffices
  static constexpr uint32_t kMaxDynamic = 232448;
  static constexpr uint32_t kDynamicBytes = (kTotal + 1024 <= kMaxDynamic) ? kTotal + 1024 : kMaxDynamic;
  static_assert(kTotal <= kMaxDynamic, "shared-memory plan exceeds 227 KB");
};

// Monotonic float <-> uint32 map (0 = below everything) for atomicMax on thresholds.
__device__ __forceinline__ uint32_t thr_encode(float f) {
  const uint32_t b = __float_as_uint(f);
  return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}
// Largest float strictly below the encoded value (so that `v > result` means `v >= value`).
__device__ __forceinline__ float thr_decode_below(uint32_t u) {
  if (u == 0) return -INFINITY;
  const uint32_t w = u - 1;
  const float f = __uint_as_float((w & 0x80000000u) ? (w & 0x7FFFFFFFu) : ~w);
  return (f == 0.0f) ? __uint_as_float(0x80000001u) : f;
}

// one named barrier per epilogue group (its four warps stage and read their own 128 inverse norms)
__device__ __forceinline__ void epilogue_bar_sync(int group) {
  asm volatile("bar.sync %0, 128;" ::"r"(1 + group) : "memory");
}

// Warp-cooperative prune of one row's candidate buffer: sort, keep the best k, return the new
// threshold (score of the k-th best, or -inf while fewer than k candidates exist).  Entry i of the
// row lives at row_buf[i ^ swz] (swz = row % 32 for the shared-memory buffers, 0 in global memory).
template <int CAP>
__device__ __forceinline__ void prune_row(uint2* row_buf, int swz, int count, int k, float& new_thr,
                                          int& new_count, float (&s)[CAP / 32], int (&idx)[CAP / 32]) {
  constexpr int E = CAP / 32;
  const int lane = static_cast<int>(lane_id());
#pragma unroll
  for (int e = 0; e < E; ++e) {
    const int i = e * 32 + lane;
    if (i < count) {
      const uint2 v = row_buf[i ^ swz];
      s[e] = __uint_as_float(v.x);
      idx[e] = static_cast<int>(v.y);
    } else {
      s[e] = -INFINITY;
      idx[e] = INT_MAX;
    }
  }
  if constexpr (E == 1) {
    // 32 entries, one per lane: rank every entry by counting the entries that sort before it.  The
    // 32 steps are independent (shuffle throughput, ~300 cycles) where the bitonic network is a chain
    // of 15 dependent shuffle steps (~800): the prune sits on the path that gates the accumulator
    // hand-off of all 16 epilogue warps of a pair.
    const float ms = s[0];
    const int mi = idx[0];
    int rank = 0;
#pragma unroll
    for (int j = 0; j < 32; ++j) {
      const float os = __shfl_sync(kFullMask, ms, j);
      const int oi = __shfl_sync(kFullMask, mi, j);
      rank += pair_before(os, oi, ms, mi) ? 1 : 0;
    }
    new_count = min(count, k);
    __syncwarp();
    if (lane < count && rank < k) row_buf[rank ^ swz] = make_uint2(__float_as_uint(ms), static_cast<uint32_t>(mi));
    __syncwarp();
    // sorted order back into registers (slot i on lane i), as the callers expect
    if (lane < new_count) {
      const uint2 v = row_buf[lane ^ swz];
      s[0] = __uint_as_float(v.x);
      idx[0] = static_cast<int>(v.y);
    } else {
      s[0] = -INFINITY;
      idx[0] = INT_MAX;
    }
    const float kth = __shfl_sync(kFullMask, s[0], (k - 1) & 31);
    new_thr = (count >= k) ? kth : -INFINITY;
  } else {
    warp_sort_desc<E>(s, idx);
    float kth = -INFINITY;
#pragma unroll
    for (int e = 0; e < E; ++e) {
      const int i = e * 32 + lane;
      if (i < k && i < count) row_buf[i ^ swz] = make_uint2(__float_as_uint(s[e]), static_cast<uint32_t>(idx[e]));
      const float cand = __shfl_sync(kFullMask, s[e], (k - 1) & 31);
      if (e == ((k - 1) >> 5)) kth = cand;
    }
    new_count = min(count, k);
    new_thr = (count >= k) ? kth : -INFINITY;
  }
}

// In-tile prune of a LARGE buffer (k > 16: 256 entries in global memory) without sorting it: the k-th
// best score is found by a bitwise bisection over the order-preserving integer image of the scores
// (32 rounds of warp ballots over the lanes' registers), and the entries at or above it are compacted
// to the front of the buffer, unsorted — order only matters at the item end, which sorts what is left.
// About 1100 instructions against about 2600 for the 256-entry bitonic network plus its stores.
// Ties at the k-th score are all kept (they arrived earlier, i.e. they have lower rows than anything
// that can still arrive in this item); if so many tie that the buffer would stay more than half-way
// to full, the caller falls back to the sorting prune, which keeps exactly k.  Returns false then.
template <int CAP>
__device__ __forceinline__ bool prune_row_select(uint2* row_buf, int count, int k, float& new_thr, int& new_count) {
  constexpr int E = CAP / 32;
  const int lane = static_cast<int>(lane_id());
  uint2 v[E];
  uint32_t enc[E];
#pragma unroll
  for (int e = 0; e < E; ++e) {
    const int i = e * 32 + lane;
    v[e] = make_uint2(0u, 0u);
    enc[e] = 0u;  // below every real score
    if (i < count) {
      v[e] = row_buf[i];
      enc[e] = thr_encode(__uint_as_float(v[e].x));
    }
  }
  __syncwarp();
  uint32_t prefix = 0;
#pragma unroll 1
  for (int bit = 31; bit >= 0; --bit) {
    const uint32_t cand = prefix | (1u << bit);
    int ge = 0;
#pragma unroll
    for (int e = 0; e < E; ++e) ge += __popc(__ballot_sync(kFullMask, enc[e] >= cand));
    if (ge >= k) prefix = cand;
  }
  // prefix = the k-th largest encoded score
  int kept_total = 0;
#pragma unroll
  for (int e = 0; e < E; ++e) kept_total += __popc(__ballot_sync(kFullMask, enc[e] >= prefix));
  if (2 * kept_total > CAP + k) return false;  // a pile of ties: let the sorting prune cut to exactly k
  int kept = 0;
#pragma unroll
  for (int e = 0; e < E; ++e) {
    const bool kp = enc[e] >= prefix;
    const uint32_t bal = __ballot_sync(kFullMask, kp);
    if (kp) row_buf[kept + __popc(bal & ((1u << lane) - 1u))] = v[e];
    kept += __popc(bal);
  }
  __syncwarp();
  new_count = kept;
  // decode: prefix is the encoding of the k-th best score itself
  new_thr = __uint_as_float((prefix & 0x80000000u) ? (prefix & 0x7FFFFFFFu) : ~prefix);
  return true;
}

// ---- grouped selection (image-level search) ----------------------------------------------------
// Every store row r carries a group id g(r) >= 0.  A group's score is the best score of its rows and
// its representative is its first row in (score desc, row asc) order; the result is the k best
// representatives.  Empty entries are (-inf, INT_MAX) with group -1.  An entry may be dropped as soon
// as an entry of its group that sorts before it is known: it can never be a representative.

// group of a candidate (global row; the table is indexed by store-local row)
__device__ __forceinline__ int row_group_of(const int32_t* row_group, int index_base, int idx) {
  return idx != INT_MAX ? __ldg(row_group + (idx - index_base)) : -1;
}

// One entry per lane, in any order.  Returns the entry's rank among the entries that are first of
// their group, or -1 if an entry of the same group sorts before it (or it is empty); `distinct` = the
// number of groups present.  The rank counting of prune_row plus one compare per step.
__device__ __forceinline__ int grouped_rank32(float ms, int mi, int mg, int& distinct) {
  uint32_t before = 0;
  bool dup = false;
#pragma unroll
  for (int j = 0; j < 32; ++j) {
    const float os = __shfl_sync(kFullMask, ms, j);
    const int oi = __shfl_sync(kFullMask, mi, j);
    const int og = __shfl_sync(kFullMask, mg, j);
    const bool b = pair_before(os, oi, ms, mi);
    before |= b ? (1u << j) : 0u;
    dup |= b && og == mg;
  }
  const bool alive = mi != INT_MAX && !dup;
  const uint32_t am = __ballot_sync(kFullMask, alive);
  distinct = __popc(am);
  return alive ? __popc(am & before) : -1;
}

// warp_sort_desc over (score, row, group) triples; BY_GROUP: order by (group asc, score desc, row asc)
template <bool BY_GROUP>
__device__ __forceinline__ bool entry_before(float sa, int ia, int ga, float sb, int ib, int gb) {
  if constexpr (BY_GROUP) return ga < gb || (ga == gb && pair_before(sa, ia, sb, ib));
  else return pair_before(sa, ia, sb, ib);
}

template <int E, bool BY_GROUP>
__device__ __forceinline__ void warp_sort3(float (&s)[E], int (&idx)[E], int (&g)[E]) {
  const uint32_t lane = lane_id();
  constexpr int TOTAL = 32 * E;
#pragma unroll
  for (int k = 2; k <= TOTAL; k <<= 1) {
#pragma unroll
    for (int j = k >> 1; j > 0; j >>= 1) {
      if (j >= 32) {
        const int je = j >> 5;
#pragma unroll
        for (int e = 0; e < E; ++e) {
          const int pe = e ^ je;
          if (pe > e) {
            const bool desc_block = ((e * 32) & k) == 0;
            const bool lower_first = entry_before<BY_GROUP>(s[e], idx[e], g[e], s[pe], idx[pe], g[pe]);
            if (desc_block ? !lower_first : lower_first) {
              float ts = s[e]; s[e] = s[pe]; s[pe] = ts;
              int ti = idx[e]; idx[e] = idx[pe]; idx[pe] = ti;
              int tg = g[e]; g[e] = g[pe]; g[pe] = tg;
            }
          }
        }
      } else {
#pragma unroll
        for (int e = 0; e < E; ++e) {
          const int i = e * 32 + static_cast<int>(lane);
          const float os = __shfl_xor_sync(kFullMask, s[e], j);
          const int oi = __shfl_xor_sync(kFullMask, idx[e], j);
          const int og = __shfl_xor_sync(kFullMask, g[e], j);
          const bool desc_block = ((i & k) == 0);
          const bool i_am_lower = ((lane & j) == 0);
          const bool mine_first = entry_before<BY_GROUP>(s[e], idx[e], g[e], os, oi, og);
          const bool keep_mine = (desc_block == i_am_lower) ? mine_first : !mine_first;
          if (!keep_mine) { s[e] = os; idx[e] = oi; g[e] = og; }
        }
      }
    }
  }
}

// 32*E entries (element i = e*32 + lane, any order) -> the first entry of every group, sorted by
// (score desc, row asc), empties behind them.  Returns the number of groups.  Two sorts: by group
// to find the non-first entries (a neighbour of the same group sorts before them), then by score.
template <int E>
__device__ __forceinline__ int grouped_select(float (&s)[E], int (&idx)[E], int (&g)[E]) {
  const int lane = static_cast<int>(lane_id());
  warp_sort3<E, true>(s, idx, g);
  int distinct = 0;
  int carry = INT_MIN;  // group of element e*32 - 1
#pragma unroll
  for (int e = 0; e < E; ++e) {
    const int up = __shfl_up_sync(kFullMask, g[e], 1);
    const int prev = lane ? up : carry;
    carry = __shfl_sync(kFullMask, g[e], 31);
    const bool dead = idx[e] == INT_MAX || prev == g[e];
    distinct += __popc(__ballot_sync(kFullMask, !dead));
    if (dead) { s[e] = -INFINITY; idx[e] = INT_MAX; g[e] = -1; }
  }
  warp_sort3<E, false>(s, idx, g);
  return distinct;
}

// Grouped form of prune_row: keep the representatives of the best k groups of the buffer, return the
// score of the k-th (or -inf while fewer than k groups are present).  No bisection variant: a
// selection without sorting cannot tell which entries share a group.
template <int CAP>
__device__ __forceinline__ void prune_row_grouped(uint2* row_buf, int swz, int count, int k, const int32_t* row_group,
                                                  int index_base, float& new_thr, int& new_count) {
  constexpr int E = CAP / 32;
  const int lane = static_cast<int>(lane_id());
  float s[E];
  int idx[E], g[E];
#pragma unroll
  for (int e = 0; e < E; ++e) {
    const int i = e * 32 + lane;
    s[e] = -INFINITY;
    idx[e] = INT_MAX;
    if (i < count) {
      const uint2 v = row_buf[i ^ swz];
      s[e] = __uint_as_float(v.x);
      idx[e] = static_cast<int>(v.y);
    }
    g[e] = row_group_of(row_group, index_base, idx[e]);
  }
  if constexpr (E == 1) {
    int distinct;
    const int rank = grouped_rank32(s[0], idx[0], g[0], distinct);
    new_count = min(distinct, k);
    __syncwarp();
    if (rank >= 0 && rank < k) row_buf[rank ^ swz] = make_uint2(__float_as_uint(s[0]), static_cast<uint32_t>(idx[0]));
    __syncwarp();
    const uint32_t km = __ballot_sync(kFullMask, rank == k - 1);
    new_thr = km ? __shfl_sync(kFullMask, s[0], __ffs(km) - 1) : -INFINITY;
  } else {
    const int distinct = grouped_select<E>(s, idx, g);
    __syncwarp();
    float kth = -INFINITY;
#pragma unroll
    for (int e = 0; e < E; ++e) {
      const int i = e * 32 + lane;
      if (i < k && i < distinct) row_buf[i ^ swz] = make_uint2(__float_as_uint(s[e]), static_cast<uint32_t>(idx[e]));
      const float cand = __shfl_sync(kFullMask, s[e], (k - 1) & 31);
      if (e == ((k - 1) >> 5)) kth = cand;
    }
    __syncwarp();
    new_count = min(distinct, k);
    new_thr = (distinct >= k) ? kth : -INFINITY;
  }
}

// ---- range search ------------------------------------------------------------------------------
// A store row e is a hit of query row q when score = fl(raw · rnorm_q) >= tau, raw = fl(dot · rnorm_e)
// being what the epilogue holds after scaling: the product K5 forms for search(), so a hit's score is
// bit for bit the one search() reports.

// Raw-score bound of one query row: every raw r of a hit satisfies r > bound, so the fast path's
// `vmax > thr` never drops a hit.  Argument (round-to-nearest, rq = rnorm_q finite and > 0): let
// t = pred(tau), the float just below tau.  fl is monotone, so r · rq <= t would give fl(r · rq) <= t
// < tau: a hit has r · rq > t, i.e. r > t / rq in exact arithmetic.  The quotient is formed in double
// (t and rq are floats, so it is within 2^-53 relative of t / rq and never overflows or underflows),
// rounded down to float, and stepped down one more float: a double rounding error of 2^-53 relative
// can move it across at most one float, so the result is <= t / rq < r.  Rows with rq = 0 or +inf
// (an overflowing norm) get no bound: every column takes the exact test.
__device__ __forceinline__ float range_raw_bound(float tau, float rq) {
  if (!(rq > 0.f) || isinf(rq)) return -INFINITY;
  const float t = nextafterf(tau, -INFINITY);
  const float b = __double2float_rd(static_cast<double>(t) / static_cast<double>(rq));
  return nextafterf(b, -INFINITY);
}

// Rare path of one 32-column chunk: the exact test of every column of the rows whose chunk maximum
// passed the bound, then one append per warp.  Lanes' hit counts are prefix-summed, one 64-bit
// atomicAdd reserves the warp's slots, and a record is written only when its slot is below the
// capacity; the counter keeps counting past it, so the caller learns the exact total.  Columns past
// the store's end (ncols) and the query's own row (self_row, -1 when off) are never hits.
__device__ __forceinline__ void range_append(const uint32_t (&r)[32], bool pass, float rq, int qrow, int cbase,
                                             int ncols, int gcol0, int self_row, const KnnParams& p) {
  const int lane = static_cast<int>(lane_id());
  uint32_t hits = 0;
  if (pass) {
#pragma unroll
    for (int j = 0; j < 32; ++j) {
      const float s = __fmul_rn(__uint_as_float(r[j]), rq);
      const bool take = s >= p.range_tau && cbase + j < ncols && gcol0 + cbase + j != self_row;
      hits |= take ? (1u << j) : 0u;
    }
  }
  const int mine = __popc(hits);
  int incl = mine;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int t = __shfl_up_sync(kFullMask, incl, o);
    if (lane >= o) incl += t;
  }
  const int total = __shfl_sync(kFullMask, incl, 31);
  if (total == 0) return;
  unsigned long long base = 0;
  if (lane == 31) base = atomicAdd(p.range_count, static_cast<unsigned long long>(total));
  base = __shfl_sync(kFullMask, base, 31);
  unsigned long long slot = base + static_cast<unsigned long long>(incl - mine);
  if (!hits) return;
  // unrolled over the columns: an index taken from the hit mask would move the accumulator registers
  // to local memory for the whole epilogue
#pragma unroll
  for (int j = 0; j < 32; ++j) {
    if ((hits >> j) & 1u) {
      if (slot < static_cast<unsigned long long>(p.range_cap)) {
        int32_t* rec = p.range_rec + 3 * slot;
        rec[0] = qrow;
        rec[1] = gcol0 + cbase + j;
        rec[2] = static_cast<int32_t>(__float_as_uint(__fmul_rn(__uint_as_float(r[j]), rq)));
      }
      ++slot;
    }
  }
}

// ---- maxsim ------------------------------------------------------------------------------------
// atomic max of an fp32 value: a non-negative float orders like its bits as a signed int, a negative
// one inversely to its bits as an unsigned int, so the pair signed max / unsigned min updates the
// value in place (the slot starts at -inf).  -0 is turned into +0 first, so that the two never race
// through different updates.
__device__ __forceinline__ void atomic_max_f32(float* addr, float v) {
  v = (v == 0.f) ? 0.f : v;
  if (__float_as_int(v) >= 0) atomicMax(reinterpret_cast<int*>(addr), __float_as_int(v));
  else atomicMin(reinterpret_cast<unsigned int*>(addr), __float_as_uint(v));
}

// GROUPED: image-level search (knn_search_grouped_kernel).  The k-th best DISTINCT-GROUP score of
// any subset of the store is a lower bound of the global one, so the fast path, the shared bound and
// the item-end skip stay as they are; only where a threshold is derived — the buffer prune, the
// item-end merge into the running list and the finalising merge — entries are de-duplicated by group
// before k are counted.
//
// RANGE: range search (knn_range_kernel, CAP = 32 variants only).  The threshold is fixed and known
// before the first tile, so the epilogue keeps the fast path and replaces the rest: no candidate
// buffers, prunes, shared bound or item end; the rare path tests every column of the chunk exactly
// and appends the hits to a global record buffer (range_append).
//
// F8: the operands are E4M3 rows (knn_search_fp8_kernel).  The producer moves them as 16-bit pairs
// (p.d = d16 / 2, tensor maps of UINT16), so a k-block is still one 128-byte swizzle row of BK units,
// now 128 elements: the ring, the TMA boxes, the descriptors and their 32-byte step per MMA (K = 32
// under kind::f8f6f4) and the whole epilogue are those of the bf16 kernel; only the MMA kind changes.
//
// MAXSIM: the per-(query row, group) maxima of multi-vector search (knn_maxsim_kernel, CAP = 32
// variants only).  The epilogue keeps the fast path's scaling and chunk maximum and drops everything
// else (thresholds, buffers, prunes, shared bound, item end): a chunk of one group folds its maximum
// into the row's running (group, max) pair, a mixed chunk walks its columns by the staged group ids,
// and a pair is flushed into p.cell_max by atomic max when the group changes and at the item end.
// Atomics, because a group can be cut by an N-split or between the two epilogue groups' halves.
template <int CAP, int NCTA, bool RES, bool GROUPED, bool RANGE = false, bool F8 = false, bool MAXSIM = false>
__device__ __forceinline__ void knn_search_body(const CUtensorMap& tmap_q, const CUtensorMap& tmap_e, const KnnParams& p) {
  static_assert(!F8 || (!GROUPED && !RANGE), "the fp8 scan is a plain search");
  static_assert(!MAXSIM || (!GROUPED && !RANGE && !F8 && CAP == 32), "maxsim is its own mode of the CAP = 32 plan");
  using L = KnnSmem<CAP, NCTA, RES, GROUPED, RANGE, MAXSIM>;
  constexpr int STAGES = L::STAGES;
  constexpr int kEpiGroups = L::G;
  constexpr int kGroupCols = BN / kEpiGroups;
  constexpr uint32_t B_STAGE_BYTES = L::B_STAGE_BYTES;
  // NCTA == 2: this CTA and its cluster peer form one MMA of M = 256 (cta_group::2).  Rank r owns
  // query rows [128 r, 128 r + 128) of the 256-row block and loads store rows [128 r, 128 r + 128) of
  // every 256-row store tile; the leader (rank 0) issues the MMAs for both.
  const uint32_t rank = (NCTA == 2) ? cluster_ctarank() : 0u;
  const long long unit = blockIdx.x / NCTA, num_units = gridDim.x / NCTA;
  constexpr int E = CAP / 32;
  extern __shared__ uint8_t smem_raw[];
  // align by offsetting the shared array itself (not through an integer round trip) so the compiler
  // keeps the shared address space and emits LDS/STS instead of generic loads and stores
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  if (threadIdx.x == 0 && static_cast<uint32_t>(smem - smem_raw) + L::kTotal > L::kDynamicBytes) {
    printf("isx: knn_search_kernel: dynamic shared memory window is not 1024-byte aligned\n");
    __trap();
  }

  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + L::kBarOff);
  uint64_t* full_bar = bars;
  uint64_t* empty_bar = bars + STAGES;
  uint64_t* tmem_full = bars + 2 * STAGES;
  uint64_t* tmem_empty = bars + 2 * STAGES + ACC_STAGES;
  uint64_t* a_full = bars + 2 * STAGES + 2 * ACC_STAGES;
  uint64_t* a_empty = a_full + 1;
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(smem + L::kTmemPtrOff);
  float* rnorm_s = reinterpret_cast<float*>(smem + L::kRnormOff);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int num_kb = (p.d + BK - 1) / BK;
  ISX_PROF_DECL;
#ifdef ISX_KNN_PROFILE
  const long long prof_kernel_t0 = clock64();
#endif

  if (warp == 0 && lane == 0) {
    prefetch_tmap(&tmap_q);
    prefetch_tmap(&tmap_e);
  }
  if (warp == 1 && lane == 0) {
    for (int i = 0; i < STAGES; ++i) { mbar_init(&full_bar[i], NCTA); mbar_init(&empty_bar[i], 1); }
    mbar_init(a_full, NCTA);
    mbar_init(a_empty, 1);
    for (int i = 0; i < ACC_STAGES; ++i) { mbar_init(&tmem_full[i], 1); mbar_init(&tmem_empty[i], 4 * kEpiGroups * NCTA); }
    fence_mbar_init();
  }
  if (warp == 2) {
    if (NCTA == 2) { tmem_alloc_pair(tmem_ptr, 512); tmem_relinquish_pair(); }
    else { tmem_alloc(tmem_ptr, 512); tmem_relinquish(); }
  }
  tc_fence_before();
  if (NCTA == 2) cluster_sync_all(); else __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;

  if (warp == 0) {
    // ===================== TMA producer =====================
    if (lane == 0) {
      uint32_t stage = 0, phase = 0;
      // Lockstep throttle.  Units that run at the same time stream the same store rows (items are
      // ordered split-major and equally long) and share them through L2 — as long as they stay
      // within a window of each other.  Epilogues of different length (large k) let them drift, and
      // every tile is then fetched from HBM once per query block.  Every kThrottleEvery tiles a unit
      // publishes how many tiles it has loaded and waits until the slowest unit is within
      // kThrottleWindow tiles (all units are co-resident: grid <= #SMs, one CTA per SM).  k = 100:
      // DRAM reads 37.8 GB -> ~5 GB per pass, 23.5 -> 21 ms.
      // Units are normally co-resident (grid <= #SMs, one CTA per SM); the wait gives up after 2 ms.
      const uint32_t kThrottleEvery = p.throttle_every;  // a power of two
      const uint32_t kThrottleWindow = p.throttle_window;
      uint32_t seq = 0, item_no = 0;
      bool throttle_on = true;
      constexpr uint64_t kThrottleGiveUpNs = 2000000;  // 2 ms: above the longest item end (k = 100: ~0.3 ms)
      for (long long item = unit; item < p.items; item += num_units) {
        const int split = static_cast<int>(item / p.mb);
        const int mblk = static_cast<int>(item - static_cast<long long>(split) * p.mb);
        const long long nb0 = p.nb * split / p.splits, nb1 = p.nb * (split + 1) / p.splits;
        const int32_t m0 = (mblk * NCTA + static_cast<int>(rank)) * BM;
        if (RES) {
          // resident query tile: wait until the previous item's MMAs have read it, then load all k-blocks
          mbar_wait(a_empty, (item_no & 1u) ^ 1u);
          if (NCTA == 2) mbar_arrive_expect_tx_leader(a_full, static_cast<uint32_t>(num_kb) * A_STAGE_BYTES);
          else mbar_arrive_expect_tx(a_full, static_cast<uint32_t>(num_kb) * A_STAGE_BYTES);
          for (int kb = 0; kb < num_kb; ++kb) {
            uint8_t* a_res = smem + L::kAOff + kb * A_STAGE_BYTES;
            if (NCTA == 2) tma_load_2d_pair(a_res, &tmap_q, a_full, kb * BK, m0, kEvictLast);
            else tma_load_2d(a_res, &tmap_q, a_full, kb * BK, m0, kEvictLast);
          }
          ++item_no;
        }
        for (long long nb = nb0; nb < nb1; ++nb, ++seq) {
          if ((seq & (kThrottleEvery - 1)) == 0) {
            volatile uint32_t* prog = p.progress;
            if (rank == 0) prog[unit] = seq;
            if (throttle_on && seq > kThrottleWindow) {
              ISX_PROF_BEGIN();
              uint64_t t0 = 0;
              while (true) {
                uint32_t slowest = 0xFFFFFFFFu;
                for (int u = 0; u < static_cast<int>(num_units); ++u) slowest = min(slowest, prog[u]);
                if (slowest + kThrottleWindow >= seq) break;
                __nanosleep(256);
                const uint64_t now = global_timer_ns();
                if (t0 == 0) t0 = now;
                else if (now - t0 > kThrottleGiveUpNs) {
                  // The throttle is an optimisation, never a dependency: if some unit is this far
                  // behind (its CTA pair has not been scheduled yet because another kernel holds SMs,
                  // or it is stuck behind a long item end), stop synchronising for the rest of the launch.
                  throttle_on = false;
                  break;
                }
              }
              ISX_PROF_END(1);
            }
          }
          const int32_t n0 = static_cast<int32_t>(nb * BN) + static_cast<int32_t>(rank) * (BN / NCTA);
          for (int kb = 0; kb < num_kb; ++kb) {
            ISX_PROF_BEGIN();
            mbar_wait(&empty_bar[stage], phase ^ 1);
            ISX_PROF_END(0);
            uint8_t* a_dst = smem + L::kAOff + (RES ? 0 : stage) * A_STAGE_BYTES;
            uint8_t* b_dst = smem + L::kBOff + stage * B_STAGE_BYTES;
            constexpr uint32_t kStageTx = (RES ? 0u : A_STAGE_BYTES) + B_STAGE_BYTES;
            if (NCTA == 2) {
              // both CTAs report to the leader's barrier (count 2, 2 x 32 KB of transactions)
              mbar_arrive_expect_tx_leader(&full_bar[stage], kStageTx);
              if (!RES) tma_load_2d_pair(a_dst, &tmap_q, &full_bar[stage], kb * BK, m0, kEvictLast);
              tma_load_2d_pair(b_dst, &tmap_e, &full_bar[stage], kb * BK, n0, kEvictNormal);
            } else {
              mbar_arrive_expect_tx(&full_bar[stage], kStageTx);
              if (!RES) tma_load_2d(a_dst, &tmap_q, &full_bar[stage], kb * BK, m0, kEvictLast);
              tma_load_2d(b_dst, &tmap_e, &full_bar[stage], kb * BK, n0, kEvictNormal);
            }
            if (++stage == STAGES) { stage = 0; phase ^= 1; }
          }
        }
      }
      if (rank == 0) *(volatile uint32_t*)(p.progress + unit) = 0xFFFFFFFFu;  // done: never the slowest again
      if (rank == 0) { ISX_PROF_FLUSH(0); ISX_PROF_FLUSH(1); }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    if (lane == 0 && rank == 0) {
      constexpr uint32_t idesc = make_idesc(F8 ? 0 /*e4m3*/ : 1 /*bf16*/, BM * NCTA, BN);
      uint32_t stage = 0, phase = 0, acc = 0, acc_phase = 0, item_no = 0;
      for (long long item = unit; item < p.items; item += num_units) {
        const int split = static_cast<int>(item / p.mb);
        const long long nb0 = p.nb * split / p.splits, nb1 = p.nb * (split + 1) / p.splits;
        if (RES) {
          mbar_wait(a_full, item_no & 1u);
          tc_fence_after();
          ++item_no;
        }
        for (long long nb = nb0; nb < nb1; ++nb) {
          ISX_PROF_BEGIN();
          mbar_wait(&tmem_empty[acc], acc_phase ^ 1);
          ISX_PROF_END(2);
          tc_fence_after();
          const uint32_t d_tmem = tmem_base + acc * BN;
          for (int kb = 0; kb < num_kb; ++kb) {
            ISX_PROF_BEGIN();
            mbar_wait(&full_bar[stage], phase);
            ISX_PROF_END(3);
            tc_fence_after();
            const uint32_t a_addr = smem_u32(smem + L::kAOff + (RES ? kb : static_cast<int>(stage)) * A_STAGE_BYTES);
            const uint32_t b_addr = smem_u32(smem + L::kBOff + stage * B_STAGE_BYTES);
#pragma unroll
            for (int k = 0; k < BK / UMMA_K; ++k) {
              const uint64_t a_desc = make_kmajor_sw128_desc(a_addr + k * UMMA_K * 2);
              const uint64_t b_desc = make_kmajor_sw128_desc(b_addr + k * UMMA_K * 2);
              if constexpr (F8) {
                if (NCTA == 2) tc_mma_f8_pair(d_tmem, a_desc, b_desc, idesc, (kb | k) != 0);
                else tc_mma_f8(d_tmem, a_desc, b_desc, idesc, (kb | k) != 0);
              } else {
                if (NCTA == 2) tc_mma_f16_pair(d_tmem, a_desc, b_desc, idesc, (kb | k) != 0);
                else tc_mma_f16(d_tmem, a_desc, b_desc, idesc, (kb | k) != 0);
              }
            }
            // frees the smem slot (in both CTAs of a pair) once these MMAs have read it
            if (NCTA == 2) tc_commit_pair(&empty_bar[stage]); else tc_commit(&empty_bar[stage]);
            if (++stage == STAGES) { stage = 0; phase ^= 1; }
          }
          // accumulator complete
          if (NCTA == 2) tc_commit_pair(&tmem_full[acc]); else tc_commit(&tmem_full[acc]);
          if (++acc == ACC_STAGES) { acc = 0; acc_phase ^= 1; }
        }
        // the resident query tile may be overwritten once every MMA of this item has read it
        if (RES) { if (NCTA == 2) tc_commit_pair(a_empty); else tc_commit(a_empty); }
      }
      ISX_PROF_FLUSH(2);
      ISX_PROF_FLUSH(3);
    }
  } else if (warp >= kEpilogueWarp0) {
    // ===================== epilogue: fused top-k =====================
    constexpr int CHUNK = L::CHUNK;
    const int ew = warp & 3;                  // the TMEM lane quarter this warp may read
    const int eg = (warp - kEpilogueWarp0) >> 2;  // column group
    const int row = ew * 32 + lane;           // query row inside the tile
    const int et = threadIdx.x - kEpilogueWarp0 * 32;  // 0..255: the store row whose inverse norm this thread stages
    uint2* cand_base;
    constexpr uint32_t cand_stride = CAP;
    if (L::kSmemCand) {
      cand_base = reinterpret_cast<uint2*>(smem + L::kCandOff) + static_cast<size_t>(eg) * BM * CAP;
    } else {
      cand_base = p.cand_global + (static_cast<size_t>(blockIdx.x) * kEpiGroups + eg) * BM * CAP;
    }
    const int my_swz = L::kSmemCand ? lane : 0;
    uint2* my_buf = cand_base + static_cast<size_t>(row) * cand_stride;
    uint2* warp_buf = cand_base + static_cast<size_t>(ew * 32) * cand_stride;

    uint32_t acc = 0, acc_phase = 0;
    float s_reg[E];
    int i_reg[E];
    for (long long item = unit; item < p.items; item += num_units) {
      const int split = static_cast<int>(item / p.mb);
      const int mblk = static_cast<int>(item - static_cast<long long>(split) * p.mb);
      const long long nb0 = p.nb * split / p.splits, nb1 = p.nb * (split + 1) / p.splits;
      const int m0 = (mblk * NCTA + static_cast<int>(rank)) * BM;
      const int qrow = m0 + row;
      const bool row_valid = qrow < p.q;
      // all-pairs graph: the query is itself a store row and must not be its own neighbour.  The test
      // sits in the rare path only (a query's own score is its maximum, so the tile that holds it
      // always takes that path once and appends nothing for it).
      const int self_row = (p.self_base >= 0) ? p.self_base + qrow : -1;
      // `thr`: a candidate must beat it.  It is the larger of this item's own k-th best and the
      // bound every CTA working on the same query publishes in thr_shared: anything below the k-th
      // best of ANY subset of the store cannot be in the global top-k, so other splits' progress
      // prunes this one (the partial list may then hold fewer than k entries; the merge pads).
      float thr = row_valid ? -INFINITY : INFINITY;
      float range_rq = 0.f;  // range search: the query's inverse norm
      if constexpr (RANGE) {
        if (row_valid) {
          range_rq = __ldg(p.query_rnorm + qrow);
          thr = range_raw_bound(p.range_tau, range_rq);
        }
      }
      int cnt = 0;
      float row_best = -INFINITY;  // best score this item has appended for the row

      // Per-tile staging runs one tile ahead: the store rows' inverse norms of tile nb + 1 and the
      // shared bound of this row are fetched into registers while tile nb is being selected, so their
      // global-memory latency never sits between two tiles (it did: ~600 cycles per tile, visible at
      // d = 256 where a tile is only 2048 MMA cycles long).
      float pre_rn = 0.f, pre_rn2 = 0.f;
      uint32_t pre_thr = 0;
      int pre_g = -1, pre_g2 = -1;  // grouped: groups of the store rows whose inverse norms this thread stages
      auto prefetch_tile = [&](long long nb_) {
        const long long n0_ = nb_ * BN;
        pre_rn = (n0_ + et < p.n) ? __ldg(p.store_rnorm + n0_ + et) : 0.f;
        if (kEpiGroups == 1) pre_rn2 = (n0_ + et + 128 < p.n) ? __ldg(p.store_rnorm + n0_ + et + 128) : 0.f;
        if constexpr (GROUPED || MAXSIM) {
          pre_g = (n0_ + et < p.n) ? __ldg(p.row_group + n0_ + et) : -1;
          if (kEpiGroups == 1) pre_g2 = (n0_ + et + 128 < p.n) ? __ldg(p.row_group + n0_ + et + 128) : -1;
        }
        if constexpr (!RANGE && !MAXSIM) {
          if (row_valid) pre_thr = *reinterpret_cast<const volatile uint32_t*>(p.thr_shared + qrow);
        }
      };
      // maxsim: the row's running (group, maximum) pair and its flush into cell_max
      int ms_g = -1;
      float ms_max = -INFINITY;
      auto maxsim_flush = [&]() {
        const long long gi = static_cast<long long>(ms_g) - p.group_base;
        if (row_valid && gi >= 0 && gi < p.num_groups)
          atomic_max_f32(p.cell_max + static_cast<size_t>(qrow) * static_cast<size_t>(p.num_groups) + gi, ms_max);
      };
      prefetch_tile(nb0);

      for (long long nb = nb0; nb < nb1; ++nb) {
        const long long n0 = nb * BN;
        const int ncols = static_cast<int>(min(static_cast<long long>(BN), p.n - n0));
        const int gcol0 = static_cast<int>(n0) + p.index_base;  // global row of the tile's first column
        // publish this tile's inverse norms (the previous user of this slot was tile nb-2, whose
        // readers all passed the barrier of tile nb-1)
        float* rn = rnorm_s + acc * BN;
        rn[et] = pre_rn;
        if (kEpiGroups == 1) rn[et + 128] = pre_rn2;
        int* chunk_uni = reinterpret_cast<int*>(smem + L::kChunkUniOff) + acc * (BN / 32);
        int* gid_s = reinterpret_cast<int*>(smem + L::kGroupIdOff) + acc * BN;
        if constexpr (MAXSIM) {
          gid_s[et] = pre_g;
          if (kEpiGroups == 1) gid_s[et + 128] = pre_g2;
        }
        if constexpr (GROUPED || MAXSIM) {
          // the 32 rows this warp stages are one selection chunk: flag it when they are all one group
          const int g0 = __shfl_sync(kFullMask, pre_g, 0);
          const bool uni = __all_sync(kFullMask, pre_g == g0 && pre_g >= 0);
          if (lane == 0) chunk_uni[et >> 5] = uni ? 1 : 0;
          if (kEpiGroups == 1) {
            const int g1 = __shfl_sync(kFullMask, pre_g2, 0);
            const bool uni1 = __all_sync(kFullMask, pre_g2 == g1 && pre_g2 >= 0);
            if (lane == 0) chunk_uni[(et + 128) >> 5] = uni1 ? 1 : 0;
          }
        }
        if constexpr (!RANGE && !MAXSIM) {
          if (row_valid) thr = fmaxf(thr, thr_decode_below(pre_thr));
        }
        if (nb + 1 < nb1) prefetch_tile(nb + 1);
        ISX_PROF_BEGIN();
        epilogue_bar_sync(eg);
        ISX_PROF_END(5);

        // Selection of one 32-column chunk held in registers.  Fast path (almost every chunk): scale
        // by the inverse norms (packed FMUL2), maxima of the eight 4-column groups and of the chunk
        // (FMNMX3), ONE warp-uniform test against the rows' thresholds.
        // Rare path (some row of the warp has a survivor; per tile and warp that is about one event at
        // the metric's shape, and all 16 epilogue warps of a pair gate the accumulator hand-off, so
        // its cost is what bounds the kernel at small d): rows walk only the groups that hold a
        // survivor and append; a row's buffer is pruned (sorted, best k kept, threshold raised) only
        // when the appends of this chunk could overflow it.  Rows whose threshold is still so low that
        // more groups survive than a pruned buffer can take (cold start) use the windowed walk.
        // Measured and dropped: (a) a cheaper chunk-level bound (raw maximum times the chunk's largest
        // inverse norm): at a 1-in-10^5 selection rate a bound 5 % loose passes 3-5 x as often; with the
        // store SORTED by norm (row ids carried beside it) the bound is tight and only 0.66 of a warp's 4
        // chunks per tile reach the scaling, but the fast path is not bound by those instructions
        // (2690 -> 2530 select cycles per tile at d = 256) while the id lookup in the appends and the
        // tie handling a permuted order needs double the cost of a rare-path event: 6.2 ms against 4.4;
        // (b) a warp-cooperative walk, one surviving row at a time (ballot + popc ranking): rows with
        // survivors come in groups, and serialising them costs more than a predicated walk.
        auto prune_rows = [&](uint32_t need) {
          if (need) ISX_PROF_BEGIN2();
          const uint32_t need0 = need;
          (void)need0;
          while (need) {
            ISX_PROF_COUNT(12, 1);
            const int rr = __ffs(need) - 1;
            need &= need - 1;
            __syncwarp();
            const int c = __shfl_sync(kFullMask, cnt, rr);
            float nthr;
            int ncnt;
            bool done = false;
            if constexpr (!L::kSmemCand && !GROUPED) {
              // large buffers: select the k-th best and compact, no sort (c >= k here: a prune is only
              // asked for when the buffer is close to full)
              if (c >= p.k) done = prune_row_select<CAP>(warp_buf + static_cast<size_t>(rr) * cand_stride, c, p.k, nthr, ncnt);
            }
            if constexpr (GROUPED)
              prune_row_grouped<CAP>(warp_buf + static_cast<size_t>(rr) * cand_stride, L::kSmemCand ? rr : 0, c, p.k,
                                     p.row_group, p.index_base, nthr, ncnt);
            else if (!done)
              prune_row<CAP>(warp_buf + static_cast<size_t>(rr) * cand_stride, L::kSmemCand ? rr : 0, c, p.k, nthr, ncnt,
                             s_reg, i_reg);
            __syncwarp();
            if (lane == rr) {
              cnt = ncnt;
              if (nthr > thr) {
                thr = nthr;
                atomicMax(p.thr_shared + qrow, thr_encode(nthr));
              }
            }
          }
          if (need0) { ISX_PROF_END2(16); ISX_PROF_COUNT(17, 1); }
        };
        // scale one chunk by the inverse norms; maxima of its eight 4-column groups and of the chunk
        auto scale_chunk = [&](uint32_t (&r)[32], int cbase, float (&g)[8]) -> float {
          const float4* rn4 = reinterpret_cast<const float4*>(rn + cbase);
          float vmax = -INFINITY;
#pragma unroll
          for (int j = 0; j < 8; ++j) {
#ifdef ISX_KNN_PROFILE
            const float4 w = (p.debug_skip_select & 2) ? make_float4(0.0625f, 0.0625f, 0.0625f, 0.0625f) : rn4[j];
#else
            const float4 w = rn4[j];
#endif
            mul_f32x2(r[4 * j + 0], r[4 * j + 1], w.x, w.y);
            mul_f32x2(r[4 * j + 2], r[4 * j + 3], w.z, w.w);
            g[j] = fmaxf(fmaxf(__uint_as_float(r[4 * j + 0]), __uint_as_float(r[4 * j + 1])),
                         fmaxf(__uint_as_float(r[4 * j + 2]), __uint_as_float(r[4 * j + 3])));
            vmax = fmaxf(vmax, g[j]);
          }
          return vmax;
        };
        // maxsim: fold one chunk into the running pair (group ids are warp-uniform: one column at a time)
        auto maxsim_chunk = [&](const uint32_t (&r)[32], int cbase, float vmax) {
          if (chunk_uni[cbase >> 5]) {
            const int g = gid_s[cbase];
            if (g != ms_g) { maxsim_flush(); ms_g = g; ms_max = vmax; }
            else ms_max = fmaxf(ms_max, vmax);
            return;
          }
#pragma unroll
          for (int j = 0; j < 32; ++j) {
            const int g = gid_s[cbase + j];
            const float v = __uint_as_float(r[j]);
            if (g != ms_g) { maxsim_flush(); ms_g = g; ms_max = v; }
            else ms_max = fmaxf(ms_max, v);
          }
        };
        // rare path of one chunk
        auto collect_chunk = [&](uint32_t (&r)[32], int cbase, const float (&g)[8], float vmax) {
          if constexpr (MAXSIM) {
            maxsim_chunk(r, cbase, vmax);
            return;
          }
          if (!__any_sync(kFullMask, vmax > thr)) return;
          ISX_PROF_COUNT(10, 1);
          if constexpr (RANGE) {
            range_append(r, vmax > thr, range_rq, qrow, cbase, ncols, gcol0, self_row, p);
            return;
          }
          ISX_PROF_BEGIN1();
          const bool hit = vmax > thr;
          if constexpr (GROUPED) {
            // All 32 rows of the chunk belong to one group (per-cell stores with >= 32 cells per image):
            // only the chunk's best column can represent that group, so a row appends that one entry
            // instead of every column above its threshold.  This is what keeps the correlated cells of
            // the best images, which pass the distinct-group threshold in bulk, from flooding the buffers.
            if (chunk_uni[cbase >> 5]) {
              prune_rows(__ballot_sync(kFullMask, hit && cnt >= CAP));
              if (hit) {
                int jb = 31;
#pragma unroll
                for (int j = 31; j >= 0; --j) jb = (__uint_as_float(r[j]) == vmax) ? j : jb;
                my_buf[cnt ^ my_swz] = make_uint2(__float_as_uint(vmax), static_cast<uint32_t>(gcol0 + cbase + jb));
                ++cnt;
                row_best = fmaxf(row_best, vmax);
              }
              __syncwarp();
              ISX_PROF_END1(13);
              return;
            }
          }
          int ngrp = 0;
#pragma unroll
          for (int j = 0; j < 8; ++j) ngrp += (g[j] > thr) ? 1 : 0;
          ISX_PROF_COUNT(20, __popc(__ballot_sync(kFullMask, hit)));
          if (CAP - kSmallK >= 32 || !__any_sync(kFullMask, hit && 4 * ngrp > CAP - p.k)) {
            prune_rows(__ballot_sync(kFullMask, hit && cnt + 4 * ngrp > CAP));
            ISX_PROF_BEGIN2();
            // chunks that hold neither the end of the store nor a row's own column (all but a handful)
            // append branch-free: one compare and a handful of predicated instructions per column, no
            // dependent chain but the counter.  The walk group by group with its per-group branches
            // costs a single warp ~980 cycles per event (latency of a serial, divergent instruction
            // stream), this one ~750 (-DISX_KNN_PROFILE; k = 100 at d = 256: 10.9 -> 9.9 ms).
            const bool edge = cbase + 32 > ncols || static_cast<uint32_t>(self_row - gcol0 - cbase) < 32u;
            if (!__any_sync(kFullMask, hit && edge)) {
              if (hit) {
                ISX_PROF_COUNT(11, static_cast<unsigned long long>(-cnt));
#pragma unroll
                for (int j = 0; j < 32; ++j) {
                  const bool take = __uint_as_float(r[j]) > thr;
                  if (take) my_buf[cnt ^ my_swz] = make_uint2(r[j], static_cast<uint32_t>(gcol0 + cbase + j));
                  cnt += take ? 1 : 0;
                }
                ISX_PROF_COUNT(11, static_cast<unsigned long long>(cnt));
                row_best = fmaxf(row_best, vmax);  // the chunk's maximum is one of the appended scores
              }
            } else if (hit) {
#pragma unroll
              for (int gi = 0; gi < 8; ++gi) {
                if (g[gi] > thr) {
#pragma unroll
                  for (int e = 0; e < 4; ++e) {
                    const int j = 4 * gi + e;
                    if (__uint_as_float(r[j]) > thr && cbase + j < ncols && gcol0 + cbase + j != self_row) {
                      my_buf[cnt ^ my_swz] = make_uint2(r[j], static_cast<uint32_t>(gcol0 + cbase + j));
                      ++cnt;
                      row_best = fmaxf(row_best, __uint_as_float(r[j]));
                      ISX_PROF_COUNT(11, 1);
                    }
                  }
                }
              }
            }
            __syncwarp();
            ISX_PROF_END2(21);
          } else {
            ISX_PROF_COUNT(19, 1);
#pragma unroll
            for (int h = 0; h < 32 / CHUNK; ++h) {
              prune_rows(__ballot_sync(kFullMask, cnt > CAP - CHUNK));
              if (vmax > thr) {
#pragma unroll
                for (int j = h * CHUNK; j < (h + 1) * CHUNK; ++j) {
                  if (__uint_as_float(r[j]) > thr && cbase + j < ncols && gcol0 + cbase + j != self_row) {
                    my_buf[cnt ^ my_swz] = make_uint2(r[j], static_cast<uint32_t>(gcol0 + cbase + j));
                    ++cnt;
                    row_best = fmaxf(row_best, __uint_as_float(r[j]));
                    ISX_PROF_COUNT(11, 1);
                  }
                }
              }
            }
          }
          ISX_PROF_END1(13);
        };

        ISX_PROF_BEGIN();
        mbar_wait(&tmem_full[acc], acc_phase);
        ISX_PROF_END(4);
        tc_fence_after();
        ISX_PROF_BEGIN();
        const int c0 = eg * kGroupCols;  // this group's first column of the tile
        const uint32_t taddr = tmem_base + (static_cast<uint32_t>(ew * 32) << 16) + acc * BN + c0;
        // (Measured and dropped: loading a group's whole 128-column share first and releasing the stage
        // before any selection: slower, d = 256 5.8 ms against 4.6 — the epilogue is bound by its own
        // instruction stream, ~180 scheduler cycles per 32 columns of which the inverse-norm loads and
        // multiplies are 64, not by the hand-off.  A bound per 4-column group — raw group maximum times
        // the group's largest inverse norm, 30 instructions per chunk in front of the exact scaling —
        // does not pay either: for N(0, 1) rows it passes about twice as often as the exact test.
        // Reading the inverse norms straight from global memory (L1, prefetched a tile ahead) to drop
        // the staging barrier: 10.2 ms against 4.4 at d = 256 — the L1 path cannot feed 8 broadcast
        // 16-byte loads per 32 columns and warp.)
        uint32_t ra[32], rb[32];
        // Software pipeline over the 32-column chunks with two register buffers: the tcgen05.ld of chunk
        // c + 1 is in flight while chunk c is scaled and tested, so a warp's load latency (~300 cycles
        // while the pair's MMAs run) hides behind its own instruction stream instead of relying on the
        // other warp of its scheduler.  Against issuing both loads of a 64-column step together and
        // waiting for both: d = 256 4.51 -> 4.38 ms, d = 64 3.91 -> 3.65 ms, the 500 k x 256 graph
        // 124.9 -> 118.5 ms, 164 -> 148 registers (same box, back to back).
        tmem_ld_32x32(taddr, ra);
#pragma unroll 1
        for (int ld = 0; ld < kGroupCols / 32; ld += 2) {
          const int cb = c0 + ld * 32;
          tc_wait_ld_regs(ra);
          tmem_ld_32x32(taddr + (ld + 1) * 32, rb);
          ISX_PROF_COUNT(9, 2);
#ifdef ISX_KNN_PROFILE
          if (!(p.debug_skip_select & 1))
#endif
          {
            float ga[8];
            const float va = scale_chunk(ra, cb, ga);
            collect_chunk(ra, cb, ga, va);
          }
          tc_wait_ld_regs(rb);
          if (ld + 2 < kGroupCols / 32) {
            tmem_ld_32x32(taddr + (ld + 2) * 32, ra);
          } else {
            // every TMEM read of this tile has landed: release the accumulator stage
            tc_fence_before();
            __syncwarp();
            if (lane == 0) {
              if (NCTA == 2) mbar_arrive_leader(&tmem_empty[acc]); else mbar_arrive(&tmem_empty[acc]);
            }
          }
#ifdef ISX_KNN_PROFILE
          if (!(p.debug_skip_select & 1))
#endif
          {
            float gb[8];
            const float vb = scale_chunk(rb, cb + 32, gb);
            collect_chunk(rb, cb + 32, gb, vb);
          }
        }
        // Off the hand-off path (the accumulator stage is already released): prune the rows whose
        // buffers are more than half-way from k to full, so that a prune inside the next tiles' chunk
        // loops — where it delays the release every other warp of the pair waits for — stays an exception.
        if constexpr (!RANGE && !MAXSIM) prune_rows(__ballot_sync(kFullMask, 2 * cnt > CAP + p.k));
        ISX_PROF_END(6);
        if (++acc == ACC_STAGES) { acc = 0; acc_phase ^= 1; }
      }
      // range search: the hits are in the record buffer already; there is no list to merge
      if constexpr (RANGE) continue;
      // maxsim: the row's last pair of the item; there is no list to merge either
      if constexpr (MAXSIM) {
        maxsim_flush();
        continue;
      }

      // item done: sort every row's candidates and merge the best k into the query's RUNNING list in
      // global memory (under a per-query lock; lists of different items never share a store row, so
      // the union has no duplicates and its top-k does not depend on the merge order).  The k-th best
      // of the running list — of every store row any finished item has seen for this query — is
      // published as the shared bound.  Bounds taken from single items never get past the k-th best
      // of one item's rows (z = 3.1 sigma for 10 k rows against 4.3 sigma for the whole 1 M-row
      // store, i.e. 50 x as many survivors per chunk); with the running list the bound follows the
      // whole store seen so far.
      // Rows whose best candidate is below the bound the grid has reached meanwhile cannot change
      // their running list (the bound is a lower bound of the final k-th best; `>` against the value
      // just below it keeps ties): they skip the sort, the lock and the merge — about half the rows
      // of an item in steady state.
      ISX_PROF_BEGIN();
      uint32_t todo;
      {
        const uint32_t bound_u = row_valid ? *reinterpret_cast<const volatile uint32_t*>(p.thr_shared + qrow) : 0u;
        todo = __ballot_sync(kFullMask, row_valid && cnt > 0 && row_best > thr_decode_below(bound_u));
      }
      if constexpr (E == 1) {
        // 32-entry buffers.  The per-row chain (sort, lock, fence, load, merge, store, fence, unlock) is
        // mostly global-memory latency, so it is run in phases over all rows at once:
        //  A  sort every row; the sorted best k stay in the row's shared-memory buffer;
        //  B  every lane TRIES the lock of its own row once (no lane ever waits while the warp
        //     holds a lock, so warps contending for the same rows cannot deadlock);
        //  C  for the rows whose lock was taken, four at a time: issue the loads of four running
        //     lists, then merge and write them back one after the other;
        //  D  one fence, then every lane publishes its row's bound and releases its lock.
        // Rows whose lock was busy go through B-D again.
        {
          uint32_t t = todo;
          while (t) {
            const int rr = __ffs(t) - 1;
            t &= t - 1;
            __syncwarp();
            const int c = __shfl_sync(kFullMask, cnt, rr);
            float nthr;
            int ncnt;
            if constexpr (GROUPED)
              prune_row_grouped<CAP>(warp_buf + static_cast<size_t>(rr) * cand_stride, L::kSmemCand ? rr : 0, c, p.k,
                                     p.row_group, p.index_base, nthr, ncnt);
            else
              prune_row<CAP>(warp_buf + static_cast<size_t>(rr) * cand_stride, L::kSmemCand ? rr : 0, c, p.k, nthr, ncnt,
                             s_reg, i_reg);
            if (lane == rr) cnt = ncnt;
          }
          __syncwarp();
        }
        ISX_PROF_COUNT(14, __popc(todo));
        ISX_PROF_BEGIN1();
        uint32_t pending = todo;
        uint64_t t0 = 0;
        while (pending) {
          const bool mine = (pending >> lane) & 1u;
          const bool got = mine && atomicCAS(p.run_lock + qrow, 0u, 1u) == 0u;
          uint32_t gotm = __ballot_sync(kFullMask, got);
          if (gotm == 0) {
            __nanosleep(128);
            const uint64_t now = global_timer_ns();
            if (t0 == 0) t0 = now;
            else if (now - t0 > ISX_MBAR_TIMEOUT_NS) {
              if (lane == 0) printf("isx: knn_search_kernel: running-list locks timed out (rows %08x of block %d)\n", pending, m0);
              __trap();
            }
            continue;
          }
          pending &= ~gotm;
          __threadfence();
          float kth_mine = -INFINITY;
          bool kth_valid_mine = false;
          const int slot = CAP - 1 - lane;  // the running list's entry this lane holds in the bitonic input
          while (gotm) {
            int rows[4];
            float ls[4];
            int li[4];
#pragma unroll
            for (int b = 0; b < 4; ++b) {
              rows[b] = gotm ? __ffs(gotm) - 1 : -1;
              if (gotm) gotm &= gotm - 1;
              ls[b] = -INFINITY;
              li[b] = -1;
              if (rows[b] >= 0 && slot < p.k) {
                const size_t base = static_cast<size_t>(m0 + ew * 32 + rows[b]) * p.k;
                li[b] = __ldcg(p.run_idx + base + slot);
                ls[b] = __ldcg(p.run_scores + base + slot);
              }
            }
#pragma unroll
            for (int b = 0; b < 4; ++b) {
              if (rows[b] < 0) continue;  // warp-uniform
              const int rr = rows[b];
              const int c = __shfl_sync(kFullMask, cnt, rr);
              const uint2* buf = warp_buf + static_cast<size_t>(rr) * cand_stride;
              float sv = -INFINITY;
              int iv = INT_MAX;
              if (lane < c) {
                const uint2 v = buf[lane ^ (L::kSmemCand ? rr : 0)];
                sv = __uint_as_float(v.x);
                iv = static_cast<int>(v.y);
              }
              if (li[b] >= 0) { sv = ls[b]; iv = li[b]; }
              if constexpr (GROUPED) {
                // the item's groups and the running list's groups may overlap: rank the union with
                // de-duplication and store the best k groups; no bound while fewer than k are present
                int distinct;
                const int rank = grouped_rank32(sv, iv, row_group_of(p.row_group, p.index_base, iv), distinct);
                const size_t base = static_cast<size_t>(m0 + ew * 32 + rr) * p.k;
                __syncwarp();
                if (rank >= 0 && rank < p.k) {
                  p.run_scores[base + rank] = sv;
                  p.run_idx[base + rank] = iv;
                }
                if (lane >= distinct && lane < p.k) {
                  p.run_scores[base + lane] = -INFINITY;
                  p.run_idx[base + lane] = -1;
                }
                const uint32_t km = __ballot_sync(kFullMask, rank == p.k - 1);
                const float cs = km ? __shfl_sync(kFullMask, sv, __ffs(km) - 1) : -INFINITY;
                if (lane == rr) { kth_mine = cs; kth_valid_mine = km != 0; }
                continue;
              }
              s_reg[0] = sv;
              i_reg[0] = iv;
              warp_merge_desc<E>(s_reg, i_reg);
              const size_t base = static_cast<size_t>(m0 + ew * 32 + rr) * p.k;
              if (lane < p.k) {
                p.run_scores[base + lane] = s_reg[0];
                p.run_idx[base + lane] = (i_reg[0] != INT_MAX) ? i_reg[0] : -1;
              }
              const float cs = __shfl_sync(kFullMask, s_reg[0], p.k - 1);
              const int ci = __shfl_sync(kFullMask, i_reg[0], p.k - 1);
              if (lane == rr) { kth_mine = cs; kth_valid_mine = ci != INT_MAX; }
            }
          }
          __threadfence();
          __syncwarp();
          if (got) {
            if (kth_valid_mine) atomicMax(p.thr_shared + qrow, thr_encode(kth_mine));
            atomicExch(p.run_lock + qrow, 0u);
          }
          ISX_PROF_COUNT(15, 1);
        }
        ISX_PROF_END1(18);
      } else {
        // 256-entry buffers (k > 16), the same phase structure: the per-row chain used to be
        // sort -> lock spin -> fence -> running-list loads -> merge -> stores -> fence -> unlock, ~18 k cycles
        // a row and 32 rows in sequence (measured at k = 100: 1357 cycles per tile, 8.6 % of the kernel, with
        // the MMAs stalled behind two full accumulator stages meanwhile).  Now
        //  A  every row is sorted first; its best k stay in the row's buffer (global memory, L2);
        //  B  every lane TRIES the lock of its own row once;
        //  C  the rows whose lock was taken are merged one after the other (bitonic merge with the
        //     running list) without any lock or fence latency in between;
        //  D  one fence, then every lane publishes its row's bound and releases its lock.
        {
          // A: a row's buffer holds everything that beat the row's threshold when it was appended; by
          // now the grid's bound for the query (the k-th best of every finished item's rows) is usually
          // higher.  Entries below it can never reach the final top-k: they are dropped first, and only
          // the survivors (a few dozen of up to 256, k / i of them for the i-th item of a query) are
          // sorted, in the smallest network that holds them — the 256-entry sort was 17 k cycles a row.
          uint32_t t = todo;
          while (t) {
            const int rr = __ffs(t) - 1;
            t &= t - 1;
            __syncwarp();
            const int c = __shfl_sync(kFullMask, cnt, rr);
            const int qr = m0 + ew * 32 + rr;
            uint2* buf = warp_buf + static_cast<size_t>(rr) * cand_stride;
            const float bound = thr_decode_below(*reinterpret_cast<const volatile uint32_t*>(p.thr_shared + qr));
            uint2 v[E];
            uint32_t keepm = 0;
#pragma unroll
            for (int e = 0; e < E; ++e) {
              const int i = e * 32 + lane;
              v[e] = make_uint2(0u, 0u);
              if (i < c) {
                v[e] = buf[i];
                if (__uint_as_float(v[e].x) > bound) keepm |= 1u << e;
              }
            }
            __syncwarp();
            int kept = 0;
#pragma unroll
            for (int e = 0; e < E; ++e) {
              const bool kp = (keepm >> e) & 1u;
              const uint32_t bal = __ballot_sync(kFullMask, kp);
              if (kp) buf[kept + __popc(bal & ((1u << lane) - 1u))] = v[e];
              kept += __popc(bal);
            }
            __syncwarp();
            float nthr;
            int ncnt;
            if constexpr (GROUPED) {
              if (kept <= 32) prune_row_grouped<32>(buf, 0, kept, p.k, p.row_group, p.index_base, nthr, ncnt);
              else if (kept <= 64) prune_row_grouped<64>(buf, 0, kept, p.k, p.row_group, p.index_base, nthr, ncnt);
              else if (kept <= 128) prune_row_grouped<128>(buf, 0, kept, p.k, p.row_group, p.index_base, nthr, ncnt);
              else prune_row_grouped<CAP>(buf, 0, kept, p.k, p.row_group, p.index_base, nthr, ncnt);
            } else if (kept <= 32) {
              float s1[1];
              int i1[1];
              prune_row<32>(buf, 0, kept, p.k, nthr, ncnt, s1, i1);
            } else if (kept <= 64) {
              float s2[2];
              int i2[2];
              prune_row<64>(buf, 0, kept, p.k, nthr, ncnt, s2, i2);
            } else if (kept <= 128) {
              float s4[4];
              int i4[4];
              prune_row<128>(buf, 0, kept, p.k, nthr, ncnt, s4, i4);
            } else {
              prune_row<CAP>(buf, 0, kept, p.k, nthr, ncnt, s_reg, i_reg);
            }
            if (lane == rr) cnt = ncnt;
          }
          __syncwarp();
        }
        ISX_PROF_COUNT(14, __popc(todo));
        uint32_t pending = todo & __ballot_sync(kFullMask, cnt > 0);
        uint64_t t0 = 0;
        while (pending) {
          const bool mine = (pending >> lane) & 1u;
          const bool got = mine && atomicCAS(p.run_lock + qrow, 0u, 1u) == 0u;
          uint32_t gotm = __ballot_sync(kFullMask, got);
          if (gotm == 0) {
            __nanosleep(128);
            const uint64_t now = global_timer_ns();
            if (t0 == 0) t0 = now;
            else if (now - t0 > ISX_MBAR_TIMEOUT_NS) {
              if (lane == 0) printf("isx: knn_search_kernel: running-list locks timed out (rows %08x of block %d)\n", pending, m0);
              __trap();
            }
            continue;
          }
          pending &= ~gotm;
          __threadfence();
          float kth_mine = -INFINITY;
          bool kth_valid_mine = false;
          while (gotm) {
            const int rr = __ffs(gotm) - 1;
            gotm &= gotm - 1;
            const int c = __shfl_sync(kFullMask, cnt, rr);
            const int qr = m0 + ew * 32 + rr;
            const uint2* buf = warp_buf + static_cast<size_t>(rr) * cand_stride;
            float* gs = p.run_scores + static_cast<size_t>(qr) * p.k;
            int32_t* gi = p.run_idx + static_cast<size_t>(qr) * p.k;
            // bitonic input: slots [0, c) this item's best (sorted descending, c <= k), the running list
            // reversed at the top (slot CAP-1-j = its j-th best), (-inf, none) in between
#pragma unroll
            for (int e = 0; e < E; ++e) {
              const int i = e * 32 + lane;
              float sv = -INFINITY;
              int iv = INT_MAX;
              if (i < c) {
                const uint2 v = buf[i];
                sv = __uint_as_float(v.x);
                iv = static_cast<int>(v.y);
              }
              const int j = CAP - 1 - i;
              if (j < p.k) {
                const int id = __ldcg(gi + j);
                const float sc = __ldcg(gs + j);
                if (id >= 0) { sv = sc; iv = id; }
              }
              s_reg[e] = sv;
              i_reg[e] = iv;
            }
            if constexpr (GROUPED) {
              // the union may hold a group twice (once from this item, once from the running list);
              // dropped entries sort last as (-inf, none), so slot k-1 is empty while fewer than k remain
              int g_reg[E];
#pragma unroll
              for (int e = 0; e < E; ++e) g_reg[e] = row_group_of(p.row_group, p.index_base, i_reg[e]);
              grouped_select<E>(s_reg, i_reg, g_reg);
            } else {
              warp_merge_desc<E>(s_reg, i_reg);
            }
            float kth = -INFINITY;
            bool kth_valid = false;
#pragma unroll
            for (int e = 0; e < E; ++e) {
              const int i = e * 32 + lane;
              if (i < p.k) {
                gs[i] = s_reg[e];
                gi[i] = (i_reg[e] != INT_MAX) ? i_reg[e] : -1;
              }
              const float cs = __shfl_sync(kFullMask, s_reg[e], (p.k - 1) & 31);
              const int ci = __shfl_sync(kFullMask, i_reg[e], (p.k - 1) & 31);
              if (e == ((p.k - 1) >> 5)) { kth = cs; kth_valid = ci != INT_MAX; }
            }
            if (lane == rr) { kth_mine = kth; kth_valid_mine = kth_valid; }
          }
          __threadfence();
          __syncwarp();
          if (got) {
            if (kth_valid_mine) atomicMax(p.thr_shared + qrow, thr_encode(kth_mine));
            atomicExch(p.run_lock + qrow, 0u);
          }
          ISX_PROF_COUNT(15, 1);
        }
      }
      __syncwarp();
      ISX_PROF_END(8);
    }
    if (warp == kEpilogueWarp0 && lane == 0 && rank == 0) {
      ISX_PROF_FLUSH(4); ISX_PROF_FLUSH(5); ISX_PROF_FLUSH(6); ISX_PROF_FLUSH(8);
      ISX_PROF_FLUSH(9); ISX_PROF_FLUSH(10); ISX_PROF_FLUSH(11); ISX_PROF_FLUSH(12); ISX_PROF_FLUSH(16); ISX_PROF_FLUSH(17); ISX_PROF_FLUSH(18); ISX_PROF_FLUSH(19); ISX_PROF_FLUSH(20); ISX_PROF_FLUSH(21); ISX_PROF_FLUSH(22); ISX_PROF_FLUSH(13); ISX_PROF_FLUSH(14); ISX_PROF_FLUSH(15);
    }
#ifdef ISX_KNN_PROFILE
    if (warp == kEpilogueWarp0 && rank == 0) {  // appends: summed over the warp's 32 rows
      unsigned long long a = prof_acc[11];
      for (int o = 16; o > 0; o >>= 1) a += __shfl_xor_sync(kFullMask, a, o);
      if (lane == 0) atomicAdd(p.prof + 11, a);
    }
#endif
  }
#ifdef ISX_KNN_PROFILE
  if (threadIdx.x == 0 && rank == 0) atomicAdd(p.prof + 7, static_cast<unsigned long long>(clock64() - prof_kernel_t0));
#endif

  tc_fence_before();
  if (NCTA == 2) cluster_sync_all(); else __syncthreads();  // a pair's CTAs may not exit while the peer uses them
  if (warp == 2) {
    tc_fence_after();
    if (NCTA == 2) tmem_dealloc_pair(tmem_base, 512); else tmem_dealloc(tmem_base, 512);
  }
}

template <int CAP, int NCTA, bool RES>
__global__ void __launch_bounds__(knn_threads(CAP), 1)
knn_search_kernel(const __grid_constant__ CUtensorMap tmap_q, const __grid_constant__ CUtensorMap tmap_e,
                  const KnnParams p) {
  knn_search_body<CAP, NCTA, RES, false>(tmap_q, tmap_e, p);
}

template <int CAP, int NCTA, bool RES>
__global__ void __launch_bounds__(knn_threads(CAP), 1)
knn_search_grouped_kernel(const __grid_constant__ CUtensorMap tmap_q, const __grid_constant__ CUtensorMap tmap_e,
                          const KnnParams p) {
  knn_search_body<CAP, NCTA, RES, true>(tmap_q, tmap_e, p);
}

template <int NCTA, bool RES>
__global__ void __launch_bounds__(knn_threads(32), 1)
knn_range_kernel(const __grid_constant__ CUtensorMap tmap_q, const __grid_constant__ CUtensorMap tmap_e,
                 const KnnParams p) {
  knn_search_body<32, NCTA, RES, false, true>(tmap_q, tmap_e, p);
}

template <int CAP, int NCTA, bool RES>
__global__ void __launch_bounds__(knn_threads(CAP), 1)
knn_search_fp8_kernel(const __grid_constant__ CUtensorMap tmap_q, const __grid_constant__ CUtensorMap tmap_e,
                      const KnnParams p) {
  knn_search_body<CAP, NCTA, RES, false, false, true>(tmap_q, tmap_e, p);
}

template <int NCTA, bool RES>
__global__ void __launch_bounds__(knn_threads(32), 1)
knn_maxsim_kernel(const __grid_constant__ CUtensorMap tmap_q, const __grid_constant__ CUtensorMap tmap_e,
                  const KnnParams p) {
  knn_search_body<32, NCTA, RES, false, false, false, true>(tmap_q, tmap_e, p);
}

// ------------------------------------------------------------------------------------------
// K5: merge g sorted-or-not partial lists per query into the final top-k.  One warp per query.
// ------------------------------------------------------------------------------------------
// Finalising straight into peer memory: the packed records of this rank are stored into slot
// `slot_off` of every peer's gather buffer over NVLink (peer-mapped device pointers), so that
// "finalise + all-gather" is one kernel and the ranks only need a barrier before they merge.
constexpr int kMaxPeers = 16;
struct PeerOut {
  uint2* ptr[kMaxPeers];
  int n;
  long long slot_off;  // in records
};

// Partial lists come either as two arrays (scores fp32, idx int32) or — idx == nullptr — as packed
// 8-byte records {fp32 score, int32 index} (what one all-gather moves); the result likewise
// (out_idx == nullptr: packed records at out_scores).
template <int CAP>
__global__ void __launch_bounds__(128)
topk_merge_kernel(const float* __restrict__ scores, const int32_t* __restrict__ idx, int g, int q, int k,
                  const float* __restrict__ query_scale, float* __restrict__ out_scores,
                  int32_t* __restrict__ out_idx, const PeerOut peers) {
  constexpr int E = CAP / 32;
  const int lane = threadIdx.x & 31;
  const int query = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (query >= q) return;
  // registers hold a sorted window of CAP entries; the best `keep` survive each round and the
  // remaining CAP - keep slots are refilled with fresh candidates
  const int keep = k;
  const int fresh = CAP - keep;
  // the search's running lists hold raw scores: scale them by the query's inverse norm here
  const float qscale = query_scale ? query_scale[query] : 1.0f;
  const uint2* rec = reinterpret_cast<const uint2*>(scores);
  float s[E];
  int id[E];
#pragma unroll
  for (int e = 0; e < E; ++e) { s[e] = -INFINITY; id[e] = INT_MAX; }
  const long long total = static_cast<long long>(g) * k;
  for (long long base = 0; base < total; base += fresh) {
#pragma unroll
    for (int e = 0; e < E; ++e) {
      const int pos = e * 32 + lane;
      if (pos >= keep) {
        const long long c = base + (pos - keep);
        float sv = -INFINITY;
        int iv = INT_MAX;
        if (c < total) {
          const long long part = c / k, j = c - part * k;
          const size_t off = (static_cast<size_t>(part) * q + query) * k + j;
          if (idx) {
            const int raw = idx[off];
            if (raw >= 0) { sv = scores[off] * qscale; iv = raw; }
          } else {
            const uint2 v = rec[off];
            if (static_cast<int>(v.y) >= 0) { sv = __uint_as_float(v.x) * qscale; iv = static_cast<int>(v.y); }
          }
        }
        s[e] = sv;
        id[e] = iv;
      }
    }
    warp_sort_desc<E>(s, id);
  }
#pragma unroll
  for (int e = 0; e < E; ++e) {
    const int pos = e * 32 + lane;
    if (pos < k) {
      const bool have = id[e] != INT_MAX;
      const float sv = have ? s[e] : -INFINITY;
      const int iv = have ? id[e] : -1;
      const size_t o = static_cast<size_t>(query) * k + pos;
      const uint2 rec2 = make_uint2(__float_as_uint(sv), static_cast<uint32_t>(iv));
      if (peers.n > 0) {
#pragma unroll 1
        for (int pi = 0; pi < peers.n; ++pi) peers.ptr[pi][peers.slot_off + o] = rec2;
      } else if (out_idx) { out_scores[o] = sv; out_idx[o] = iv; }
      else reinterpret_cast<uint2*>(out_scores)[o] = rec2;
    }
  }
}

int launch_merge(const float* scores, const int32_t* idx, int g, int q, int k, const float* query_scale,
                 float* out_scores, int32_t* out_idx, cudaStream_t stream, const PeerOut* peers_in = nullptr) {
  const int warps_per_block = 4;
  const int blocks = (q + warps_per_block - 1) / warps_per_block;
  PeerOut peers;
  peers.n = 0;
  peers.slot_off = 0;
  if (peers_in) peers = *peers_in;
  if (k <= 32)
    topk_merge_kernel<64><<<blocks, 128, 0, stream>>>(scores, idx, g, q, k, query_scale, out_scores, out_idx, peers);
  else
    topk_merge_kernel<256><<<blocks, 128, 0, stream>>>(scores, idx, g, q, k, query_scale, out_scores, out_idx, peers);
  ISX_CHECK_CUDA(cudaGetLastError());
  return ISX_OK;
}

// Grouped form: merge g partial lists of (score, row, group) into the k best groups per query, one
// entry per group (its first in (score desc, row asc) order).  Input either as 12-byte records
// {fp32 score bits, row, group} (`records`, what one all-gather of grouped results moves) or as the
// search's running lists (`scores`, `idx`), whose groups are looked up in `row_group` (store-local
// rows, idx - index_base) and whose raw scores are scaled by `query_scale`.  A group that appears in
// several lists (cut by a shard or N-split boundary) comes out once.  Padding: idx < 0.
template <int CAP>
__global__ void __launch_bounds__(128)
topk_merge_grouped_kernel(const int32_t* __restrict__ records, const float* __restrict__ scores,
                          const int32_t* __restrict__ idx, const int32_t* __restrict__ row_group, int index_base,
                          int g, int q, int k, const float* __restrict__ query_scale, float* __restrict__ out_scores,
                          int32_t* __restrict__ out_rows, int32_t* __restrict__ out_groups) {
  constexpr int E = CAP / 32;
  const int lane = threadIdx.x & 31;
  const int query = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (query >= q) return;
  // the window keeps the best k groups of everything read so far; CAP - k slots take fresh entries
  const int fresh = CAP - k;
  const float qscale = query_scale ? query_scale[query] : 1.0f;
  float s[E];
  int id[E], gr[E];
#pragma unroll
  for (int e = 0; e < E; ++e) { s[e] = -INFINITY; id[e] = INT_MAX; gr[e] = -1; }
  const long long total = static_cast<long long>(g) * k;
  for (long long base = 0; base < total; base += fresh) {
#pragma unroll
    for (int e = 0; e < E; ++e) {
      const int pos = e * 32 + lane;
      if (pos >= k) {
        const long long c = base + (pos - k);
        s[e] = -INFINITY;
        id[e] = INT_MAX;
        gr[e] = -1;
        if (c < total) {
          const long long part = c / k, j = c - part * k;
          const size_t off = (static_cast<size_t>(part) * q + query) * k + j;
          if (records) {
            const int3 v = *reinterpret_cast<const int3*>(records + 3 * off);
            if (v.y >= 0) { s[e] = __int_as_float(v.x) * qscale; id[e] = v.y; gr[e] = v.z; }
          } else {
            const int raw = idx[off];
            if (raw >= 0) { s[e] = scores[off] * qscale; id[e] = raw; gr[e] = row_group[raw - index_base]; }
          }
        }
      }
    }
    grouped_select<E>(s, id, gr);
  }
#pragma unroll
  for (int e = 0; e < E; ++e) {
    const int pos = e * 32 + lane;
    if (pos < k) {
      const bool have = id[e] != INT_MAX;
      const size_t o = static_cast<size_t>(query) * k + pos;
      out_scores[o] = have ? s[e] : -INFINITY;
      out_rows[o] = have ? id[e] : -1;
      out_groups[o] = have ? gr[e] : -1;
    }
  }
}

int launch_merge_grouped(const int32_t* records, const float* scores, const int32_t* idx, const int32_t* row_group,
                         int index_base, int g, int q, int k, const float* query_scale, float* out_scores,
                         int32_t* out_rows, int32_t* out_groups, cudaStream_t stream) {
  const int blocks = (q + 3) / 4;
  if (k <= 32)
    topk_merge_grouped_kernel<64><<<blocks, 128, 0, stream>>>(records, scores, idx, row_group, index_base, g, q, k,
                                                              query_scale, out_scores, out_rows, out_groups);
  else
    topk_merge_grouped_kernel<256><<<blocks, 128, 0, stream>>>(records, scores, idx, row_group, index_base, g, q, k,
                                                               query_scale, out_scores, out_rows, out_groups);
  ISX_CHECK_CUDA(cudaGetLastError());
  return ISX_OK;
}

// ------------------------------------------------------------------------------------------
// K5r: exact re-score of candidate lists (the second stage of the fp8 search).  One warp per query:
// every candidate row (global; -1 and rows outside the store are skipped) gets the bf16 dot product
// in fp32 — each lane sums its 8-element slices in a fixed order, then a butterfly, so every lane
// holds the same bits — and score = fl(fl(dot * rnorm_e) * rnorm_q), the epilogue's and K5's product
// order.  The best k by (score desc, row asc) are written, padded with (-inf, -1); a row listed twice
// comes out once.  Nothing depends on timing: repeated calls give identical bits.
// ------------------------------------------------------------------------------------------
template <int E>
__global__ void __launch_bounds__(128)
rescore_kernel(const __nv_bfloat16* __restrict__ store, const float* __restrict__ rnorm, long long n,
               const __nv_bfloat16* __restrict__ queries, const float* __restrict__ qrnorm, int q, int d,
               const int32_t* __restrict__ cand, int kc, int index_base, int k, float* __restrict__ out_scores,
               int32_t* __restrict__ out_idx) {
  const int lane = threadIdx.x & 31;
  const int query = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (query >= q) return;
  const __nv_bfloat16* qp = queries + static_cast<size_t>(query) * d;
  const float rq = qrnorm[query];
  float s[E];
  int id[E];
#pragma unroll
  for (int e = 0; e < E; ++e) {
    s[e] = -INFINITY;
    id[e] = INT_MAX;
    const int j0 = e * 32;
    const int mine = (j0 + lane < kc) ? cand[static_cast<size_t>(query) * kc + j0 + lane] : -1;
    const int cnt = min(32, kc - j0);
#pragma unroll 1
    for (int l = 0; l < cnt; ++l) {
      const int r = __shfl_sync(kFullMask, mine, l);
      const long long local = static_cast<long long>(r) - index_base;
      if (r < 0 || local < 0 || local >= n) continue;  // warp-uniform
      const __nv_bfloat16* ep = store + local * d;
      float acc = 0.f;
#pragma unroll 4
      for (int i = lane * 8; i < d; i += 256) {
        const uint4 a = ld_nc_v4(ep + i), b = ld_nc_v4(qp + i);
        const uint32_t wa[4] = {a.x, a.y, a.z, a.w}, wb[4] = {b.x, b.y, b.z, b.w};
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          acc = fmaf(__uint_as_float(wa[j] << 16), __uint_as_float(wb[j] << 16), acc);
          acc = fmaf(__uint_as_float(wa[j] & 0xFFFF0000u), __uint_as_float(wb[j] & 0xFFFF0000u), acc);
        }
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(kFullMask, acc, o);
      if (lane == l) {
        s[e] = __fmul_rn(__fmul_rn(acc, __ldg(rnorm + local)), rq);
        id[e] = r;
      }
    }
  }
  warp_sort_desc<E>(s, id);
  // a row listed twice sorts next to its copy: drop the later one and sort again (rare)
  bool dup[E];
  bool any = false;
  int carry = INT_MAX;  // row of element e * 32 - 1
#pragma unroll
  for (int e = 0; e < E; ++e) {
    const int up = __shfl_up_sync(kFullMask, id[e], 1);
    const int prev = lane ? up : carry;
    carry = __shfl_sync(kFullMask, id[e], 31);
    dup[e] = id[e] != INT_MAX && id[e] == prev;
    any |= dup[e];
  }
  if (__any_sync(kFullMask, any)) {
#pragma unroll
    for (int e = 0; e < E; ++e) {
      if (dup[e]) { s[e] = -INFINITY; id[e] = INT_MAX; }
    }
    warp_sort_desc<E>(s, id);
  }
#pragma unroll
  for (int e = 0; e < E; ++e) {
    const int pos = e * 32 + lane;
    if (pos < k) {
      const bool have = id[e] != INT_MAX;
      out_scores[static_cast<size_t>(query) * k + pos] = have ? s[e] : -INFINITY;
      out_idx[static_cast<size_t>(query) * k + pos] = have ? id[e] : -1;
    }
  }
  for (int pos = 32 * E + lane; pos < k; pos += 32) {
    out_scores[static_cast<size_t>(query) * k + pos] = -INFINITY;
    out_idx[static_cast<size_t>(query) * k + pos] = -1;
  }
}

// ------------------------------------------------------------------------------------------
// K6: set scores and top-k of multi-vector (maxsim) search.  One CTA per query set S = rows [s0, s1):
// a thread owns the columns col0 + tid, col0 + tid + 256, ... (consecutive threads read consecutive
// columns of a cell_max row) and scores each as
//   score = fl(sum over c = s0 .. s1-1, in that order, of fl(cell_max[c][col] * rnorm_q[c])) / |S|
// (fp32 adds and a correctly rounded divide: no contraction, no reordering).  A column whose score is
// -inf (a group without rows) is not a result.  The CTA keeps its best k in shared memory, sorted by
// (score desc, group asc); a round of 256 columns with any column that sorts before the k-th appends
// those to the list and re-sorts the 512 slots (bitonic).  Output: k packed records {score bits,
// group_base + col} per set, padded with (-inf, -1): the format isx_topk_merge_packed merges.
// ------------------------------------------------------------------------------------------
constexpr int kSetThreads = 256;
constexpr int kSetSlots = 512;  // k <= 128 kept + 256 fresh, rounded up to a power of two

__global__ void __launch_bounds__(kSetThreads)
maxsim_sets_topk_kernel(const float* __restrict__ cell_max, const float* __restrict__ qrnorm, int q, long long ld,
                        int col0, int col1, const int64_t* __restrict__ set_off, int k, int group_base,
                        uint2* __restrict__ records) {
  __shared__ float ls[kSetSlots];
  __shared__ int li[kSetSlots];
  const int tid = threadIdx.x;
  const int set = blockIdx.x;
  // offsets come from the caller: clamp them to the matrix so that a malformed set reads nothing outside it
  const long long lo = set_off[set], hi = set_off[set + 1];
  const long long s0 = min(max(lo, 0ll), static_cast<long long>(q));
  const long long s1 = min(max(hi, s0), static_cast<long long>(q));
  for (int i = tid; i < kSetSlots; i += kSetThreads) { ls[i] = -INFINITY; li[i] = INT_MAX; }
  __syncthreads();
  const float set_size = static_cast<float>(s1 - s0);  // exact below 2^24
  if (s1 > s0) {
    for (int base = col0; base < col1; base += kSetThreads) {
      const int c = base + tid;
      float sc = -INFINITY;
      const int id = group_base + c;
      if (c < col1) {
        const float* col = cell_max + c;
        float sum = 0.f;
#pragma unroll 8
        for (long long r = s0; r < s1; ++r) sum = __fadd_rn(sum, __fmul_rn(__ldg(col + r * ld), __ldg(qrnorm + r)));
        sc = __fdiv_rn(sum, set_size);
      }
      const bool cand = sc > -INFINITY && pair_before(sc, id, ls[k - 1], li[k - 1]);
      if (__syncthreads_or(cand)) {
        ls[k + tid] = cand ? sc : -INFINITY;
        li[k + tid] = cand ? id : INT_MAX;
        __syncthreads();
        for (int size = 2; size <= kSetSlots; size <<= 1) {
          for (int stride = size >> 1; stride > 0; stride >>= 1) {
            const int i = 2 * tid - (tid & (stride - 1));
            const int j = i + stride;
            const bool desc = (i & size) == 0;
            const float si = ls[i], sj = ls[j];
            const int ii = li[i], ij = li[j];
            if (desc ? pair_before(sj, ij, si, ii) : pair_before(si, ii, sj, ij)) {
              ls[i] = sj; ls[j] = si; li[i] = ij; li[j] = ii;
            }
            __syncthreads();
          }
        }
        for (int i = k + tid; i < kSetSlots; i += kSetThreads) { ls[i] = -INFINITY; li[i] = INT_MAX; }
        __syncthreads();
      }
    }
  }
  for (int j = tid; j < k; j += kSetThreads) {
    const bool have = li[j] != INT_MAX;
    records[static_cast<size_t>(set) * k + j] =
        make_uint2(__float_as_uint(have ? ls[j] : -INFINITY), static_cast<uint32_t>(have ? li[j] : -1));
  }
}

__global__ void __launch_bounds__(256) fill_f32_kernel(float* __restrict__ x, long long n, float v) {
  for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < n;
       i += static_cast<long long>(gridDim.x) * blockDim.x)
    x[i] = v;
}

size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

struct KnnWorkspace {
  size_t run_scores_off, run_idx_off, zero_off, zero_bytes, cand_off, total;
};

// Offsets depend on (q, k) only — not on the store block — so that a search can be CONTINUED over
// several store blocks with the same workspace (ISX_KNN_CONTINUE).  `max_grid` = the SM count.
KnnWorkspace knn_workspace(int max_grid, int q, int k) {
  KnnWorkspace w;
  size_t off = 0;
  w.run_scores_off = off;
  off = align_up(off + static_cast<size_t>(q) * k * sizeof(float), 256);
  w.run_idx_off = off;  // set to -1 (empty) before every search
  off = align_up(off + static_cast<size_t>(q) * k * sizeof(int32_t), 256);
  w.zero_off = off;  // thr_shared[q], progress[256], run_lock[q]: zeroed together before every search
  w.zero_bytes = (2 * static_cast<size_t>(q) + 256) * sizeof(uint32_t);
  off = align_up(off + w.zero_bytes, 256);
  w.cand_off = off;
  if (k > kSmallK) off = align_up(off + static_cast<size_t>(max_grid) * epi_groups(256) * BM * 256 * sizeof(uint2), 256);
  w.total = off + 256;
  return w;
}

template <int CAP, int NCTA, bool RES = false, bool GROUPED = false, bool RANGE = false, bool F8 = false,
          bool MAXSIM = false>
int launch_search(const CUtensorMap& tq, const CUtensorMap& te, const KnnParams& p, int grid, cudaStream_t stream) {
  static_assert(!RANGE || (CAP == 32 && !GROUPED), "range search has the CAP = 32 plan only");
  static_assert(!F8 || (!GROUPED && !RANGE), "the fp8 scan is a plain search");
  static_assert(!MAXSIM || (CAP == 32 && !GROUPED && !RANGE && !F8), "maxsim has the CAP = 32 plan only");
  auto kern = MAXSIM ? knn_maxsim_kernel<NCTA, RES>
              : F8   ? knn_search_fp8_kernel<CAP, NCTA, RES>
              : RANGE ? knn_range_kernel<NCTA, RES>
                      : GROUPED ? knn_search_grouped_kernel<CAP, NCTA, RES> : knn_search_kernel<CAP, NCTA, RES>;
  const int smem = static_cast<int>(KnnSmem<CAP, NCTA, RES, GROUPED, RANGE, MAXSIM>::kDynamicBytes);
  ISX_CHECK_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(static_cast<unsigned>(grid));
  cfg.blockDim = dim3(knn_threads(CAP));
  cfg.dynamicSmemBytes = static_cast<size_t>(smem);
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = NCTA;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  ISX_CHECK_CUDA(cudaLaunchKernelEx(&cfg, kern, tq, te, p));
  return ISX_OK;
}

// Lockstep window in tiles: measured best 16-32 at bf16 d = 1280 (640 KB of store rows per tile); it is
// a footprint in L2, so it scales with 1 / row bytes, and the poll interval (a third of it, rounded down
// to a power of two) with it: one poll reads every unit's counter, ~1 us, against 0.6 us per tile at
// bf16 d = 256.
void set_throttle(KnnParams& p, int row_bytes) {
  constexpr uint32_t base = 24;
  const uint64_t scaled = static_cast<uint64_t>(base) * 2560u / static_cast<uint32_t>(std::max(row_bytes, 128));
  p.throttle_window = static_cast<uint32_t>(std::min<uint64_t>(std::max<uint64_t>(scaled, base), 1u << 30));
  uint32_t every = 8;
  while (every * 2 <= p.throttle_window / 3 && every < 1024) every *= 2;
  p.throttle_every = every;
}

#ifdef ISX_KNN_PROFILE
// Diagnostic build: every launch of the shared K4 body (search, grouped and range) flushes its wait
// counters into p.prof, so every entry point sets it.
int set_profile(KnnParams& p, cudaStream_t stream) {
  static unsigned long long* d_prof = nullptr;
  if (!d_prof) ISX_CHECK_CUDA(cudaMalloc(&d_prof, 24 * sizeof(unsigned long long)));
  ISX_CHECK_CUDA(cudaMemsetAsync(d_prof, 0, 24 * sizeof(unsigned long long), stream));
  p.prof = d_prof;
  p.debug_skip_select = getenv("ISX_KNN_SKIP_SELECT") ? atoi(getenv("ISX_KNN_SKIP_SELECT")) : 0;
  return ISX_OK;
}
#endif

// CTA pairs halve the shared-memory fill and operand-read traffic per SM (each CTA stages half of
// every store tile).  They need at least two 128-query blocks to pay off.
int knn_ncta(int q) { return q > BM ? 2 : 1; }

// Argument checks every search entry point (plain, grouped, range) makes.
int check_search_args(const char* fn, const void* store, int64_t n, const void* queries, int q, int d,
                      int64_t index_base, int64_t query_index_base, bool no_self) {
  ISX_REQUIRE(d % 8 == 0, "%s: d = %d must be a multiple of 8 (16-byte rows for TMA)", fn, d);
  ISX_REQUIRE(n < (1ll << 31) - BN, "%s: at most 2^31 store rows per call (n=%lld); shard the store", fn, (long long)n);
  ISX_REQUIRE(index_base >= 0 && index_base + n < (1ll << 31), "%s: index_base + n must fit in int32", fn);
  ISX_REQUIRE(!no_self || (query_index_base >= 0 && query_index_base + q < (1ll << 31)),
              "%s: query_index_base + q must fit in int32 (got %lld)", fn, (long long)query_index_base);
  ISX_REQUIRE((reinterpret_cast<uintptr_t>(queries) & 15u) == 0 && (reinterpret_cast<uintptr_t>(store) & 15u) == 0,
              "%s: store and queries must be 16-byte aligned", fn);
  return ISX_OK;
}

// What a search launch needs beyond its workspace: the variant's CTA count, the plan, the two tensor
// maps and the parameters every entry point sets alike.
struct KnnLaunch {
  int ncta;
  KnnPlan plan;
  CUtensorMap tq, te;
  KnnParams p;
};

// k is the length of the running lists (kSmallK for range search, which runs the k <= kSmallK variant).
// dtype: BFLOAT16 for bf16 rows; UINT16 for the fp8 scan, whose E4M3 rows are moved as 16-bit pairs
// (d = d16 / 2) so that a box row is 128 bytes in both.
int prepare_search(KnnLaunch& L, const void* store, const float* store_rnorm, int64_t n, const void* queries,
                   const float* query_rnorm, int q, int d, int k, int64_t index_base, int64_t query_index_base,
                   bool no_self, int sms, cudaStream_t stream,
                   CUtensorMapDataType dtype = CU_TENSOR_MAP_DATA_TYPE_BFLOAT16) {
  L.ncta = (sms >= 2) ? knn_ncta(q) : 1;
  L.plan = plan_knn(n, q, sms, L.ncta);
  int rc = encode_tmap_2d(&L.tq, dtype, 2, queries, static_cast<uint64_t>(q),
                          static_cast<uint64_t>(d), static_cast<uint64_t>(d) * 2, BM, BK, CU_TENSOR_MAP_SWIZZLE_128B);
  if (rc != ISX_OK) return rc;
  rc = encode_tmap_2d(&L.te, dtype, 2, store, static_cast<uint64_t>(n),
                      static_cast<uint64_t>(d), static_cast<uint64_t>(d) * 2, BN / L.ncta, BK, CU_TENSOR_MAP_SWIZZLE_128B);
  if (rc != ISX_OK) return rc;
  KnnParams& p = L.p;
  p = {};
  p.q = q; p.d = d; p.k = k; p.n = n;
  p.mb = L.plan.mb; p.splits = L.plan.splits; p.nb = L.plan.nb; p.items = L.plan.items;
  p.index_base = static_cast<int>(index_base);
  p.self_base = no_self ? static_cast<int>(query_index_base) : -1;
  p.store_rnorm = store_rnorm;
  p.query_rnorm = query_rnorm;
  set_throttle(p, 2 * d);
#ifdef ISX_KNN_PROFILE
  rc = set_profile(p, stream);
  if (rc != ISX_OK) return rc;
#else
  (void)stream;
#endif
  return ISX_OK;
}

// The one choice of kernel variant (CAP, NCTA, RES).  Plain, grouped and range search pick the same
// variant for the same (q, d, k <= kSmallK): same MMA shapes, same scaling, so their scores are bit
// for bit equal.  F8 (the E4M3 scan, p.d in 16-bit pairs) follows the same rules, and so does MAXSIM
// (run with p.k = kSmallK, like range search), whose maxima are therefore maxima of search()'s values.
template <bool GROUPED, bool RANGE, bool F8 = false, bool MAXSIM = false>
int launch_variant(const KnnLaunch& L, cudaStream_t stream) {
  static_assert(!MAXSIM || (!GROUPED && !RANGE && !F8), "maxsim excludes the grouped, range and fp8 modes");
  const KnnParams& p = L.p;
  const int grid = L.plan.grid;
  if constexpr (!RANGE && !MAXSIM) {
    if (p.k > kSmallK)
      return L.ncta == 2 ? launch_search<256, 2, false, GROUPED, false, F8>(L.tq, L.te, p, grid, stream)
                         : launch_search<256, 1, false, GROUPED, false, F8>(L.tq, L.te, p, grid, stream);
  }
  if (L.ncta == 1) return launch_search<32, 1, false, GROUPED, RANGE, F8, MAXSIM>(L.tq, L.te, p, grid, stream);
  // short rows (at most 512 bytes: the resident tile's 4 k-blocks), small k: the query tile stays resident
  if (p.d <= 256) return launch_search<32, 2, true, GROUPED, RANGE, F8, MAXSIM>(L.tq, L.te, p, grid, stream);
  return launch_search<32, 2, false, GROUPED, RANGE, F8, MAXSIM>(L.tq, L.te, p, grid, stream);
}

}  // namespace
}  // namespace isx

using namespace isx;

extern "C" {

int isx_row_rnorm_bf16(const void* x, int64_t n, int d, float eps, float* rnorm, isx_stream_t stream_) {
  const char* fn = "isx_row_rnorm_bf16";
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  ISX_REQUIRE(n >= 0 && d > 0, "%s: need n >= 0 and d > 0 (n=%lld d=%d)", fn, (long long)n, d);
  if (n == 0) return ISX_OK;
  ISX_REQUIRE(x && rnorm, "%s: null pointer", fn);
  int sms = 148;
  int rc = device_sm_count(&sms);
  if (rc != ISX_OK) return rc;
  const long long want = (n + 7) / 8;
  const int blocks = static_cast<int>(std::max<long long>(1, std::min<long long>(want, static_cast<long long>(sms) * 16)));
  row_rnorm_kernel<<<blocks, 256, 0, stream>>>(static_cast<const __nv_bfloat16*>(x), n, d, eps, rnorm);
  ISX_CHECK_CUDA(cudaGetLastError());
  return ISX_OK;
}

int isx_maps_to_rows_bf16(const float* maps, int64_t n, int C, int hw, int pool, void* rows, isx_stream_t stream_) {
  const char* fn = "isx_maps_to_rows_bf16";
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  ISX_REQUIRE(n >= 0 && C > 0 && hw > 0, "%s: need n >= 0, C > 0, hw > 0 (n=%lld C=%d hw=%d)", fn, (long long)n, C, hw);
  ISX_REQUIRE(pool == 0 || pool == 1, "%s: pool must be 0 or 1 (got %d)", fn, pool);
  if (n == 0) return ISX_OK;
  ISX_REQUIRE(maps && rows, "%s: null pointer", fn);
  int sms = 148;
  int rc = device_sm_count(&sms);
  if (rc != ISX_OK) return rc;
  if (pool) {
    const long long want = (n * C + 7) / 8;
    const int blocks = static_cast<int>(std::max<long long>(1, std::min<long long>(want, static_cast<long long>(sms) * 16)));
    maps_pool_rows_kernel<<<blocks, 256, 0, stream>>>(maps, n, C, hw, static_cast<__nv_bfloat16*>(rows));
  } else {
    const long long tiles = static_cast<long long>((C + 31) / 32) * ((hw + 31) / 32) * n;
    const int blocks = static_cast<int>(std::max<long long>(1, std::min<long long>(tiles, static_cast<long long>(sms) * 16)));
    maps_to_rows_kernel<<<blocks, 256, 0, stream>>>(maps, n, C, hw, static_cast<__nv_bfloat16*>(rows));
  }
  ISX_CHECK_CUDA(cudaGetLastError());
  return ISX_OK;
}

size_t isx_knn_workspace_bytes(int64_t n, int q, int d, int k) {
  (void)d;
  if (n <= 0 || q <= 0 || k <= 0 || k > kMaxK) return 0;
  int sms = 148;
  if (device_sm_count(&sms) != ISX_OK) sms = 148;
  return knn_workspace(sms, q, k).total;
}

static int knn_search_impl(const char* fn, const void* store, const float* store_rnorm, int64_t n, const void* queries,
                           const float* query_rnorm, int q, int d, int k, int64_t index_base,
                           int64_t query_index_base, int flags, float* out_scores, int32_t* out_idx,
                           void* workspace, size_t workspace_bytes, isx_stream_t stream_, const PeerOut* peers,
                           const int32_t* row_group = nullptr, int32_t* out_groups = nullptr, bool f8 = false) {
  // row_group != nullptr: grouped search (isx_knn_search_grouped), flags 0, outputs (scores, rows, groups)
  // f8: store and queries are E4M3 rows of d bytes (isx_knn_search_fp8)
  const bool grouped = row_group != nullptr || out_groups != nullptr;
  const bool cont = (flags & ISX_KNN_CONTINUE) != 0, finalize = (flags & ISX_KNN_NO_FINALIZE) == 0;
  const bool packed = (flags & ISX_KNN_PACKED) != 0, no_self = (flags & ISX_KNN_EXCLUDE_SELF) != 0;
  ISX_REQUIRE((flags & ~(ISX_KNN_CONTINUE | ISX_KNN_NO_FINALIZE | ISX_KNN_EXCLUDE_SELF | ISX_KNN_PACKED)) == 0,
              "%s: unknown flag bits 0x%x", fn, flags);
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  ISX_REQUIRE(q > 0 && d > 0 && k > 0 && n >= 0, "%s: need q, d, k > 0 and n >= 0 (q=%d d=%d k=%d n=%lld)", fn, q, d, k, (long long)n);
  ISX_REQUIRE(k <= kMaxK, "%s: k = %d exceeds the supported maximum of %d", fn, k, kMaxK);
  int rc = check_search_args(fn, store, n, queries, q, d, index_base, query_index_base, no_self);
  if (rc != ISX_OK) return rc;
  ISX_REQUIRE(queries && query_rnorm, "%s: null pointer", fn);
  ISX_REQUIRE(!finalize || peers || (out_scores && (packed || out_idx)), "%s: null output pointer", fn);
  ISX_REQUIRE(!grouped || (out_groups && flags == 0 && !peers), "%s: null output pointer", fn);
  ISX_REQUIRE(!grouped || n == 0 || row_group, "%s: null row_group pointer", fn);
  int sms = 148;
  rc = device_sm_count(&sms);
  if (rc != ISX_OK) return rc;
  const KnnWorkspace ws = knn_workspace(sms, q, k);
  ISX_REQUIRE(workspace != nullptr && workspace_bytes >= ws.total, "%s: workspace too small (%zu < %zu)", fn,
              workspace_bytes, ws.total);
  uint8_t* wbase = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(workspace) + 255) & ~uintptr_t(255));
  float* run_scores = reinterpret_cast<float*>(wbase + ws.run_scores_off);
  int32_t* run_idx = reinterpret_cast<int32_t*>(wbase + ws.run_idx_off);
  uint32_t* zero_base = reinterpret_cast<uint32_t*>(wbase + ws.zero_off);
  if (!cont) {
    // a new search: empty running lists, no bounds, no locks
    ISX_CHECK_CUDA(cudaMemsetAsync(zero_base, 0, ws.zero_bytes, stream));
    ISX_CHECK_CUDA(cudaMemsetAsync(run_idx, 0xFF, static_cast<size_t>(q) * k * sizeof(int32_t), stream));
  }
  if (n == 0) {
    // nothing to search in this block: the lists stay as they are
    if (!finalize) return ISX_OK;
    if (grouped)
      return launch_merge_grouped(nullptr, run_scores, run_idx, row_group, static_cast<int>(index_base), 1, q, k,
                                  query_rnorm, out_scores, out_idx, out_groups, stream);
    return launch_merge(run_scores, run_idx, 1, q, k, query_rnorm, out_scores, packed ? nullptr : out_idx, stream, peers);
  }
  ISX_REQUIRE(store && store_rnorm, "%s: null store pointer", fn);
  KnnLaunch L;
  // the fp8 scan moves its E4M3 rows (d bytes) as d / 2 16-bit pairs
  rc = prepare_search(L, store, store_rnorm, n, queries, query_rnorm, q, f8 ? d / 2 : d, k, index_base, query_index_base,
                      no_self, sms, stream, f8 ? CU_TENSOR_MAP_DATA_TYPE_UINT16 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16);
  if (rc != ISX_OK) return rc;
  KnnParams& p = L.p;
  p.run_scores = run_scores;
  p.run_idx = run_idx;
  p.cand_global = reinterpret_cast<uint2*>(wbase + ws.cand_off);
  p.thr_shared = zero_base;
  p.progress = p.thr_shared + q;
  p.run_lock = p.progress + 256;
  p.row_group = row_group;
  // a continued search keeps the lists and the bounds they imply; only the lockstep counters restart
  if (cont) ISX_CHECK_CUDA(cudaMemsetAsync(p.progress, 0, 256 * sizeof(uint32_t), stream));
  rc = grouped ? launch_variant<true, false>(L, stream)
               : f8 ? launch_variant<false, false, true>(L, stream) : launch_variant<false, false>(L, stream);
  if (rc != ISX_OK) return rc;
#ifdef ISX_KNN_PROFILE
  {
    const KnnPlan& plan = L.plan;
    const int ncta = L.ncta;
    unsigned long long h[24];
    ISX_CHECK_CUDA(cudaStreamSynchronize(stream));
    ISX_CHECK_CUDA(cudaMemcpy(h, p.prof, sizeof(h), cudaMemcpyDeviceToHost));
    const double units = static_cast<double>(plan.grid / ncta);
    const double tiles = static_cast<double>(plan.nb) * plan.mb / units;  // per unit
    fprintf(stderr,
            "isx knn profile (cycles per tile per unit; %d units, %.0f tiles each, splits %d): kernel %.0f | producer: "
            "wait-empty %.0f throttle %.0f | mma: wait-tmem-empty %.0f wait-full %.0f | epilogue warp 4: bar %.0f "
            "wait-tmem-full %.0f select %.0f item-final %.0f\n",
            plan.grid / ncta, tiles, plan.splits, h[7] / units / tiles, h[0] / units / tiles, h[1] / units / tiles,
            h[2] / units / tiles, h[3] / units / tiles, h[5] / units / tiles, h[4] / units / tiles, h[6] / units / tiles,
            h[8] / units / tiles);
    fprintf(stderr,
            "isx knn profile (warp 4 of every leader CTA, per tile): chunks %.2f, with survivors %.3f, appends %.3f, "
            "prunes %.3f (in %.3f calls, %.0f cycles), cycles in the rare path %.0f (group walks %.0f; windowed events %.4f; rows with survivors %.3f), in the item-end lock/merge phases %.0f; per item: rows merged %.1f, lock rounds %.1f\n",
            h[9] / units / tiles, h[10] / units / tiles, h[11] / units / tiles, h[12] / units / tiles, h[17] / units / tiles,
            h[16] / units / tiles, h[13] / units / tiles, h[21] / units / tiles, h[19] / units / tiles, h[20] / units / tiles, h[18] / units / tiles,
            h[14] / units / (static_cast<double>(plan.items) / units), h[15] / units / (static_cast<double>(plan.items) / units));
  }
#endif
  if (!finalize) return ISX_OK;
  if (grouped)
    return launch_merge_grouped(nullptr, p.run_scores, p.run_idx, row_group, p.index_base, 1, q, k, query_rnorm,
                                out_scores, out_idx, out_groups, stream);
  // finalize: scale the running lists by the queries' inverse norms, order by the final
  // (score desc, row asc); packed: one 8-byte record per hit (what a single all-gather moves)
  return launch_merge(p.run_scores, p.run_idx, 1, q, k, query_rnorm, out_scores, packed ? nullptr : out_idx, stream, peers);
}

int isx_knn_search_ex(const void* store, const float* store_rnorm, int64_t n, const void* queries,
                      const float* query_rnorm, int q, int d, int k, int64_t index_base,
                      int64_t query_index_base, int flags, float* out_scores, int32_t* out_idx,
                      void* workspace, size_t workspace_bytes, isx_stream_t stream) {
  return knn_search_impl("isx_knn_search_ex", store, store_rnorm, n, queries, query_rnorm, q, d, k, index_base,
                         query_index_base, flags, out_scores, out_idx, workspace, workspace_bytes, stream, nullptr);
}

int isx_knn_search_scatter(const void* store, const float* store_rnorm, int64_t n, const void* queries,
                           const float* query_rnorm, int q, int d, int k, int64_t index_base,
                           int64_t query_index_base, int flags, void* const* peer_bufs, int n_peers, int slot,
                           void* workspace, size_t workspace_bytes, isx_stream_t stream) {
  const char* fn = "isx_knn_search_scatter";
  ISX_REQUIRE(peer_bufs != nullptr && n_peers >= 1 && n_peers <= kMaxPeers, "%s: need 1..%d peer buffers (got %d)", fn,
              kMaxPeers, n_peers);
  ISX_REQUIRE(slot >= 0 && slot < n_peers, "%s: slot %d outside [0, %d)", fn, slot, n_peers);
  ISX_REQUIRE((flags & (ISX_KNN_NO_FINALIZE | ISX_KNN_PACKED)) == 0, "%s: the scatter is the finalising pass (flags 0x%x)", fn, flags);
  PeerOut peers;
  peers.n = n_peers;
  peers.slot_off = static_cast<long long>(slot) * q * k;
  for (int i = 0; i < n_peers; ++i) {
    ISX_REQUIRE(peer_bufs[i] != nullptr && (reinterpret_cast<uintptr_t>(peer_bufs[i]) & 7u) == 0,
                "%s: peer buffer %d is null or not 8-byte aligned", fn, i);
    peers.ptr[i] = static_cast<uint2*>(peer_bufs[i]);
  }
  return knn_search_impl(fn, store, store_rnorm, n, queries, query_rnorm, q, d, k, index_base, query_index_base, flags,
                         nullptr, nullptr, workspace, workspace_bytes, stream, &peers);
}

int isx_knn_search(const void* store, const float* store_rnorm, int64_t n, const void* queries,
                   const float* query_rnorm, int q, int d, int k, int64_t index_base,
                   float* out_scores, int32_t* out_idx, void* workspace, size_t workspace_bytes,
                   isx_stream_t stream) {
  return isx_knn_search_ex(store, store_rnorm, n, queries, query_rnorm, q, d, k, index_base, 0, 0, out_scores,
                           out_idx, workspace, workspace_bytes, stream);
}

int isx_quantize_rows_e4m3(const void* x, int64_t n, int d, int d16, void* out, float* rnorm, isx_stream_t stream_) {
  const char* fn = "isx_quantize_rows_e4m3";
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  ISX_REQUIRE(n >= 0 && d > 0, "%s: need n >= 0 and d > 0 (n=%lld d=%d)", fn, (long long)n, d);
  ISX_REQUIRE(d16 >= d && d16 % 16 == 0, "%s: d16 = %d must be a multiple of 16 and >= d = %d", fn, d16, d);
  if (n == 0) return ISX_OK;
  ISX_REQUIRE(x && out && rnorm, "%s: null pointer", fn);
  ISX_REQUIRE((reinterpret_cast<uintptr_t>(out) & 15u) == 0, "%s: out must be 16-byte aligned", fn);
  int sms = 148;
  int rc = device_sm_count(&sms);
  if (rc != ISX_OK) return rc;
  const long long want = (n + 7) / 8;
  const int blocks = static_cast<int>(std::max<long long>(1, std::min<long long>(want, static_cast<long long>(sms) * 16)));
  quantize_e4m3_kernel<<<blocks, 256, 0, stream>>>(static_cast<const __nv_bfloat16*>(x), n, d, d16,
                                                   static_cast<uint8_t*>(out), rnorm);
  ISX_CHECK_CUDA(cudaGetLastError());
  return ISX_OK;
}

int isx_knn_search_fp8(const void* store8, const float* rnorm8, int64_t n, const void* queries8, const float* qrnorm8,
                       int q, int d16, int k, int64_t index_base, float* out_scores, int32_t* out_idx, void* workspace,
                       size_t workspace_bytes, isx_stream_t stream) {
  const char* fn = "isx_knn_search_fp8";
  ISX_REQUIRE(d16 > 0 && d16 % 16 == 0, "%s: d16 = %d must be a positive multiple of 16 (16-byte rows for TMA)", fn, d16);
  return knn_search_impl(fn, store8, rnorm8, n, queries8, qrnorm8, q, d16, k, index_base, 0, 0, out_scores, out_idx,
                         workspace, workspace_bytes, stream, nullptr, nullptr, nullptr, true);
}

int isx_knn_rescore(const void* store, const float* rnorm, int64_t n, const void* queries, const float* qrnorm, int q,
                    int d, const int32_t* cand, int kc, int64_t index_base, int k, float* out_scores, int32_t* out_idx,
                    isx_stream_t stream_) {
  const char* fn = "isx_knn_rescore";
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  ISX_REQUIRE(q >= 0 && d > 0 && n >= 0, "%s: need q >= 0, d > 0 and n >= 0 (q=%d d=%d n=%lld)", fn, q, d, (long long)n);
  ISX_REQUIRE(kc >= 1 && kc <= kMaxK && k >= 1 && k <= kMaxK, "%s: need 1 <= kc, k <= %d (kc=%d k=%d)", fn, kMaxK, kc, k);
  int rc = check_search_args(fn, store, n, queries, q, d, index_base, 0, false);
  if (rc != ISX_OK) return rc;
  if (q == 0) return ISX_OK;
  ISX_REQUIRE(queries && qrnorm && cand && out_scores && out_idx && (n == 0 || (store && rnorm)), "%s: null pointer", fn);
  const int blocks = (q + 3) / 4;
  const int base = static_cast<int>(index_base);
  if (kc <= 32)
    rescore_kernel<1><<<blocks, 128, 0, stream>>>(static_cast<const __nv_bfloat16*>(store), rnorm, n,
                                                  static_cast<const __nv_bfloat16*>(queries), qrnorm, q, d, cand, kc, base,
                                                  k, out_scores, out_idx);
  else if (kc <= 64)
    rescore_kernel<2><<<blocks, 128, 0, stream>>>(static_cast<const __nv_bfloat16*>(store), rnorm, n,
                                                  static_cast<const __nv_bfloat16*>(queries), qrnorm, q, d, cand, kc, base,
                                                  k, out_scores, out_idx);
  else
    rescore_kernel<4><<<blocks, 128, 0, stream>>>(static_cast<const __nv_bfloat16*>(store), rnorm, n,
                                                  static_cast<const __nv_bfloat16*>(queries), qrnorm, q, d, cand, kc, base,
                                                  k, out_scores, out_idx);
  ISX_CHECK_CUDA(cudaGetLastError());
  return ISX_OK;
}

int isx_topk_merge(const float* scores, const int32_t* idx, int g, int q, int k, float* out_scores,
                   int32_t* out_idx, isx_stream_t stream_) {
  const char* fn = "isx_topk_merge";
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  ISX_REQUIRE(g >= 0 && q > 0 && k > 0, "%s: need g >= 0, q > 0, k > 0 (g=%d q=%d k=%d)", fn, g, q, k);
  ISX_REQUIRE(k <= kMaxK, "%s: k = %d exceeds the supported maximum of %d", fn, k, kMaxK);
  ISX_REQUIRE(out_scores && out_idx && (g == 0 || (scores && idx)), "%s: null pointer", fn);
  return launch_merge(scores, idx, g, q, k, nullptr, out_scores, out_idx, stream);
}

int isx_knn_search_grouped(const void* store, const float* store_rnorm, const int32_t* row_group, int64_t n,
                           const void* queries, const float* query_rnorm, int q, int d, int k, int64_t index_base,
                           float* out_scores, int32_t* out_rows, int32_t* out_groups, void* workspace,
                           size_t workspace_bytes, isx_stream_t stream) {
  return knn_search_impl("isx_knn_search_grouped", store, store_rnorm, n, queries, query_rnorm, q, d, k, index_base, 0,
                         0, out_scores, out_rows, workspace, workspace_bytes, stream, nullptr, row_group, out_groups);
}

int isx_topk_merge_grouped(const int32_t* records, int g, int q, int k, float* out_scores, int32_t* out_rows,
                           int32_t* out_groups, isx_stream_t stream_) {
  const char* fn = "isx_topk_merge_grouped";
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  ISX_REQUIRE(g >= 0 && q > 0 && k > 0, "%s: need g >= 0, q > 0, k > 0 (g=%d q=%d k=%d)", fn, g, q, k);
  ISX_REQUIRE(k <= kMaxK, "%s: k = %d exceeds the supported maximum of %d", fn, k, kMaxK);
  ISX_REQUIRE(out_scores && out_rows && out_groups && (g == 0 || records), "%s: null pointer", fn);
  ISX_REQUIRE((reinterpret_cast<uintptr_t>(records) & 3u) == 0, "%s: records must be 4-byte aligned", fn);
  return launch_merge_grouped(g ? records : nullptr, nullptr, nullptr, nullptr, 0, g, q, k, nullptr, out_scores,
                              out_rows, out_groups, stream);
}

int isx_topk_merge_packed(const void* records, int g, int q, int k, float* out_scores, int32_t* out_idx,
                          isx_stream_t stream_) {
  const char* fn = "isx_topk_merge_packed";
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  ISX_REQUIRE(g >= 0 && q > 0 && k > 0, "%s: need g >= 0, q > 0, k > 0 (g=%d q=%d k=%d)", fn, g, q, k);
  ISX_REQUIRE(k <= kMaxK, "%s: k = %d exceeds the supported maximum of %d", fn, k, kMaxK);
  ISX_REQUIRE(out_scores && out_idx && (g == 0 || records), "%s: null pointer", fn);
  ISX_REQUIRE((reinterpret_cast<uintptr_t>(records) & 7u) == 0, "%s: records must be 8-byte aligned", fn);
  if (g == 0) return launch_merge(out_scores, out_idx, 0, q, k, nullptr, out_scores, out_idx, stream);
  return launch_merge(static_cast<const float*>(records), nullptr, g, q, k, nullptr, out_scores, out_idx, stream);
}

int isx_knn_range(const void* store, const float* store_rnorm, int64_t n, const void* queries,
                  const float* query_rnorm, int q, int d, float threshold, int64_t index_base,
                  int64_t query_index_base, int flags, int32_t* records, int64_t capacity,
                  unsigned long long* count, void* workspace, size_t workspace_bytes, isx_stream_t stream_) {
  const char* fn = "isx_knn_range";
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  const bool cont = (flags & ISX_KNN_CONTINUE) != 0, no_self = (flags & ISX_KNN_EXCLUDE_SELF) != 0;
  ISX_REQUIRE((flags & ~(ISX_KNN_CONTINUE | ISX_KNN_EXCLUDE_SELF)) == 0, "%s: unknown flag bits 0x%x", fn, flags);
  ISX_REQUIRE(std::isfinite(threshold), "%s: the threshold must be finite (got %g)", fn, static_cast<double>(threshold));
  ISX_REQUIRE(q > 0 && d > 0 && n >= 0, "%s: need q, d > 0 and n >= 0 (q=%d d=%d n=%lld)", fn, q, d, (long long)n);
  int rc = check_search_args(fn, store, n, queries, q, d, index_base, query_index_base, no_self);
  if (rc != ISX_OK) return rc;
  ISX_REQUIRE(capacity >= 0 && capacity < (1ll << 60), "%s: capacity out of range (%lld)", fn, (long long)capacity);
  ISX_REQUIRE(queries && query_rnorm && count && (capacity == 0 || records), "%s: null pointer", fn);
  ISX_REQUIRE((reinterpret_cast<uintptr_t>(records) & 3u) == 0 && (reinterpret_cast<uintptr_t>(count) & 7u) == 0,
              "%s: records must be 4-byte and count 8-byte aligned", fn);
  ISX_REQUIRE(workspace != nullptr && workspace_bytes >= ISX_KNN_RANGE_WORKSPACE_BYTES,
              "%s: workspace too small (%zu < %d)", fn, workspace_bytes, ISX_KNN_RANGE_WORKSPACE_BYTES);
  if (!cont) ISX_CHECK_CUDA(cudaMemsetAsync(count, 0, sizeof(unsigned long long), stream));
  if (n == 0) return ISX_OK;
  ISX_REQUIRE(store && store_rnorm, "%s: null store pointer", fn);
  int sms = 148;
  rc = device_sm_count(&sms);
  if (rc != ISX_OK) return rc;
  KnnLaunch L;
  rc = prepare_search(L, store, store_rnorm, n, queries, query_rnorm, q, d, kSmallK, index_base, query_index_base,
                      no_self, sms, stream);
  if (rc != ISX_OK) return rc;
  KnnParams& p = L.p;
  p.progress = reinterpret_cast<uint32_t*>((reinterpret_cast<uintptr_t>(workspace) + 255) & ~uintptr_t(255));
  p.range_tau = threshold;
  p.range_rec = records;
  p.range_cap = capacity;
  p.range_count = count;
  ISX_CHECK_CUDA(cudaMemsetAsync(p.progress, 0, 256 * sizeof(uint32_t), stream));
  return launch_variant<false, true>(L, stream);
}

int isx_knn_maxsim(const void* store, const float* store_rnorm, const int32_t* row_group, int64_t n, const void* queries,
                   const float* query_rnorm, int q, int d, int64_t group_base, int64_t num_groups, float* cell_max,
                   void* workspace, size_t workspace_bytes, isx_stream_t stream_) {
  const char* fn = "isx_knn_maxsim";
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  ISX_REQUIRE(q > 0 && d > 0 && n >= 0, "%s: need q, d > 0 and n >= 0 (q=%d d=%d n=%lld)", fn, q, d, (long long)n);
  ISX_REQUIRE(num_groups >= 1 && group_base >= 0 && group_base + num_groups <= (1ll << 31),
              "%s: need num_groups >= 1 and 0 <= group_base, group_base + num_groups <= 2^31 (got %lld, %lld)", fn,
              (long long)group_base, (long long)num_groups);
  int rc = check_search_args(fn, store, n, queries, q, d, 0, 0, false);
  if (rc != ISX_OK) return rc;
  ISX_REQUIRE(queries && query_rnorm && cell_max, "%s: null pointer", fn);
  ISX_REQUIRE((reinterpret_cast<uintptr_t>(cell_max) & 3u) == 0, "%s: cell_max must be 4-byte aligned", fn);
  ISX_REQUIRE(workspace != nullptr && workspace_bytes >= ISX_KNN_RANGE_WORKSPACE_BYTES,
              "%s: workspace too small (%zu < %d)", fn, workspace_bytes, ISX_KNN_RANGE_WORKSPACE_BYTES);
  int sms = 148;
  rc = device_sm_count(&sms);
  if (rc != ISX_OK) return rc;
  const long long cells = static_cast<long long>(q) * num_groups;
  const int fill_blocks = static_cast<int>(std::max<long long>(1, std::min<long long>((cells + 255) / 256, static_cast<long long>(sms) * 16)));
  fill_f32_kernel<<<fill_blocks, 256, 0, stream>>>(cell_max, cells, -INFINITY);
  ISX_CHECK_CUDA(cudaGetLastError());
  if (n == 0) return ISX_OK;
  ISX_REQUIRE(store && store_rnorm && row_group, "%s: null store pointer", fn);
  KnnLaunch L;
  rc = prepare_search(L, store, store_rnorm, n, queries, query_rnorm, q, d, kSmallK, 0, 0, false, sms, stream);
  if (rc != ISX_OK) return rc;
  KnnParams& p = L.p;
  p.progress = reinterpret_cast<uint32_t*>((reinterpret_cast<uintptr_t>(workspace) + 255) & ~uintptr_t(255));
  p.row_group = row_group;
  p.cell_max = cell_max;
  p.group_base = static_cast<int>(group_base);
  p.num_groups = static_cast<int>(std::min<int64_t>(num_groups, INT_MAX));
  ISX_CHECK_CUDA(cudaMemsetAsync(p.progress, 0, 256 * sizeof(uint32_t), stream));
  return launch_variant<false, false, false, true>(L, stream);
}

int isx_maxsim_sets_topk(const float* cell_max, const float* query_rnorm, int q, int64_t num_groups, int64_t col_begin,
                         int64_t col_end, const int64_t* set_offsets, int num_sets, int k, int64_t group_base,
                         void* records, isx_stream_t stream_) {
  const char* fn = "isx_maxsim_sets_topk";
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  ISX_REQUIRE(q >= 0 && num_sets >= 0 && num_groups >= 1, "%s: need q, num_sets >= 0 and num_groups >= 1", fn);
  ISX_REQUIRE(k >= 1 && k <= kMaxK, "%s: need 1 <= k <= %d (k=%d)", fn, kMaxK, k);
  ISX_REQUIRE(0 <= col_begin && col_begin <= col_end && col_end <= num_groups,
              "%s: need 0 <= col_begin <= col_end <= num_groups (got %lld, %lld, %lld)", fn, (long long)col_begin,
              (long long)col_end, (long long)num_groups);
  ISX_REQUIRE(group_base >= 0 && group_base + num_groups <= (1ll << 31), "%s: group ids must fit in int32", fn);
  if (num_sets == 0) return ISX_OK;
  ISX_REQUIRE(set_offsets && records && (q == 0 || (cell_max && query_rnorm)), "%s: null pointer", fn);
  ISX_REQUIRE((reinterpret_cast<uintptr_t>(records) & 7u) == 0, "%s: records must be 8-byte aligned", fn);
  maxsim_sets_topk_kernel<<<num_sets, kSetThreads, 0, stream>>>(cell_max, query_rnorm, q, num_groups,
                                                                static_cast<int>(col_begin), static_cast<int>(col_end),
                                                                set_offsets, k, static_cast<int>(group_base),
                                                                static_cast<uint2*>(records));
  ISX_CHECK_CUDA(cudaGetLastError());
  return ISX_OK;
}

}  // extern "C"
