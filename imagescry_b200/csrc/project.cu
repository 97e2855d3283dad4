// Stage 2 of the sift path: L2-normalise (+ spatial mean pool) + PCA projection, fused.
//
// Replaces, behind the C ABI in include/imagescry_b200.h,
//   /root/reference/src/imagescry/models/embedding.py:74       F.normalize(x, p=2, dim=1)
//   /root/reference/src/imagescry/data.py:112-118              EmbeddingBatch.get_flat_vectors
//   /root/reference/src/imagescry/models/decomposition.py:79-91 PCA.forward: (x - mean) @ components
//   /root/reference/src/imagescry/models/pipelines.py:82-84    reshape(B,h,w,k).permute(0,3,1,2)
//
// K3  l2norm_project_kernel (per-cell mode): the fp32 B x E x h x w feature map is read ONCE.
//   out[cell, :] = rnorm[cell] * (x[cell, :] . W) + bias,   bias = -(mean . W),
//   rnorm[cell] = 1 / max(||x[cell, :]||, 1e-12)
// which equals (x/||x|| - mean) . W.  The contraction runs on tcgen05 tensor cores with fp32-class
// accuracy: x and W are split into bf16 hi + lo parts and three MMAs (hi.hi + lo.hi + hi.lo)
// accumulate into the same fp32 TMEM tile (error ~2^-16 relative per product, far inside the 1e-3
// tolerance; a single bf16 or tf32 pass is not).
//
//   warp 0       TMA producer for the packed weight tiles (W_hi, W_lo; bf16, K-major, 128B swizzle)
//   warp 1       MMA issuer (one elected lane)
//   warp 2       TMEM allocation
//   warps 4-7    epilogue: tcgen05.ld, scale by the cell's inverse norm, add bias, store rows of `out`
//   warps 8-15   transform: coalesced fp32 loads of the NCHW map (cells are the contiguous dim, so a
//                warp reads 128 contiguous bytes per channel), accumulate the per-cell sum of squares,
//                split to bf16 hi/lo and write K-major swizzled operand tiles for the MMA.
//
// K3p l2norm_pool_kernel (pool mode): one pass over the map with 16-cell slabs staged in shared
// memory by cp.async; per image the spatial mean of the normalised cells comes out as E floats,
// which then go through the same projection kernel as an n x F matrix (normalize = 0).
#include "common.cuh"

#include <cuda_fp16.h>

#include <algorithm>

namespace isx {
namespace {

constexpr int PM = 128;  // cells per tile (TMEM lanes)
constexpr int PK = 64;   // features per k-block
constexpr int P_UMMA_K = 16;
constexpr int kTransformWarp0 = 8;
// transform warps: 8 in the register-path kernels (32 features per thread and k-block), 16 in the
// staged kernel (16 features per thread: twice the warps hide the LDS / barrier / fence latencies)
constexpr int transform_warps(bool staged) { return staged ? 16 : 8; }
constexpr int proj_threads(bool staged) { return (kTransformWarp0 + transform_warps(staged)) * 32; }
constexpr int kMaxComponents = 256;

constexpr uint32_t A_PART_BYTES = PM * PK * 2;           // 16 KB (one of hi / lo)
constexpr uint32_t A_STAGE_BYTES_P = 2 * A_PART_BYTES;   // hi + lo
constexpr int P_ACC_STAGES = 2;

// The per-cell kernels run on CTA pairs (cta_group::2): each CTA transforms its own 128 cells but
// stages only half of the weight rows of every k-block, so the L2 -> shared-memory weight stream per
// SM halves and the freed shared memory buys a third stage for both rings of the register path.
// STAGED: the raw fp32 128-cell x 64-feature boxes of the map arrive by TMA into a three-deep ring
// (96 KB in flight per SM, no registers involved); the transform warps read them from shared
// memory.  The weight and converted-operand rings then have two stages each.
template <bool STAGED>
struct ProjSmem {
  static constexpr uint32_t W_PART_BYTES = (kMaxComponents / 2) * PK * 2;  // 16 KB per CTA of a pair
  static constexpr uint32_t W_STAGE_BYTES = 2 * W_PART_BYTES;              // hi + lo
  static constexpr int A_STAGES = STAGED ? 2 : 3;
  static constexpr int W_STAGES = STAGED ? 2 : 3;
  static constexpr int RAW_STAGES = STAGED ? 3 : 0;
  static constexpr uint32_t RAW_STAGE_BYTES = PM * PK * 4;                   // 32 KB
  static constexpr uint32_t kAOff = 0;
  static constexpr uint32_t kWOff = kAOff + A_STAGES * A_STAGE_BYTES_P;
  static constexpr uint32_t kRawOff = kWOff + W_STAGES * W_STAGE_BYTES;
  static constexpr uint32_t kSsOff = kRawOff + RAW_STAGES * RAW_STAGE_BYTES;
  static constexpr uint32_t kBarOff = kSsOff + P_ACC_STAGES * 2 * PM * 4;    // after ss[acc][half][row]
  static constexpr uint32_t kNumBars = 2 * A_STAGES + 2 * W_STAGES + 4 * P_ACC_STAGES + 2 * RAW_STAGES;
  static constexpr uint32_t kTmemPtrOff = kBarOff + kNumBars * 8;
  static constexpr uint32_t kTotal = kTmemPtrOff + 16;
  static constexpr uint32_t kMaxDynamic = 232448;
  static constexpr uint32_t kDynamicBytes = (kTotal + 1024 <= kMaxDynamic) ? kTotal + 1024 : kMaxDynamic;
  static_assert(kTotal <= kMaxDynamic, "shared-memory plan exceeds 227 KB");
};

struct PackedLayout {
  int k_pad, f_pad;
  size_t hi_off, lo_off, bias_off, h_off, total;  // h: the weights once more, as plain fp16 (single-pass mode)
};

PackedLayout packed_layout(int F, int k) {
  PackedLayout l;
  l.k_pad = (k + 15) / 16 * 16;
  l.f_pad = (F + PK - 1) / PK * PK;
  const size_t mat = static_cast<size_t>(l.k_pad) * l.f_pad * 2;
  l.hi_off = 0;
  l.lo_off = (mat + 255) / 256 * 256;
  l.bias_off = l.lo_off + (mat + 255) / 256 * 256;
  l.h_off = l.bias_off + (static_cast<size_t>(l.k_pad) * 4 + 255) / 256 * 256;
  l.total = l.h_off + (mat + 255) / 256 * 256;
  return l;
}

// One warp per component j: split every weight into bf16 hi + lo and accumulate the bias in fp64.
__global__ void __launch_bounds__(256)
pack_weights_kernel(const float* __restrict__ means, const float* __restrict__ comps, int F, int k,
                    long long ld_f, long long ld_k, int k_pad, int f_pad, __nv_bfloat16* __restrict__ w_hi,
                    __nv_bfloat16* __restrict__ w_lo, __half* __restrict__ w_h, float* __restrict__ bias) {
  const int lane = threadIdx.x & 31;
  const int j = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (j >= k_pad) return;
  double acc = 0.0;
  for (int f = lane; f < f_pad; f += 32) {
    float w = 0.f;
    if (j < k && f < F) {
      w = comps[f * ld_f + j * ld_k];
      acc += static_cast<double>(means[f]) * static_cast<double>(w);
    }
    const __nv_bfloat16 hi = __float2bfloat16_rn(w);
    const __nv_bfloat16 lo = __float2bfloat16_rn(w - __bfloat162float(hi));
    w_hi[static_cast<size_t>(j) * f_pad + f] = hi;
    w_lo[static_cast<size_t>(j) * f_pad + f] = lo;
    w_h[static_cast<size_t>(j) * f_pad + f] = __float2half_rn(w);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(kFullMask, acc, o);
  if (lane == 0) bias[j] = static_cast<float>(-acc);
}

struct ProjParams {
  const float* fmap;
  long long m_total;  // B * hw cells (rows)
  int E, hw, k, k_pad;
  int fast;           // staged kernel: one fp16 tensor pass (operands rounded to fp16, saturating) instead of
                      // the three-pass bf16 split; tmap_whi then describes the fp16 weight matrix
  int rowmajor;       // staged kernel: fmap is an n x E row-major matrix (hw == 1); tmap_x is a 2-D
                      // map with 128B-swizzled boxes of 128 rows x 32 features
  int normalize;
  long long tiles;
  const float* bias;
  float* out;
};

// STAGED: raw tiles of the map staged by TMA (tmap_x); otherwise the register path, which loads the
// map from global memory and takes any shape (tmap_x unused).
template <bool STAGED>
__global__ void __launch_bounds__(proj_threads(STAGED), 1)
l2norm_project_kernel(const __grid_constant__ CUtensorMap tmap_whi, const __grid_constant__ CUtensorMap tmap_wlo,
                      const __grid_constant__ CUtensorMap tmap_x, const ProjParams p) {
  using L = ProjSmem<STAGED>;
  constexpr int A_STAGES = L::A_STAGES, W_STAGES = L::W_STAGES, RAW_STAGES = L::RAW_STAGES;
  constexpr int TW = transform_warps(STAGED);
  constexpr uint32_t W_PART_BYTES = L::W_PART_BYTES, W_STAGE_BYTES = L::W_STAGE_BYTES;
  const uint32_t rank = cluster_ctarank();
  const long long unit = blockIdx.x / 2, num_units = gridDim.x / 2;
  extern __shared__ uint8_t smem_raw[];
  // align by offsetting the shared array itself (not through an integer round trip) so the compiler
  // keeps the shared address space and emits LDS/STS instead of generic loads and stores
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  if (threadIdx.x == 0 && static_cast<uint32_t>(smem - smem_raw) + L::kTotal > L::kDynamicBytes) {
    printf("isx: l2norm_project_kernel: dynamic shared memory window is not 1024-byte aligned\n");
    __trap();
  }
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + L::kBarOff);
  uint64_t* a_full = bars;                        // [A_STAGES]  8 transform warps per CTA (on the leader)
  uint64_t* a_empty = a_full + A_STAGES;          // [A_STAGES]  tcgen05.commit
  uint64_t* w_full = a_empty + A_STAGES;          // [W_STAGES]  TMA
  uint64_t* w_empty = w_full + W_STAGES;          // [W_STAGES]  tcgen05.commit
  uint64_t* tmem_full = w_empty + W_STAGES;       // [ACC]       tcgen05.commit
  uint64_t* tmem_empty = tmem_full + P_ACC_STAGES;  // [ACC]     4 epilogue warps
  uint64_t* ss_full = tmem_empty + P_ACC_STAGES;  // [ACC]       256 transform threads
  uint64_t* ss_empty = ss_full + P_ACC_STAGES;    // [ACC]       4 epilogue warps
  uint64_t* raw_full = ss_empty + P_ACC_STAGES;   // [RAW]       TMA (staged mode)
  uint64_t* raw_empty = raw_full + RAW_STAGES;    // [RAW]       8 transform warps
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(smem + L::kTmemPtrOff);
  float* ss_s = reinterpret_cast<float*>(smem + L::kSsOff);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int num_kb = (p.E + PK - 1) / PK;

  if (warp == 0 && lane == 0) {
    prefetch_tmap(&tmap_whi);
    prefetch_tmap(&tmap_wlo);
  }
  if (warp == 1 && lane == 0) {
    for (int i = 0; i < A_STAGES; ++i) { mbar_init(&a_full[i], TW * 2); mbar_init(&a_empty[i], 1); }
    for (int i = 0; i < W_STAGES; ++i) { mbar_init(&w_full[i], 2); mbar_init(&w_empty[i], 1); }
    for (int i = 0; i < P_ACC_STAGES; ++i) {
      mbar_init(&tmem_full[i], 1);
      mbar_init(&tmem_empty[i], 4 * 2);
      mbar_init(&ss_full[i], STAGED ? TW : TW * 32);
      mbar_init(&ss_empty[i], 4);
    }
    for (int i = 0; i < RAW_STAGES; ++i) { mbar_init(&raw_full[i], 1); mbar_init(&raw_empty[i], TW); }
    fence_mbar_init();
  }
  if (warp == 2) { tmem_alloc_pair(tmem_ptr, 512); tmem_relinquish_pair(); }
  tc_fence_before();
  cluster_sync_all();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;
  const int w_rows = p.k_pad / 2;  // weight rows (components) this CTA stages per k-block
  const uint32_t w_part_bytes = static_cast<uint32_t>(w_rows) * PK * 2;

  if (warp == 0) {
    // ===================== weight TMA producer =====================
    if (lane == 0) {
      uint32_t stage = 0, phase = 0;
      const int32_t row0 = static_cast<int32_t>(rank) * w_rows;
      for (long long tile = unit; tile < p.tiles; tile += num_units) {
        for (int kb = 0; kb < num_kb; ++kb) {
          mbar_wait(&w_empty[stage], phase ^ 1);
          uint8_t* dst = smem + L::kWOff + stage * W_STAGE_BYTES;
          if (STAGED && p.fast) {
            // single fp16 pass: one weight matrix (tmap_whi describes the fp16 copy)
            mbar_arrive_expect_tx_leader(&w_full[stage], w_part_bytes);
            tma_load_2d_pair(dst, &tmap_whi, &w_full[stage], kb * PK, row0, kEvictLast);
          } else {
            mbar_arrive_expect_tx_leader(&w_full[stage], 2 * w_part_bytes);
            tma_load_2d_pair(dst, &tmap_whi, &w_full[stage], kb * PK, row0, kEvictLast);
            tma_load_2d_pair(dst + W_PART_BYTES, &tmap_wlo, &w_full[stage], kb * PK, row0, kEvictLast);
          }
          if (++stage == W_STAGES) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    if (lane == 0 && rank == 0) {
      const uint32_t idesc = make_idesc(/*bf16*/ 1, PM * 2, static_cast<uint32_t>(p.k_pad));
      const uint32_t idesc_f16 = make_idesc(/*f16*/ 0, PM * 2, static_cast<uint32_t>(p.k_pad));
      (void)idesc_f16;
      uint32_t as = 0, aph = 0, ws = 0, wph = 0, acc = 0, acc_phase = 0;
      for (long long tile = unit; tile < p.tiles; tile += num_units) {
        mbar_wait(&tmem_empty[acc], acc_phase ^ 1);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + acc * kMaxComponents;
        for (int kb = 0; kb < num_kb; ++kb) {
          mbar_wait(&w_full[ws], wph);
          mbar_wait(&a_full[as], aph);
          tc_fence_after();
          const uint32_t a_hi = smem_u32(smem + L::kAOff + as * A_STAGE_BYTES_P);
          const uint32_t a_lo = a_hi + A_PART_BYTES;
          const uint32_t w_hi = smem_u32(smem + L::kWOff + ws * W_STAGE_BYTES);
          const uint32_t w_lo = w_hi + W_PART_BYTES;
#pragma unroll
          for (int k = 0; k < PK / P_UMMA_K; ++k) {
            const uint32_t o = k * P_UMMA_K * 2;
            const uint64_t dah = make_kmajor_sw128_desc(a_hi + o), dal = make_kmajor_sw128_desc(a_lo + o);
            const uint64_t dwh = make_kmajor_sw128_desc(w_hi + o), dwl = make_kmajor_sw128_desc(w_lo + o);
            if (STAGED && p.fast) {
              tc_mma_f16_pair(d_tmem, dah, dwh, idesc_f16, (kb | k) != 0);
            } else {
              tc_mma_f16_pair(d_tmem, dah, dwh, idesc, (kb | k) != 0);
              tc_mma_f16_pair(d_tmem, dal, dwh, idesc, 1);
              tc_mma_f16_pair(d_tmem, dah, dwl, idesc, 1);
            }
          }
          tc_commit_pair(&a_empty[as]);
          tc_commit_pair(&w_empty[ws]);
          if (++as == A_STAGES) { as = 0; aph ^= 1; }
          if (++ws == W_STAGES) { ws = 0; wph ^= 1; }
        }
        tc_commit_pair(&tmem_full[acc]);
        if (++acc == P_ACC_STAGES) { acc = 0; acc_phase ^= 1; }
      }
    }
  } else if (warp == 3) {
    if (STAGED) {
      // ===================== raw-tile TMA producer (staged kernel) =====================
      if (lane == 0) {
        uint32_t rs = 0, rph = 0;
        for (long long tile = unit; tile < p.tiles; tile += num_units) {
          const long long R0 = (tile * 2 + rank) * PM;
          const long long img = R0 / p.hw;
          const int cell = static_cast<int>(R0 - img * p.hw);
          for (int kb = 0; kb < num_kb; ++kb) {
            mbar_wait(&raw_empty[rs], rph ^ 1);
            mbar_arrive_expect_tx(&raw_full[rs], L::RAW_STAGE_BYTES);
            uint8_t* dst = smem + L::kRawOff + rs * L::RAW_STAGE_BYTES;
            if (p.rowmajor) {
              // two 128-row x 32-feature boxes (128-byte rows, 128B swizzle) per k-block
              tma_load_2d(dst, &tmap_x, &raw_full[rs], kb * PK, static_cast<int32_t>(R0), kEvictFirst);
              tma_load_2d(dst + L::RAW_STAGE_BYTES / 2, &tmap_x, &raw_full[rs], kb * PK + 32, static_cast<int32_t>(R0),
                          kEvictFirst);
            } else {
              tma_load_3d(dst, &tmap_x, &raw_full[rs], cell, kb * PK, static_cast<int32_t>(img), kEvictFirst);
            }
            if (++rs == static_cast<uint32_t>(RAW_STAGES)) { rs = 0; rph ^= 1; }
          }
        }
      }
    }
  } else if (warp >= kTransformWarp0) {
    // ===================== transform: fp32 NCHW -> bf16 hi/lo K-major tiles =====================
    const long long my_tiles = (p.tiles - unit + num_units - 1) / num_units;
    const long long total_seq = my_tiles * num_kb;
    if constexpr (STAGED) {
      // 16 warps.  Warp tw: rows 16 (tw % 8) .. +15; lanes 0-15 take feature quarter 2 (tw / 8),
      // lanes 16-31 the next quarter of the same rows (one shuffle then sums the two quarters'
      // sums of squares).  Raw box layout: [image][feature][cell], cb = min(hw, 128) cells per row.
      const int tw = warp - kTransformWarp0;
      const int m = (tw & 7) * 16 + (lane & 15);
      const int quarter = (tw >> 3) * 2 + (lane >> 4);
      const int cb = min(p.hw, PM);
      const int m_off = (m / cb) * (PK * cb) + (m % cb) + quarter * 16 * cb;
      float ss = 0.f;
      uint32_t acc = 0, acc_phase = 0, stage = 0, phase = 0, rs = 0, rph = 0;
      int pr_kb = 0;
      for (long long seq = 0; seq < total_seq; ++seq) {
        mbar_wait(&raw_full[rs], rph);
        float x[16];
        if (p.rowmajor) {
          // [2 sub-boxes][128 rows][32 features], 16-byte chunks XOR-swizzled by row % 8
          const uint8_t* rawb = smem + L::kRawOff + rs * L::RAW_STAGE_BYTES + (quarter >> 1) * (L::RAW_STAGE_BYTES / 2) + m * 128;
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            const int chunk = ((quarter & 1) * 4 + j) ^ (m & 7);
            const float4 v = *reinterpret_cast<const float4*>(rawb + chunk * 16);
            x[4 * j] = v.x; x[4 * j + 1] = v.y; x[4 * j + 2] = v.z; x[4 * j + 3] = v.w;
          }
        } else {
          const float* raw = reinterpret_cast<const float*>(smem + L::kRawOff + rs * L::RAW_STAGE_BYTES) + m_off;
#pragma unroll
          for (int i = 0; i < 16; ++i) x[i] = raw[i * cb];
        }
        // The next fill of this stage is a TMA write (async proxy) issued as soon as every warp has
        // arrived.  A bare arrive does not wait for the loads above to return (the compiler issues it
        // right behind them), so a late load could read the next fill: the proxy fence completes this
        // thread's reads of the stage before the warp releases it.
        fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0) mbar_arrive(&raw_empty[rs]);
        if (++rs == static_cast<uint32_t>(RAW_STAGES)) { rs = 0; rph ^= 1; }
        uint32_t hi[8], lo[8];
        if (p.fast) {
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            const float a = x[2 * i], b = x[2 * i + 1];
            ss = fmaf(a, a, ss);
            ss = fmaf(b, b, ss);
            // one fp16 operand (11-bit significand), saturating: lower half = a, upper half = b
            asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(hi[i]) : "f"(b), "f"(a));
            lo[i] = 0u;
          }
        } else {
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            const float a = x[2 * i], b = x[2 * i + 1];
            ss = fmaf(a, a, ss);
            ss = fmaf(b, b, ss);
            // hi = x truncated to bf16 (a mask); lo = RN_bf16(x - hi): |x - hi - lo| <= 2^-16 |x|
            const uint32_t ab = __float_as_uint(a), bb = __float_as_uint(b);
            hi[i] = __byte_perm(ab, bb, 0x7632);
            const float la = a - __uint_as_float(ab & 0xFFFF0000u);
            const float lb = b - __uint_as_float(bb & 0xFFFF0000u);
            const __nv_bfloat162 l2 = __floats2bfloat162_rn(la, lb);
            lo[i] = *reinterpret_cast<const uint32_t*>(&l2);
          }
        }
        mbar_wait(&a_empty[stage], phase ^ 1);
        uint8_t* a_hi = smem + L::kAOff + stage * A_STAGE_BYTES_P + m * 128;
        uint8_t* a_lo = a_hi + A_PART_BYTES;
#pragma unroll
        for (int c = 0; c < 2; ++c) {
          const int chunk = (quarter * 2 + c) ^ (m & 7);  // 128B swizzle: 16-byte chunk index XOR row % 8
          *reinterpret_cast<uint4*>(a_hi + chunk * 16) = make_uint4(hi[4 * c], hi[4 * c + 1], hi[4 * c + 2], hi[4 * c + 3]);
          if (!p.fast)
            *reinterpret_cast<uint4*>(a_lo + chunk * 16) = make_uint4(lo[4 * c], lo[4 * c + 1], lo[4 * c + 2], lo[4 * c + 3]);
        }
        fence_proxy_async_smem();  // generic-proxy writes -> visible to the tensor core's async proxy
        __syncwarp();
        if (lane == 0) mbar_arrive_leader(&a_full[stage]);
        if (++stage == static_cast<uint32_t>(A_STAGES)) { stage = 0; phase ^= 1; }
        if (++pr_kb == num_kb) {
          // last k-block of the tile: publish the row's sum of squares over this warp's two quarters
          pr_kb = 0;
          const float both = ss + __shfl_xor_sync(kFullMask, ss, 16);
          mbar_wait(&ss_empty[acc], acc_phase ^ 1);
          if (lane < 16) ss_s[(acc * 2 + (tw >> 3)) * PM + m] = both;
          __syncwarp();
          if (lane == 0) mbar_arrive(&ss_full[acc]);
          ss = 0.f;
          if (++acc == P_ACC_STAGES) { acc = 0; acc_phase ^= 1; }
        }
      }
    } else {
    const int t = threadIdx.x - kTransformWarp0 * 32;  // 0..255
    const int m = t & (PM - 1);                        // row (cell) inside the tile
    const int half = t >> 7;                           // which 32 of the k-block's 64 features

    // Two cursors walk the flattened (tile, k-block) sequence without any division: `ld` issues the
    // global loads one k-block ahead of `pr`, which converts and publishes the operand tiles.
    struct Cursor {
      long long tile_iter;
      int kb;
    };
    Cursor ld = {0, 0};
    const float* ld_base = nullptr;  // &fmap[img][0][cell] of this thread's row in ld's tile
    bool ld_valid = false;
    auto seek_tile = [&](long long tile_iter) {
      const long long tile = unit + tile_iter * num_units;
      const long long R = (tile * 2 + rank) * PM + m;
      ld_valid = tile_iter < my_tiles && R < p.m_total;
      const long long img = ld_valid ? R / p.hw : 0;  // once per tile
      const long long cell = ld_valid ? R - img * p.hw : 0;
      ld_base = p.fmap + img * p.E * static_cast<long long>(p.hw) + cell;
    };
    seek_tile(0);
    auto ld_f32 = [](const float* ptr) {
      float v;
      asm volatile("ld.global.nc.L1::no_allocate.f32 %0, [%1];" : "=f"(v) : "l"(ptr));
      return v;
    };
    auto load_block = [&](float (&x)[32]) {
      const int f0 = ld.kb * PK + half * 32;
      const float* src = ld_base + static_cast<long long>(f0) * p.hw;
#pragma unroll
      for (int i = 0; i < 32; ++i) {
        x[i] = (ld_valid && f0 + i < p.E) ? ld_f32(src) : 0.f;
        src += p.hw;
      }
      if (++ld.kb == num_kb) { ld.kb = 0; seek_tile(++ld.tile_iter); }
    };

    float ss = 0.f;
    uint32_t acc = 0, acc_phase = 0, stage = 0, phase = 0;
    int pr_kb = 0;
    auto process = [&](float (&x)[32]) {
      uint32_t hi[16], lo[16];
#pragma unroll
      for (int i = 0; i < 16; ++i) {
        const float a = x[2 * i], b = x[2 * i + 1];
        ss = fmaf(a, a, ss);
        ss = fmaf(b, b, ss);
        // hi = x truncated to bf16 (a mask, no conversion); lo = RN_bf16(x - hi), the subtraction is
        // exact.  |x - hi - lo| <= 2^-16 |x|.
        const uint32_t ab = __float_as_uint(a), bb = __float_as_uint(b);
        hi[i] = __byte_perm(ab, bb, 0x7632);
        const float la = a - __uint_as_float(ab & 0xFFFF0000u);
        const float lb = b - __uint_as_float(bb & 0xFFFF0000u);
        const __nv_bfloat162 l2 = __floats2bfloat162_rn(la, lb);
        lo[i] = *reinterpret_cast<const uint32_t*>(&l2);
      }
      mbar_wait(&a_empty[stage], phase ^ 1);
      uint8_t* a_hi = smem + L::kAOff + stage * A_STAGE_BYTES_P + m * 128;
      uint8_t* a_lo = a_hi + A_PART_BYTES;
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        const int chunk = (half * 4 + c) ^ (m & 7);  // 128B swizzle: 16-byte chunk index XOR row % 8
        *reinterpret_cast<uint4*>(a_hi + chunk * 16) = make_uint4(hi[4 * c], hi[4 * c + 1], hi[4 * c + 2], hi[4 * c + 3]);
        *reinterpret_cast<uint4*>(a_lo + chunk * 16) = make_uint4(lo[4 * c], lo[4 * c + 1], lo[4 * c + 2], lo[4 * c + 3]);
      }
      fence_proxy_async_smem();  // generic-proxy writes -> visible to the tensor core's async proxy
      __syncwarp();
      if (lane == 0) mbar_arrive_leader(&a_full[stage]);
      if (++stage == static_cast<uint32_t>(A_STAGES)) { stage = 0; phase ^= 1; }
      if (++pr_kb == num_kb) {
        // last k-block of the tile: publish this thread's share of the row's sum of squares
        pr_kb = 0;
        mbar_wait(&ss_empty[acc], acc_phase ^ 1);
        ss_s[(acc * 2 + half) * PM + m] = ss;
        mbar_arrive(&ss_full[acc]);
        ss = 0.f;
        if (++acc == P_ACC_STAGES) { acc = 0; acc_phase ^= 1; }
      }
    };

    float xa[32], xb[32];
    if (total_seq > 0) load_block(xa);
    for (long long seq = 0; seq < total_seq; seq += 2) {
      if (seq + 1 < total_seq) load_block(xb);
      process(xa);
      if (seq + 1 < total_seq) {
        if (seq + 2 < total_seq) load_block(xa);
        process(xb);
      }
    }
    }  // register path
  } else if (warp >= 4 && warp < 8) {
    // ===================== epilogue =====================
    const int ew = warp - 4;  // == warp % 4: TMEM lane quarter
    const int row = ew * 32 + lane;
    uint32_t acc = 0, acc_phase = 0;
    const bool vec_ok = (p.k & 3) == 0 && (reinterpret_cast<uintptr_t>(p.out) & 15u) == 0;
    for (long long tile = unit; tile < p.tiles; tile += num_units) {
      const long long R = (tile * 2 + rank) * PM + row;
      mbar_wait(&ss_full[acc], acc_phase);
      float rn = 1.0f;
      if (p.normalize) {
        const float ssum = ss_s[(acc * 2 + 0) * PM + row] + ss_s[(acc * 2 + 1) * PM + row];
        rn = 1.0f / fmaxf(sqrtf(ssum), 1e-12f);
      }
      __syncwarp();
      if (lane == 0) mbar_arrive(&ss_empty[acc]);
      mbar_wait(&tmem_full[acc], acc_phase);
      tc_fence_after();
      const uint32_t taddr = tmem_base + (static_cast<uint32_t>(ew * 32) << 16) + acc * kMaxComponents;
      float* orow = p.out + R * p.k;
#pragma unroll 1
      for (int c0 = 0; c0 < p.k_pad; c0 += 16) {
        uint32_t r[16];
        tmem_ld_32x16(taddr + c0, r);
        tc_wait_ld();
        if (R < p.m_total) {
          float v[16];
#pragma unroll
          for (int j = 0; j < 16; ++j) v[j] = fmaf(__uint_as_float(r[j]), rn, __ldg(p.bias + c0 + j));
          if (vec_ok && c0 + 16 <= p.k) {
#pragma unroll
            for (int j = 0; j < 4; ++j)
              *reinterpret_cast<float4*>(orow + c0 + 4 * j) = make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
          } else {
#pragma unroll
            for (int j = 0; j < 16; ++j)
              if (c0 + j < p.k) orow[c0 + j] = v[j];
          }
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive_leader(&tmem_empty[acc]);
      if (++acc == P_ACC_STAGES) { acc = 0; acc_phase ^= 1; }
    }
  }

  tc_fence_before();
  cluster_sync_all();
  if (warp == 2) {
    tc_fence_after();
    tmem_dealloc_pair(tmem_base, 512);
  }
}

// ------------------------------------------------------------------------------------------
// K3d: the per-cell kernel with NO raw staging (CTA pairs).  It takes the maps the TMA boxes of the
// staged kernel cannot express (e.g. 7 x 10 cells, or a map pointer off a 16-byte boundary) when its
// epilogue can: k % 4 == 0 and E % 16 == 0 (launch_project has the rules).
// Measured at config 3b, which a mode switch (since removed) sent here with an L2 prefetcher in warp 3
// (also removed), it runs at the staged kernel's speed (1.79 against 1.78 ms): with the raw ring
// and the A tiles gone from shared memory the port carries 128 KB per k-block instead of 272 KB and
// nothing got faster, which is what shows that the three tensor passes (1.15 PFLOP/s issued next to
// 3.6 TB/s of HBM traffic, at the 1 kW cap: 2.06 TFLOP take 1.49 ms at the sustained cuBLAS rate) — not
// shared memory — bound the exact mode.
// Shared memory carries only the weight tiles and the outgoing rows:
//   * the transform warps read the fp32 map straight from global memory — cells are the contiguous
//     dimension, so a warp's load of one channel is one 128-byte line — one k-block ahead in registers
//     (two register buffers: 32-64 KB of loads in flight per SM), accumulate the sums of squares, split to bf16 hi/lo and
//     write the A operand with tcgen05.st into TENSOR MEMORY (4 stages x 64 columns next to the
//     256-column accumulator); the MMAs take A from there (TS form);
//   * the epilogue scales by 1/||x||, adds the bias and hands 128-row x 32-column boxes (128-byte rows,
//     128B swizzle) to TMA stores: every global write is a full line instead of 16-byte pieces of
//     1 KB-strided rows.
// Per k-block a CTA's shared-memory port now moves 32 KB of weights in and 96 KB of weight reads out
// (its half and the peer's) = 1000 cycles at 128 B/clk, against 1536 tensor cycles: the kernel is bound
// by the three tensor passes that fp32-class accuracy costs, no longer by shared memory.
//   warp 0 weight TMA, warp 1 MMA issuer (leader), warp 2 TMEM alloc, warp 3 idle,
//   warps 4-7 epilogue, warps 8-23 transform: warp tw owns TMEM lane quarter tw % 4
//   (cells 32 (tw % 4) + lane of the tile) and features 16 (tw / 4) .. + 15 of every k-block.
// ------------------------------------------------------------------------------------------
constexpr int kProjDThreads = (kTransformWarp0 + 16) * 32;

struct ProjDSmem {
  static constexpr int A_STAGES = 4, W_STAGES = 2, OUT_BUFS = 8;  // one staging buffer per 32-column box of a tile
  static constexpr uint32_t W_PART_BYTES = (kMaxComponents / 2) * PK * 2;  // 16 KB
  static constexpr uint32_t W_STAGE_BYTES = 2 * W_PART_BYTES;              // hi + lo
  static constexpr uint32_t OUT_BUF_BYTES = PM * 32 * 4;                   // 128 rows x 32 columns fp32 = 16 KB
  static constexpr uint32_t kWOff = 0;
  static constexpr uint32_t kOutOff = kWOff + W_STAGES * W_STAGE_BYTES;
  static constexpr uint32_t kSsOff = kOutOff + OUT_BUFS * OUT_BUF_BYTES;   // [2][4 feature groups][128 rows]
  static constexpr uint32_t kBarOff = kSsOff + 2 * 4 * PM * 4;
  static constexpr uint32_t kNumBars = 2 * A_STAGES + 2 * W_STAGES + 2 + 4;
  static constexpr uint32_t kTmemPtrOff = kBarOff + kNumBars * 8;
  static constexpr uint32_t kTotal = kTmemPtrOff + 16;
  static constexpr uint32_t kDynamicBytes = kTotal + 1024;
  static constexpr uint32_t kAColumn0 = kMaxComponents;  // first A column in TMEM
};

__global__ void __launch_bounds__(kProjDThreads, 1)
l2norm_project_direct_kernel(const __grid_constant__ CUtensorMap tmap_whi, const __grid_constant__ CUtensorMap tmap_wlo,
                             const __grid_constant__ CUtensorMap tmap_out, const ProjParams p) {
  using L = ProjDSmem;
  constexpr int A_STAGES = L::A_STAGES, W_STAGES = L::W_STAGES;
  const uint32_t rank = cluster_ctarank();
  const long long unit = blockIdx.x / 2, num_units = gridDim.x / 2;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + L::kBarOff);
  uint64_t* a_full = bars;                       // [A]   16 transform warps x 2 CTAs (on the leader)
  uint64_t* a_empty = a_full + A_STAGES;         // [A]   tcgen05.commit (both CTAs)
  uint64_t* w_full = a_empty + A_STAGES;         // [W]   TMA of both CTAs (on the leader)
  uint64_t* w_empty = w_full + W_STAGES;         // [W]   tcgen05.commit (both CTAs)
  uint64_t* tmem_full = w_empty + W_STAGES;      // accumulator complete (both CTAs)
  uint64_t* tmem_empty = tmem_full + 1;          // 4 epilogue warps x 2 CTAs (on the leader)
  uint64_t* ss_full = tmem_empty + 1;            // [2]   16 transform warps
  uint64_t* ss_empty = ss_full + 2;              // [2]   4 epilogue warps
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(smem + L::kTmemPtrOff);
  float* ss_s = reinterpret_cast<float*>(smem + L::kSsOff);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int num_kb = (p.E + PK - 1) / PK;

  if (warp == 0 && lane == 0) {
    prefetch_tmap(&tmap_whi);
    prefetch_tmap(&tmap_wlo);
    prefetch_tmap(&tmap_out);
  }
  if (warp == 1 && lane == 0) {
    for (int i = 0; i < A_STAGES; ++i) { mbar_init(&a_full[i], 16 * 2); mbar_init(&a_empty[i], 1); }
    for (int i = 0; i < W_STAGES; ++i) { mbar_init(&w_full[i], 2); mbar_init(&w_empty[i], 1); }
    mbar_init(tmem_full, 1);
    mbar_init(tmem_empty, 4 * 2);
    for (int i = 0; i < 2; ++i) { mbar_init(&ss_full[i], 16); mbar_init(&ss_empty[i], 4); }
    fence_mbar_init();
  }
  if (warp == 2) { tmem_alloc_pair(tmem_ptr, 512); tmem_relinquish_pair(); }
  tc_fence_before();
  cluster_sync_all();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;
  const int w_rows = p.k_pad / 2;
  const uint32_t w_part_bytes = static_cast<uint32_t>(w_rows) * PK * 2;
  const long long my_tiles = (p.tiles - unit + num_units - 1) / num_units;
  const long long total_seq = my_tiles * num_kb;

  if (warp == 0) {
    // ===================== weight TMA producer =====================
    if (lane == 0) {
      uint32_t stage = 0, phase = 0;
      const int32_t row0 = static_cast<int32_t>(rank) * w_rows;
      int kb = 0;
      for (long long seq = 0; seq < total_seq; ++seq) {
        mbar_wait(&w_empty[stage], phase ^ 1);
        uint8_t* dst = smem + L::kWOff + stage * L::W_STAGE_BYTES;
        mbar_arrive_expect_tx_leader(&w_full[stage], 2 * w_part_bytes);
        tma_load_2d_pair(dst, &tmap_whi, &w_full[stage], kb * PK, row0, kEvictLast);
        tma_load_2d_pair(dst + L::W_PART_BYTES, &tmap_wlo, &w_full[stage], kb * PK, row0, kEvictLast);
        if (++stage == W_STAGES) { stage = 0; phase ^= 1; }
        if (++kb == num_kb) kb = 0;
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer (leader CTA) =====================
    if (lane == 0 && rank == 0) {
      const uint32_t idesc = make_idesc(/*bf16*/ 1, PM * 2, static_cast<uint32_t>(p.k_pad));
      uint32_t as = 0, aph = 0, ws = 0, wph = 0, tph = 0;
      for (long long tile = 0; tile < my_tiles; ++tile) {
        mbar_wait(tmem_empty, tph ^ 1);  // the epilogues of both CTAs drained the accumulator
        tc_fence_after();
        for (int kb = 0; kb < num_kb; ++kb) {
          mbar_wait(&w_full[ws], wph);
          mbar_wait(&a_full[as], aph);
          tc_fence_after();
          const uint32_t a_hi = tmem_base + L::kAColumn0 + as * 64;
          const uint32_t a_lo = a_hi + 32;
          const uint32_t w_hi = smem_u32(smem + L::kWOff + ws * L::W_STAGE_BYTES);
          const uint32_t w_lo = w_hi + L::W_PART_BYTES;
#pragma unroll
          for (int k = 0; k < PK / P_UMMA_K; ++k) {
            const uint64_t dwh = make_kmajor_sw128_desc(w_hi + k * P_UMMA_K * 2);
            const uint64_t dwl = make_kmajor_sw128_desc(w_lo + k * P_UMMA_K * 2);
            tc_mma_f16_pair_ts(tmem_base, a_hi + k * 8, dwh, idesc, (kb | k) != 0);
            tc_mma_f16_pair_ts(tmem_base, a_lo + k * 8, dwh, idesc, 1);
            tc_mma_f16_pair_ts(tmem_base, a_hi + k * 8, dwl, idesc, 1);
          }
          tc_commit_pair(&a_empty[as]);
          tc_commit_pair(&w_empty[ws]);
          if (++as == A_STAGES) { as = 0; aph ^= 1; }
          if (++ws == W_STAGES) { ws = 0; wph ^= 1; }
        }
        tc_commit_pair(tmem_full);
        tph ^= 1;
      }
    }
  } else if (warp >= kTransformWarp0) {
    // ===================== transform: fp32 map (global) -> bf16 hi/lo (TMEM) =====================
    const int tw = warp - kTransformWarp0;
    const int lq = tw & 3;            // == warp % 4: the TMEM lane quarter this warp may access
    const int fg = tw >> 2;           // feature group: 16 features of the k-block
    const int m = lq * 32 + lane;     // row (cell) inside the tile
    const uint32_t t_row = tmem_base + (static_cast<uint32_t>(lq * 32) << 16) + L::kAColumn0 + fg * 8;
    const long long hw = p.hw;
    // load cursor: one k-block ahead of the convert cursor
    long long ld_tile = 0;
    int ld_kb = 0;
    const float* ld_base = nullptr;
    bool ld_valid = false;
    auto seek = [&](long long tile_iter) {
      const long long R = ((unit + tile_iter * num_units) * 2 + rank) * PM + m;
      ld_valid = tile_iter < my_tiles && R < p.m_total;
      const long long img = ld_valid ? R / hw : 0;  // once per tile
      const long long cell = ld_valid ? R - img * hw : 0;
      ld_base = p.fmap + img * p.E * hw + cell;
    };
    seek(0);
    auto ld_f32 = [](const float* ptr) {
      float v;
      asm volatile("ld.global.nc.L1::no_allocate.f32 %0, [%1];" : "=f"(v) : "l"(ptr));
      return v;
    };
    // E % 16 == 0 (host-checked): a thread's 16 features of a k-block exist together or not at all
    auto load_block = [&](float (&x)[16]) {
      const int f0 = ld_kb * PK + fg * 16;
      const float* src = ld_base + static_cast<long long>(f0) * hw;
      const bool live = ld_valid && f0 < p.E;
      if (live) {
#pragma unroll
        for (int i = 0; i < 16; ++i) { x[i] = ld_f32(src); src += hw; }
      } else {
#pragma unroll
        for (int i = 0; i < 16; ++i) x[i] = 0.f;
      }
      if (++ld_kb == num_kb) { ld_kb = 0; seek(++ld_tile); }
    };
    float ss = 0.f;
    uint32_t as = 0, aph = 0, sst = 0, ssph = 0;
    int pr_kb = 0;
    // convert one k-block's 16 features (two halves of 8: four packed columns of hi and of lo each)
    // and hand it to the MMA
    auto process = [&](float (&x)[16]) {
      mbar_wait(&a_empty[as], aph ^ 1);
      tc_fence_after();
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        uint32_t hi[4], lo[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const float a = x[8 * h + 2 * i], b = x[8 * h + 2 * i + 1];
          ss = fmaf(a, a, ss);
          ss = fmaf(b, b, ss);
          // hi = x truncated to bf16 (a mask); lo = RN_bf16(x - hi): |x - hi - lo| <= 2^-16 |x|
          const uint32_t ab = __float_as_uint(a), bb = __float_as_uint(b);
          hi[i] = __byte_perm(ab, bb, 0x7632);
          const float la = a - __uint_as_float(ab & 0xFFFF0000u);
          const float lb = b - __uint_as_float(bb & 0xFFFF0000u);
          const __nv_bfloat162 l2 = __floats2bfloat162_rn(la, lb);
          lo[i] = *reinterpret_cast<const uint32_t*>(&l2);
        }
        tmem_st_32x4(t_row + as * 64 + 4 * h, hi);
        tmem_st_32x4(t_row + as * 64 + 32 + 4 * h, lo);
      }
      tc_wait_st();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive_leader(&a_full[as]);
      if (++as == A_STAGES) { as = 0; aph ^= 1; }
      if (++pr_kb == num_kb) {
        // last k-block of the tile: publish this warp's share of the rows' sums of squares
        pr_kb = 0;
        mbar_wait(&ss_empty[sst], ssph ^ 1);
        ss_s[(sst * 4 + fg) * PM + m] = ss;
        __syncwarp();
        if (lane == 0) mbar_arrive(&ss_full[sst]);
        ss = 0.f;
        if (++sst == 2) { sst = 0; ssph ^= 1; }
      }
    };
    // two register buffers: the loads of k-block n + 1 are in flight while k-block n waits for its
    // operand stage, is converted and stored — a whole k-block period of latency cover per warp
    float xa[16], xb[16];
    if (total_seq > 0) load_block(xa);
    for (long long seq = 0; seq < total_seq; seq += 2) {
      if (seq + 1 < total_seq) load_block(xb);
      process(xa);
      if (seq + 1 < total_seq) {
        if (seq + 2 < total_seq) load_block(xa);
        process(xb);
      }
    }
  } else if (warp >= 4 && warp < 8) {
    // ===================== epilogue =====================
    const int ew = warp - 4;  // == warp % 4: TMEM lane quarter
    const int row = ew * 32 + lane;
    const int et = threadIdx.x - 4 * 32;  // 0..127
    uint32_t sst = 0, ssph = 0, tph = 0;
    auto epi_bar = [] { asm volatile("bar.sync 1, 128;" ::: "memory"); };
    for (long long tile = unit; tile < p.tiles; tile += num_units) {
      const long long R0 = (tile * 2 + rank) * PM;
      mbar_wait(&ss_full[sst], ssph);
      float rn = 1.0f;
      if (p.normalize) {
        const float* sp = ss_s + sst * 4 * PM + row;
        const float ssum = (sp[0] + sp[PM]) + (sp[2 * PM] + sp[3 * PM]);
        rn = 1.0f / fmaxf(sqrtf(ssum), 1e-12f);
      }
      __syncwarp();
      if (lane == 0) mbar_arrive(&ss_empty[sst]);
      if (++sst == 2) { sst = 0; ssph ^= 1; }
      // the staging buffers still belong to the previous tile's TMA stores (issued a whole tile ago)
      if (et == 0) tma_store_wait_read<0>();
      epi_bar();
      mbar_wait(tmem_full, tph);
      tph ^= 1;
      tc_fence_after();
      const uint32_t taddr = tmem_base + (static_cast<uint32_t>(ew * 32) << 16);
      // Drain: the accumulator is the only one (the A stages take the other half of TMEM), so the MMAs
      // of the next tile wait for this loop.  It does nothing but load 32 columns, scale them and park
      // them in their own staging buffer — no barrier, no store wait inside — with the next load in
      // flight while a box is processed; the TMA stores go out after the accumulator is released.
      uint32_t ra[16], rb[16];
      const int nbox = (p.k_pad + 31) >> 5;
      const int nhalf = p.k_pad >> 4;  // 16-column pieces (k_pad is a multiple of 16)
      auto park = [&](const uint32_t (&r)[16], int h) {
        uint8_t* obuf = smem + L::kOutOff + (h >> 1) * L::OUT_BUF_BYTES + row * 128;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const float4 bz = __ldg(reinterpret_cast<const float4*>(p.bias + h * 16) + j);
          float4 v;
          v.x = fmaf(__uint_as_float(r[4 * j + 0]), rn, bz.x);
          v.y = fmaf(__uint_as_float(r[4 * j + 1]), rn, bz.y);
          v.z = fmaf(__uint_as_float(r[4 * j + 2]), rn, bz.z);
          v.w = fmaf(__uint_as_float(r[4 * j + 3]), rn, bz.w);
          *reinterpret_cast<float4*>(obuf + ((((h & 1) << 2) + j) ^ (row & 7)) * 16) = v;  // 128B swizzle
        }
      };
      auto release = [&] {
        // every TMEM read of this tile has landed: the MMAs of the next tile may start
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive_leader(tmem_empty);
      };
      tmem_ld_32x16(taddr, ra);
#pragma unroll 1
      for (int h = 0; h < nhalf; h += 2) {
        tc_wait_ld_regs16(ra);
        const bool more = h + 1 < nhalf;
        if (more) tmem_ld_32x16(taddr + (h + 1) * 16, rb);
        else release();
        park(ra, h);
        if (more) {
          tc_wait_ld_regs16(rb);
          if (h + 2 < nhalf) tmem_ld_32x16(taddr + (h + 2) * 16, ra);
          else release();
          park(rb, h + 1);
        }
      }
      fence_proxy_async_smem();
      epi_bar();
      if (et == 0) {
        for (int bx = 0; bx < nbox; ++bx)
          tma_store_2d(&tmap_out, smem + L::kOutOff + bx * L::OUT_BUF_BYTES, bx * 32, static_cast<int32_t>(R0));
        tma_store_commit();
      }
    }
    if (et == 0) tma_store_wait<0>();
  }

  tc_fence_before();
  cluster_sync_all();
  if (warp == 2) {
    tc_fence_after();
    tmem_dealloc_pair(tmem_base, 512);
  }
}

// ------------------------------------------------------------------------------------------
// K3p: pooled[b][e] = (1/hw) * sum_cells x[b][e][cell] * rnorm[b][cell]  — one pass over the map.
// One CTA per image at a time; 16-cell slabs [E][16] double-buffered in shared memory via cp.async.
// ------------------------------------------------------------------------------------------
constexpr int kSlabCells = 16;
constexpr int kPoolThreads = 256;
constexpr int kPoolMaxAcc = 24;  // channels per thread: E <= 64 * 24 = 1536

__device__ __forceinline__ void cp_async_4(void* smem_dst, const void* gsrc) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(smem_u32(smem_dst)), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async_16(void* smem_dst, const void* gsrc) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_u32(smem_dst)), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

__global__ void __launch_bounds__(kPoolThreads)
l2norm_pool_kernel(const float* __restrict__ fmap, int B, int E, int hw, float* __restrict__ pooled) {
  extern __shared__ __align__(16) uint8_t pool_smem[];
  float* slab[2] = {reinterpret_cast<float*>(pool_smem),
                    reinterpret_cast<float*>(pool_smem) + static_cast<size_t>(E) * kSlabCells};
  __shared__ float part[16][kSlabCells];
  __shared__ float rn_s[kSlabCells];
  const int t = threadIdx.x;
  const int nslab = (hw + kSlabCells - 1) / kSlabCells;
  const bool vec = (hw & 3) == 0 && (reinterpret_cast<uintptr_t>(fmap) & 15u) == 0;

  auto issue = [&](int b, int s, float* dst) {
    const float* src = fmap + static_cast<long long>(b) * E * hw + s * kSlabCells;
    const int cells = min(kSlabCells, hw - s * kSlabCells);
    if (vec) {
      // hw % 4 == 0: whole 16-byte quads are either inside the image row or outside
      for (int i = t; i < E * 4; i += kPoolThreads) {
        const int e = i >> 2, qd = i & 3;
        float* d = dst + e * kSlabCells + qd * 4;
        if (qd * 4 < cells) cp_async_16(d, src + static_cast<long long>(e) * hw + qd * 4);
        else *reinterpret_cast<float4*>(d) = make_float4(0.f, 0.f, 0.f, 0.f);
      }
    } else {
      for (int i = t; i < E * kSlabCells; i += kPoolThreads) {
        const int e = i >> 4, c = i & 15;
        float* d = dst + e * kSlabCells + c;
        if (c < cells) cp_async_4(d, src + static_cast<long long>(e) * hw + c);
        else *d = 0.f;
      }
    }
    cp_async_commit();
  };

  for (int b = blockIdx.x; b < B; b += gridDim.x) {
    float acc[kPoolMaxAcc];
#pragma unroll
    for (int i = 0; i < kPoolMaxAcc; ++i) acc[i] = 0.f;
    issue(b, 0, slab[0]);
    for (int s = 0; s < nslab; ++s) {
      float* cur = slab[s & 1];
      if (s + 1 < nslab) { issue(b, s + 1, slab[(s + 1) & 1]); cp_async_wait<1>(); }
      else cp_async_wait<0>();
      __syncthreads();
      // per-cell sum of squares: thread = (cell, part), 16 parts stride over the channels
      {
        const int cell = t & 15, prt = t >> 4;
        float ssq = 0.f;
        for (int e = prt; e < E; e += 16) {
          const float v = cur[e * kSlabCells + cell];
          ssq = fmaf(v, v, ssq);
        }
        part[prt][cell] = ssq;
      }
      __syncthreads();
      if (t < kSlabCells) {
        float ssq = 0.f;
#pragma unroll
        for (int i = 0; i < 16; ++i) ssq += part[i][t];
        const bool live = s * kSlabCells + t < hw;
        rn_s[t] = live ? 1.0f / fmaxf(sqrtf(ssq), 1e-12f) : 0.f;
      }
      __syncthreads();
      // weighted channel sums: thread = (channel group, quarter of the 16 cells)
      {
        const int qd = t & 3;
        const float4 w = *reinterpret_cast<const float4*>(&rn_s[qd * 4]);
#pragma unroll
        for (int i = 0; i < kPoolMaxAcc; ++i) {
          const int e = (t >> 2) + 64 * i;
          if (e < E) {
            const float4 v = *reinterpret_cast<const float4*>(cur + e * kSlabCells + qd * 4);
            acc[i] = fmaf(v.x, w.x, fmaf(v.y, w.y, fmaf(v.z, w.z, fmaf(v.w, w.w, acc[i]))));
          }
        }
      }
      __syncthreads();  // everyone is done with `cur` before it is refilled two slabs later
    }
    const float inv = 1.0f / static_cast<float>(hw);
#pragma unroll
    for (int i = 0; i < kPoolMaxAcc; ++i) {
      float v = acc[i];
      v += __shfl_xor_sync(kFullMask, v, 1);
      v += __shfl_xor_sync(kFullMask, v, 2);
      const int e = (t >> 2) + 64 * i;
      if ((t & 3) == 0 && e < E) pooled[static_cast<long long>(b) * E + e] = v * inv;
    }
  }
}

// ------------------------------------------------------------------------------------------
// K3p (TMA flavour): the same single pass, but every 16-cell slab [E][16] arrives by TMA
// (3-D tensor map over (cell, feature, image), boxes of 16 cells x 256 features) into one of two
// 80 KB buffers while the CTA works on the other: memory latency is hidden by up to 80 KB in flight
// per SM instead of per-thread cp.async granules.  Needs hw % 4 == 0 (16-byte global strides).
// ------------------------------------------------------------------------------------------
constexpr int kPoolFeatBox = 256;  // features per TMA box

__global__ void __launch_bounds__(kPoolThreads, 1)
l2norm_pool_tma_kernel(const __grid_constant__ CUtensorMap tmap, int B, int E, int hw, float* __restrict__ pooled) {
  extern __shared__ uint8_t pool_tma_raw[];
  // TMA destinations need 128-byte alignment; the dynamic window follows the static arrays below
  uint8_t* pool_smem = pool_tma_raw + ((128u - (smem_u32(pool_tma_raw) & 127u)) & 127u);
  __shared__ __align__(8) uint64_t full_bar[2];
  __shared__ float part[16][kSlabCells];
  __shared__ __align__(16) float rn_s[kSlabCells];
  const int t = threadIdx.x;
  const int nbox = (E + kPoolFeatBox - 1) / kPoolFeatBox;
  const uint32_t slab_bytes = static_cast<uint32_t>(nbox) * kPoolFeatBox * kSlabCells * 4;
  const int nslab = (hw + kSlabCells - 1) / kSlabCells;
  const long long my_images = (B - static_cast<long long>(blockIdx.x) + gridDim.x - 1) / gridDim.x;
  const long long total = my_images * nslab;

  if (t == 0) {
    prefetch_tmap(&tmap);
    mbar_init(&full_bar[0], 1);
    mbar_init(&full_bar[1], 1);
    fence_mbar_init();
  }
  __syncthreads();

  auto issue = [&](long long seq) {  // thread 0 only
    const int buf = static_cast<int>(seq & 1);
    const long long img = blockIdx.x + (seq / nslab) * gridDim.x;
    const int slab = static_cast<int>(seq % nslab);
    mbar_arrive_expect_tx(&full_bar[buf], slab_bytes);
    uint8_t* dst = pool_smem + static_cast<size_t>(buf) * slab_bytes;
    for (int bx = 0; bx < nbox; ++bx)
      tma_load_3d(dst + static_cast<size_t>(bx) * kPoolFeatBox * kSlabCells * 4, &tmap, &full_bar[buf],
                  slab * kSlabCells, bx * kPoolFeatBox, static_cast<int32_t>(img), kEvictFirst);
  };

  float acc[kPoolMaxAcc / 4];  // features t + 256 j
#pragma unroll
  for (int j = 0; j < kPoolMaxAcc / 4; ++j) acc[j] = 0.f;
  if (t == 0 && total > 0) issue(0);
  for (long long seq = 0; seq < total; ++seq) {
    const int buf = static_cast<int>(seq & 1);
    // the other buffer was released by the barrier that ended iteration seq - 1
    if (t == 0 && seq + 1 < total) issue(seq + 1);
    mbar_wait(&full_bar[buf], static_cast<uint32_t>((seq >> 1) & 1));
    const float* cur = reinterpret_cast<const float*>(pool_smem + static_cast<size_t>(buf) * slab_bytes);
    const int slab = static_cast<int>(seq % nslab);
    // per-cell sum of squares: thread = (cell, part); a warp reads two whole 64-byte rows per step
    {
      const int cell = t & 15, prt = t >> 4;
      float ssq = 0.f;
      for (int e = prt; e < E; e += 16) {
        const float v = cur[e * kSlabCells + cell];
        ssq = fmaf(v, v, ssq);
      }
      part[prt][cell] = ssq;
    }
    __syncthreads();
    if (t < kSlabCells) {
      float ssq = 0.f;
#pragma unroll
      for (int i = 0; i < 16; ++i) ssq += part[i][t];
      const bool live = slab * kSlabCells + t < hw;
      rn_s[t] = live ? 1.0f / fmaxf(sqrtf(ssq), 1e-12f) : 0.f;
    }
    __syncthreads();
    // weighted channel sums: thread owns features t + 256 j and reads their whole 16-cell rows; the
    // quad order is rotated by row so that eight lanes cover all 32 banks
    {
      const int rot = (t >> 1) & 3;
      float4 w[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) w[i] = *reinterpret_cast<const float4*>(&rn_s[((i + rot) & 3) * 4]);
#pragma unroll
      for (int j = 0; j < kPoolMaxAcc / 4; ++j) {
        const int e = t + kPoolThreads * j;
        if (e < E) {
          const float* row = cur + e * kSlabCells;
          float a = acc[j];
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            const float4 v = *reinterpret_cast<const float4*>(row + ((i + rot) & 3) * 4);
            a = fmaf(v.x, w[i].x, fmaf(v.y, w[i].y, fmaf(v.z, w[i].z, fmaf(v.w, w[i].w, a))));
          }
          acc[j] = a;
        }
      }
    }
    if (slab == nslab - 1) {
      const long long img = blockIdx.x + (seq / nslab) * gridDim.x;
      const float inv = 1.0f / static_cast<float>(hw);
#pragma unroll
      for (int j = 0; j < kPoolMaxAcc / 4; ++j) {
        const int e = t + kPoolThreads * j;
        if (e < E) pooled[img * E + e] = acc[j] * inv;
        acc[j] = 0.f;
      }
    }
    // The refill of `cur` is a TMA write (async proxy); as in the staged projection kernel's raw ring,
    // the proxy fence completes this thread's generic reads of the buffer before the barrier releases it.
    fence_proxy_async_smem();
    __syncthreads();  // everyone is done with `cur` (and part/rn_s) before the buffer is refilled
  }
}

// Launches a per-cell projection kernel on CTA pairs (clusters of two CTAs).
template <typename... Params, typename... Args>
int launch_pair(void (*kern)(Params...), int threads, uint32_t smem, int grid, cudaStream_t stream, const Args&... args) {
  ISX_CHECK_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(static_cast<unsigned>(grid));
  cfg.blockDim = dim3(static_cast<unsigned>(threads));
  cfg.dynamicSmemBytes = static_cast<size_t>(smem);
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 2;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  ISX_CHECK_CUDA(cudaLaunchKernelEx(&cfg, kern, args...));
  return ISX_OK;
}

// Projects m_total cells of an NCHW map (hw cells per image; hw == 1 for an n x E matrix).  The kernel
// follows from the input's shape and alignment alone, by the first rule that fits.
int launch_project(const float* fmap, long long m_total, int E, int hw, int k, int normalize, int fast,
                   const void* packed, float* out, cudaStream_t stream) {
  const PackedLayout l = packed_layout(E, k);
  const uint8_t* pk = static_cast<const uint8_t*>(packed);
  CUtensorMap twh, twl;  // each CTA of a pair stages half of the weight rows
  int rc = encode_tmap_2d(&twh, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, pk + l.hi_off, static_cast<uint64_t>(l.k_pad),
                          static_cast<uint64_t>(l.f_pad), static_cast<uint64_t>(l.f_pad) * 2,
                          static_cast<uint32_t>(l.k_pad / 2), PK, CU_TENSOR_MAP_SWIZZLE_128B);
  if (rc != ISX_OK) return rc;
  rc = encode_tmap_2d(&twl, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, pk + l.lo_off, static_cast<uint64_t>(l.k_pad),
                      static_cast<uint64_t>(l.f_pad), static_cast<uint64_t>(l.f_pad) * 2,
                      static_cast<uint32_t>(l.k_pad / 2), PK, CU_TENSOR_MAP_SWIZZLE_128B);
  if (rc != ISX_OK) return rc;
  int sms = 148;
  rc = device_sm_count(&sms);
  if (rc != ISX_OK) return rc;
  ProjParams p;
  p.fmap = fmap; p.m_total = m_total; p.E = E; p.hw = hw; p.k = k; p.k_pad = l.k_pad;
  p.fast = 0;
  p.rowmajor = 0;
  p.normalize = normalize;
  p.tiles = (m_total + 2 * PM - 1) / (2 * PM);  // tiles of 128 cells per CTA (256 per pair)
  p.bias = reinterpret_cast<const float*>(pk + l.bias_off);
  p.out = out;
  const int grid = static_cast<int>(std::min<long long>(sms / 2, p.tiles)) * 2;
  const bool map_aligned = (reinterpret_cast<uintptr_t>(fmap) & 15u) == 0;

  // 1. n x E row-major input (PCA.transform's flat vectors, the pooled rows): the staged kernel on a
  //    2-D map with 128B-swizzled boxes of 128 rows x 32 features.
  const bool rowmajor = hw == 1 && E % 4 == 0 && map_aligned && m_total < (1ll << 31);
  // 2. Rule 1 needs one cell per image.  A map of several cells per image takes the staged kernel on
  //    a 3-D map over (cell, feature, image) when its strides are whole 16-byte units and a tile of 128
  //    cells is a fraction of one image (hw % 128 == 0) or a whole number of images (128 % hw == 0).
  const bool boxes = hw % 4 == 0 && map_aligned && (hw % PM == 0 || PM % hw == 0);
  if (rowmajor || boxes) {
    CUtensorMap tx;
    if (rowmajor) {
      rc = encode_tmap_2d(&tx, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, fmap, static_cast<uint64_t>(m_total),
                          static_cast<uint64_t>(E), static_cast<uint64_t>(E) * 4, PM, 32, CU_TENSOR_MAP_SWIZZLE_128B);
    } else {
      const uint32_t cells_box = static_cast<uint32_t>(std::min(hw, PM));
      const uint32_t imgs_box = static_cast<uint32_t>(PM / static_cast<int>(cells_box));
      rc = encode_tmap_3d(&tx, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, fmap, static_cast<uint64_t>(hw), static_cast<uint64_t>(E),
                          static_cast<uint64_t>(m_total / hw), static_cast<uint64_t>(hw) * 4,
                          static_cast<uint64_t>(E) * hw * 4, cells_box, PK, imgs_box, CU_TENSOR_MAP_SWIZZLE_NONE);
    }
    if (rc != ISX_OK) return rc;
    if (fast) {
      // single fp16 pass: tmap_whi describes the fp16 copy of the weights
      rc = encode_tmap_2d(&twh, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, pk + l.h_off, static_cast<uint64_t>(l.k_pad),
                          static_cast<uint64_t>(l.f_pad), static_cast<uint64_t>(l.f_pad) * 2,
                          static_cast<uint32_t>(l.k_pad / 2), PK, CU_TENSOR_MAP_SWIZZLE_128B);
      if (rc != ISX_OK) return rc;
    }
    p.rowmajor = rowmajor;
    p.fast = fast;
    return launch_pair(l2norm_project_kernel<true>, proj_threads(true), ProjSmem<true>::kDynamicBytes, grid, stream,
                       twh, twl, tx, p);
  }
  // 3. The map's shape or alignment gives no TMA boxes for the staged kernel.  K3d loads any shape from
  //    global memory; its TMA-store epilogue needs 16-byte output rows and its transform whole
  //    16-feature groups.  Only the staged kernel has the fp16 pass, so these shapes run the exact
  //    three-pass split even when the fp16 pass was asked for (more accurate, never less).
  if (k % 4 == 0 && E % 16 == 0 && (reinterpret_cast<uintptr_t>(out) & 15u) == 0 && m_total < (1ll << 31)) {
    CUtensorMap tout;
    rc = encode_tmap_2d(&tout, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, out, static_cast<uint64_t>(m_total),
                        static_cast<uint64_t>(k), static_cast<uint64_t>(k) * 4, PM, 32, CU_TENSOR_MAP_SWIZZLE_128B);
    if (rc != ISX_OK) return rc;
    return launch_pair(l2norm_project_direct_kernel, kProjDThreads, ProjDSmem::kDynamicBytes, grid, stream, twh, twl,
                       tout, p);
  }
  // 4. K3d cannot write this output (or E % 16 != 0): the register path loads any shape and stores
  //    rows of k floats.  It reads no map descriptor; twh only fills the slot.
  return launch_pair(l2norm_project_kernel<false>, proj_threads(false), ProjSmem<false>::kDynamicBytes, grid, stream,
                     twh, twl, twh, p);
}

}  // namespace
}  // namespace isx

using namespace isx;

extern "C" {

size_t isx_project_packed_bytes(int F, int k) {
  if (F <= 0 || k <= 0 || k > kMaxComponents) return 0;
  return packed_layout(F, k).total;
}

int isx_project_pack(const float* feature_means, const float* comps, int F, int k, int64_t ld_f,
                     int64_t ld_k, void* packed, size_t packed_bytes, isx_stream_t stream_) {
  const char* fn = "isx_project_pack";
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  ISX_REQUIRE(F > 0 && k > 0, "%s: need F > 0 and k > 0 (F=%d k=%d)", fn, F, k);
  ISX_REQUIRE(k <= kMaxComponents, "%s: at most %d components are supported (k=%d)", fn, kMaxComponents, k);
  ISX_REQUIRE(feature_means && comps && packed, "%s: null pointer", fn);
  const PackedLayout l = packed_layout(F, k);
  ISX_REQUIRE(packed_bytes >= l.total, "%s: packed buffer too small (%zu < %zu)", fn, packed_bytes, l.total);
  ISX_REQUIRE((reinterpret_cast<uintptr_t>(packed) & 255u) == 0, "%s: packed buffer must be 256-byte aligned", fn);
  uint8_t* pk = static_cast<uint8_t*>(packed);
  const int warps_per_block = 8;
  const int blocks = (l.k_pad + warps_per_block - 1) / warps_per_block;
  pack_weights_kernel<<<blocks, 256, 0, stream>>>(feature_means, comps, F, k, ld_f, ld_k, l.k_pad, l.f_pad,
                                                  reinterpret_cast<__nv_bfloat16*>(pk + l.hi_off),
                                                  reinterpret_cast<__nv_bfloat16*>(pk + l.lo_off),
                                                  reinterpret_cast<__half*>(pk + l.h_off),
                                                  reinterpret_cast<float*>(pk + l.bias_off));
  ISX_CHECK_CUDA(cudaGetLastError());
  return ISX_OK;
}

size_t isx_l2norm_project_workspace_bytes(int B, int E, int h, int w, int k, int pool) {
  (void)h; (void)w; (void)k;
  if (!pool || B <= 0 || E <= 0) return 256;
  return static_cast<size_t>(B) * E * sizeof(float) + 256;  // pooled B x E vectors
}

static int l2norm_project_impl(const char* fn, int fast, const float* fmap, int B, int E, int h, int w, int pool,
                               int normalize, const void* packed, int k, float* out, void* workspace,
                               size_t workspace_bytes, isx_stream_t stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  ISX_REQUIRE(B > 0 && E > 0 && h > 0 && w > 0 && k > 0, "%s: dimensions must be positive (B=%d E=%d h=%d w=%d k=%d)",
              fn, B, E, h, w, k);
  ISX_REQUIRE(k <= kMaxComponents, "%s: at most %d components are supported (k=%d)", fn, kMaxComponents, k);
  ISX_REQUIRE(fmap && packed && out, "%s: null pointer", fn);
  ISX_REQUIRE((reinterpret_cast<uintptr_t>(packed) & 255u) == 0, "%s: packed buffer must be 256-byte aligned", fn);
  const long long hw = static_cast<long long>(h) * w;
  ISX_REQUIRE(hw < (1ll << 24) && static_cast<long long>(B) * hw < (1ll << 40), "%s: feature map too large", fn);
  if (!pool) {
    return launch_project(fmap, static_cast<long long>(B) * hw, E, static_cast<int>(hw), k, normalize, fast, packed, out,
                          stream);
  }
  ISX_REQUIRE(normalize, "%s: pool == 1 requires normalize == 1", fn);
  ISX_REQUIRE(E <= 64 * kPoolMaxAcc, "%s: pooled mode supports at most %d channels (E=%d)", fn, 64 * kPoolMaxAcc, E);
  const size_t need = isx_l2norm_project_workspace_bytes(B, E, h, w, k, 1);
  ISX_REQUIRE(workspace && workspace_bytes >= need, "%s: workspace too small (%zu < %zu)", fn, workspace_bytes, need);
  float* pooled = reinterpret_cast<float*>((reinterpret_cast<uintptr_t>(workspace) + 255) & ~uintptr_t(255));
  int sms = 148;
  int rc = device_sm_count(&sms);
  if (rc != ISX_OK) return rc;
  if (hw % 4 == 0 && (reinterpret_cast<uintptr_t>(fmap) & 15u) == 0) {
    // TMA-staged slabs
    CUtensorMap tm;
    rc = encode_tmap_3d(&tm, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, fmap, static_cast<uint64_t>(hw), static_cast<uint64_t>(E),
                        static_cast<uint64_t>(B), static_cast<uint64_t>(hw) * 4, static_cast<uint64_t>(E) * hw * 4,
                        kSlabCells, kPoolFeatBox, 1, CU_TENSOR_MAP_SWIZZLE_NONE);
    if (rc != ISX_OK) return rc;
    const int nbox = (E + kPoolFeatBox - 1) / kPoolFeatBox;
    const size_t smem = static_cast<size_t>(2) * nbox * kPoolFeatBox * kSlabCells * sizeof(float) + 128;
    ISX_CHECK_CUDA(cudaFuncSetAttribute(l2norm_pool_tma_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                        static_cast<int>(smem)));
    const int grid = std::min(B, sms);
    l2norm_pool_tma_kernel<<<grid, kPoolThreads, smem, stream>>>(tm, B, E, static_cast<int>(hw), pooled);
    ISX_CHECK_CUDA(cudaGetLastError());
  } else {
    const size_t smem = static_cast<size_t>(2) * E * kSlabCells * sizeof(float);
    ISX_CHECK_CUDA(cudaFuncSetAttribute(l2norm_pool_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
    const int per_sm = std::max<int>(1, static_cast<int>((220 * 1024) / (smem + 2048)));
    const int grid = std::min(B, sms * per_sm);
    l2norm_pool_kernel<<<grid, kPoolThreads, smem, stream>>>(fmap, B, E, static_cast<int>(hw), pooled);
    ISX_CHECK_CUDA(cudaGetLastError());
  }
  // project the pooled rows: an n x F matrix is a feature "map" with one cell per image
  return launch_project(pooled, B, E, 1, k, /*normalize=*/0, fast, packed, out, stream);
}

int isx_l2norm_project(const float* fmap, int B, int E, int h, int w, int pool, int normalize,
                       const void* packed, int k, float* out, void* workspace, size_t workspace_bytes,
                       isx_stream_t stream) {
  return l2norm_project_impl("isx_l2norm_project", 0, fmap, B, E, h, w, pool, normalize, packed, k, out, workspace,
                             workspace_bytes, stream);
}

int isx_l2norm_project_fp16(const float* fmap, int B, int E, int h, int w, int pool, int normalize,
                            const void* packed, int k, float* out, void* workspace, size_t workspace_bytes,
                            isx_stream_t stream) {
  return l2norm_project_impl("isx_l2norm_project_fp16", 1, fmap, B, E, h, w, pool, normalize, packed, k, out,
                             workspace, workspace_bytes, stream);
}

}  // extern "C"
