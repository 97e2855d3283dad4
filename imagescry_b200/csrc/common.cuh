// Shared device/host helpers for the imagescry_b200 sm_100a kernels.
//
// Everything here is written for Blackwell (sm_100a) only: raw PTX wrappers for
// mbarrier, TMA (cp.async.bulk.tensor), tcgen05 (MMA / TMEM alloc / TMEM load),
// plus the host-side error plumbing shared by the C-ABI entry points.
#pragma once

#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include <cstdarg>
#include <cstdio>

#include "imagescry_b200.h"  // status codes, layouts, dtypes, entry-point declarations

namespace isx {

// Per-thread last-error string (the only mutable global state of the library).
char* last_error_buffer();
int set_error(int code, const char* fmt, ...);

#define ISX_CHECK_CUDA(expr)                                                             \
  do {                                                                                   \
    cudaError_t _e = (expr);                                                             \
    if (_e != cudaSuccess) {                                                             \
      return ::isx::set_error(ISX_ERR_CUDA, "%s failed at %s:%d: %s", #expr, __FILE__,   \
                              __LINE__, cudaGetErrorString(_e));                         \
    }                                                                                    \
  } while (0)

#define ISX_REQUIRE(cond, ...)                                       \
  do {                                                               \
    if (!(cond)) {                                                   \
      return ::isx::set_error(ISX_ERR_INVALID_ARG, __VA_ARGS__);     \
    }                                                                \
  } while (0)

int device_sm_count(int* out);

// Encode a 2-D row-major tensor map: global tensor [rows][cols] of `elem_bytes`-sized elements
// (row pitch `row_pitch_bytes`), box [box_rows][box_cols], 128-byte swizzle, zero OOB fill.
int encode_tmap_2d(CUtensorMap* map, CUtensorMapDataType dtype, int elem_bytes, const void* base,
                   uint64_t rows, uint64_t cols, uint64_t row_pitch_bytes, uint32_t box_rows,
                   uint32_t box_cols, CUtensorMapSwizzle swizzle);
// 3-D variant: tensor [d2][d1][d0] with byte strides (stride1, stride2) for d1/d2.
int encode_tmap_3d(CUtensorMap* map, CUtensorMapDataType dtype, int elem_bytes, const void* base,
                   uint64_t d0, uint64_t d1, uint64_t d2, uint64_t stride1_bytes,
                   uint64_t stride2_bytes, uint32_t box0, uint32_t box1, uint32_t box2,
                   CUtensorMapSwizzle swizzle);

}  // namespace isx

#ifdef __CUDACC__
namespace isx {

constexpr uint32_t kFullMask = 0xffffffffu;

// ----------------------------------------------------------------------------
// Small utilities
// ----------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

__device__ __forceinline__ uint32_t lane_id() {
  uint32_t l;
  asm volatile("mov.u32 %0, %%laneid;" : "=r"(l));
  return l;
}

__device__ __forceinline__ bool elect_one_sync() {
  uint32_t pred = 0;
  asm volatile(
      "{\n\t"
      ".reg .pred P;\n\t"
      "elect.sync _|P, 0xffffffff;\n\t"
      "selp.b32 %0, 1, 0, P;\n\t"
      "}\n"
      : "=r"(pred));
  return pred != 0;
}

// 128-bit streaming global accesses (no L1 allocation).
__device__ __forceinline__ uint4 ld_nc_v4(const void* ptr) {
  uint4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0, %1, %2, %3}, [%4];"
               : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
               : "l"(ptr));
  return r;
}
__device__ __forceinline__ void st_na_v4(void* ptr, const uint4& v) {
  asm volatile("st.global.L1::no_allocate.v4.u32 [%0], {%1, %2, %3, %4};" ::"l"(ptr), "r"(v.x),
               "r"(v.y), "r"(v.z), "r"(v.w)
               : "memory");
}
__device__ __forceinline__ void st_cs_v4(void* ptr, const uint4& v) {
  asm volatile("st.global.cs.v4.u32 [%0], {%1, %2, %3, %4};" ::"l"(ptr), "r"(v.x), "r"(v.y),
               "r"(v.z), "r"(v.w)
               : "memory");
}

// ----------------------------------------------------------------------------
// mbarrier
// ----------------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count)
               : "memory");
}
__device__ __forceinline__ void fence_mbar_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async_smem() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)),
               "r"(bytes)
               : "memory");
}
// Suspend-time hint: the waiting thread sleeps in hardware until the phase completes (or this many
// nanoseconds pass) instead of polling, so waiting warps do not take issue slots from working ones.
constexpr uint32_t kMbarSuspendHintNs = 0x989680u;
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t"
      ".reg .pred P;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 P, [%1], %2, %3;\n\t"
      "selp.b32 %0, 1, 0, P;\n\t"
      "}\n"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity), "r"(kMbarSuspendHintNs)
      : "memory");
  return ok != 0;
}

// Bounded wait: a protocol bug turns into a trap (launch failure reported to the host) instead of a
// hung GPU.  The bound is wall-clock (%globaltimer, checked every 1024 polls): no legitimate wait
// inside these kernels lasts anywhere near it.
#ifndef ISX_MBAR_TIMEOUT_NS
#define ISX_MBAR_TIMEOUT_NS 4000000000ull
#endif
__device__ __forceinline__ uint64_t global_timer_ns() {
  uint64_t t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  if (mbar_try_wait(bar, parity)) return;
  uint32_t spins = 0;
  uint64_t t0 = 0;
  while (!mbar_try_wait(bar, parity)) {
    if ((++spins & 1023u) == 0) {
      const uint64_t now = global_timer_ns();
      if (t0 == 0) t0 = now;
      else if (now - t0 > ISX_MBAR_TIMEOUT_NS) {
        printf("isx: mbarrier wait timed out (block %d thread %d smem 0x%x parity %u)\n", blockIdx.x,
               threadIdx.x, smem_u32(bar), parity);
        __trap();
      }
    }
  }
}

// ----------------------------------------------------------------------------
// TMA
// ----------------------------------------------------------------------------
__device__ __forceinline__ void prefetch_tmap(const CUtensorMap* map) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(map)) : "memory");
}

// L2 cache-policy constants (same encodings CUTLASS uses for TMA cache hints).
constexpr uint64_t kEvictNormal = 0x1000000000000000ull;
constexpr uint64_t kEvictFirst = 0x12F0000000000000ull;
constexpr uint64_t kEvictLast = 0x14F0000000000000ull;

__device__ __forceinline__ void tma_load_2d(void* smem_dst, const CUtensorMap* map, uint64_t* bar,
                                            int32_t c0, int32_t c1, uint64_t cache_hint) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes"
      ".L2::cache_hint [%0], [%1, {%3, %4}], [%2], %5;"
      ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(bar)),
      "r"(c0), "r"(c1), "l"(cache_hint)
      : "memory");
}
__device__ __forceinline__ void tma_load_3d(void* smem_dst, const CUtensorMap* map, uint64_t* bar,
                                            int32_t c0, int32_t c1, int32_t c2,
                                            uint64_t cache_hint) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes"
      ".L2::cache_hint [%0], [%1, {%3, %4, %5}], [%2], %6;"
      ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(bar)),
      "r"(c0), "r"(c1), "r"(c2), "l"(cache_hint)
      : "memory");
}
__device__ __forceinline__ void tma_store_2d(const CUtensorMap* map, const void* smem_src,
                                             int32_t c0, int32_t c1) {
  asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.tile.bulk_group [%0, {%2, %3}], [%1];"
               ::"l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(smem_src)), "r"(c0), "r"(c1)
               : "memory");
}
__device__ __forceinline__ void tma_store_commit() {
  asm volatile("cp.async.bulk.commit_group;" ::: "memory");
}
template <int N>
__device__ __forceinline__ void tma_store_wait_read() {
  asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory");
}
template <int N>
__device__ __forceinline__ void tma_store_wait() {
  asm volatile("cp.async.bulk.wait_group %0;" ::"n"(N) : "memory");
}

// ----------------------------------------------------------------------------
// tcgen05 / TMEM
// ----------------------------------------------------------------------------
__device__ __forceinline__ void tmem_alloc(uint32_t* smem_result, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(
                   smem_u32(smem_result)),
               "r"(ncols)
               : "memory");
}
__device__ __forceinline__ void tmem_relinquish() {
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols)
               : "memory");
}
__device__ __forceinline__ void tc_fence_before() {
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_after() {
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
}
// Arrive on an mbarrier once every previously issued tcgen05.mma of this thread has completed.
__device__ __forceinline__ void tc_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(
                   smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ void tc_wait_ld() {
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

// D[tmem] (+)= A[smem] * B[smem]; kind::f16 covers bf16/fp16 inputs with fp32 accumulation.
__device__ __forceinline__ void tc_mma_f16(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc,
                                           uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
      "}\n" ::"r"(d_tmem),
      "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void tc_mma_tf32(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc,
                                            uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t"
      "}\n" ::"r"(d_tmem),
      "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}

// ----------------------------------------------------------------------------
// CTA pairs (cta_group::2): two CTAs of one cluster on the two SMs of a TPC run one MMA of M = 256.
// Shared-memory addresses of the executing CTA have bit 24 set in CTA 1 of the pair; clearing it
// names the same offset in CTA 0 (the leader).
// ----------------------------------------------------------------------------
constexpr uint32_t kPeerBitMask = 0xFEFFFFFFu;

__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// arrive (+ expect_tx) on the barrier at the same offset in the pair's leader CTA
__device__ __forceinline__ void mbar_arrive_expect_tx_leader(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cluster.b64 _, [%0], %1;" ::"r"(smem_u32(bar) & kPeerBitMask),
               "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void mbar_arrive_leader(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(smem_u32(bar) & kPeerBitMask) : "memory");
}
// TMA load into this CTA's shared memory, completion bytes reported to the leader CTA's barrier
__device__ __forceinline__ void tma_load_2d_pair(void* smem_dst, const CUtensorMap* map, uint64_t* bar,
                                                 int32_t c0, int32_t c1, uint64_t cache_hint) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes"
      ".L2::cache_hint [%0], [%1, {%3, %4}], [%2], %5;"
      ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(bar) & kPeerBitMask),
      "r"(c0), "r"(c1), "l"(cache_hint)
      : "memory");
}
__device__ __forceinline__ void tmem_alloc_pair(uint32_t* smem_result, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(
                   smem_u32(smem_result)),
               "r"(ncols)
               : "memory");
}
__device__ __forceinline__ void tmem_relinquish_pair() {
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc_pair(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols)
               : "memory");
}
// Arrive on the barrier at this offset in both CTAs of the pair once the issued MMAs completed.
__device__ __forceinline__ void tc_commit_pair(uint64_t* bar) {
  asm volatile(
      "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
      ::"r"(smem_u32(bar)), "h"(static_cast<uint16_t>(3))
      : "memory");
}
__device__ __forceinline__ void tc_mma_f16_pair(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc,
                                                uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t"
      "}\n" ::"r"(d_tmem),
      "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}

// kind::f8f6f4: 8-bit float operands (K = 32 elements = 32 bytes per instruction), fp32 accumulation.
// In its instruction descriptor the A / B format 0 is E4M3 (make_idesc(0, m, n)).
__device__ __forceinline__ void tc_mma_f8(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc,
                                          uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f8f6f4 [%0], %1, %2, %3, p;\n\t"
      "}\n" ::"r"(d_tmem),
      "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void tc_mma_f8_pair(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc,
                                               uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f8f6f4 [%0], %1, %2, %3, p;\n\t"
      "}\n" ::"r"(d_tmem),
      "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}

// Two fp32 -> two E4M3 bytes (round to nearest even, saturating to +-448): `lo` goes to the lower
// address of the returned little-endian pair.
__device__ __forceinline__ uint16_t cvt_e4m3x2(float lo, float hi) {
  uint16_t r;
  asm("cvt.rn.satfinite.e4m3x2.f32 %0, %1, %2;" : "=h"(r) : "f"(hi), "f"(lo));
  return r;
}

// A operand in tensor memory ("TS" form): D[tmem] (+)= A[tmem] * B[smem].  A is M x K with row m on
// TMEM lane m and two consecutive 16-bit K elements per 32-bit column (K = 16 -> 8 columns).
__device__ __forceinline__ void tc_mma_f16_pair_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc,
                                                   uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], [%1], %2, %3, p;\n\t"
      "}\n" ::"r"(d_tmem),
      "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// registers -> TMEM: 32 lanes x 4 consecutive 32-bit columns (one row per thread)
__device__ __forceinline__ void tmem_st_32x4(uint32_t taddr, const uint32_t (&r)[4]) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x4.b32 [%0], {%1, %2, %3, %4};" ::"r"(taddr), "r"(r[0]), "r"(r[1]),
               "r"(r[2]), "r"(r[3])
               : "memory");
}
__device__ __forceinline__ void tc_wait_st() {
  asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
}

// Shared-memory matrix descriptor for a K-major operand tile stored as rows of 128 bytes with the
// 128-byte swizzle (exactly what a SWIZZLE_128B TMA box of 128-byte inner extent produces).
// Eight rows form one 1024-byte swizzle atom; atoms are stacked along M/N (SBO = 1024 bytes).
__device__ __forceinline__ uint64_t make_kmajor_sw128_desc(uint32_t smem_addr) {
  uint64_t desc = 0;
  desc |= static_cast<uint64_t>((smem_addr & 0x3FFFF) >> 4);  // start address, 16-byte units
  desc |= static_cast<uint64_t>(1) << 16;                      // LBO (unused with swizzle)
  desc |= static_cast<uint64_t>(1024 >> 4) << 32;              // SBO: 8 rows * 128 B
  desc |= static_cast<uint64_t>(1) << 46;                      // descriptor version (sm_100)
  desc |= static_cast<uint64_t>(2) << 61;                      // SWIZZLE_128B
  return desc;
}

// Instruction descriptor for tcgen05.mma kind::f16 / kind::tf32 / kind::f8f6f4, dense, fp32
// accumulate, both operands K-major.  ab_format: 0 = f16, 1 = bf16, 2 = tf32; under kind::f8f6f4
// 0 = e4m3.
__host__ __device__ constexpr uint32_t make_idesc(uint32_t ab_format, uint32_t m, uint32_t n) {
  return (1u << 4) |                // D format: f32
         (ab_format << 7) |         // A format
         (ab_format << 10) |        // B format
         (0u << 15) | (0u << 16) |  // A, B major: K
         ((n >> 3) << 17) |         // N >> 3
         ((m >> 4) << 24);          // M >> 4
}

// TMEM -> registers: 32 lanes x 32 consecutive 32-bit columns (one row per thread).
__device__ __forceinline__ void tmem_ld_32x32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]),
        "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]),
        "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]),
        "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]),
        "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
}

// TMEM -> registers: 32 lanes x 16 consecutive 32-bit columns.
__device__ __forceinline__ void tmem_ld_32x16(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]),
        "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]),
        "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
}

// tcgen05.wait::ld that also names the 32 destination registers of the load it completes, so that no
// use of them can be scheduled above the wait (needed once loads are software-pipelined and the wait
// no longer follows its load directly).
__device__ __forceinline__ void tc_wait_ld_regs(uint32_t (&r)[32]) {
  asm volatile("tcgen05.wait::ld.sync.aligned;"
               : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7]),
                 "+r"(r[8]), "+r"(r[9]), "+r"(r[10]), "+r"(r[11]), "+r"(r[12]), "+r"(r[13]), "+r"(r[14]),
                 "+r"(r[15]), "+r"(r[16]), "+r"(r[17]), "+r"(r[18]), "+r"(r[19]), "+r"(r[20]), "+r"(r[21]),
                 "+r"(r[22]), "+r"(r[23]), "+r"(r[24]), "+r"(r[25]), "+r"(r[26]), "+r"(r[27]), "+r"(r[28]),
                 "+r"(r[29]), "+r"(r[30]), "+r"(r[31])
               :
               : "memory");
}

__device__ __forceinline__ void tc_wait_ld_regs16(uint32_t (&r)[16]) {
  asm volatile("tcgen05.wait::ld.sync.aligned;"
               : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7]),
                 "+r"(r[8]), "+r"(r[9]), "+r"(r[10]), "+r"(r[11]), "+r"(r[12]), "+r"(r[13]), "+r"(r[14]), "+r"(r[15])
               :
               : "memory");
}

// Packed fp32 multiply (FMUL2 on sm_100): (a0, a1) *= (w0, w1), each lane rounded to nearest like FMUL.
__device__ __forceinline__ void mul_f32x2(uint32_t& a0, uint32_t& a1, float w0, float w1) {
  uint64_t a, w, d;
  asm("mov.b64 %0, {%1, %2};" : "=l"(a) : "r"(a0), "r"(a1));
  asm("mov.b64 %0, {%1, %2};" : "=l"(w) : "f"(w0), "f"(w1));
  asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(w));
  asm("mov.b64 {%0, %1}, %2;" : "=r"(a0), "=r"(a1) : "l"(d));
}

// ----------------------------------------------------------------------------
// Warp-cooperative bitonic sort of 32*E (score, index) pairs, element i = e*32 + lane.
// Order: score descending, then index ascending (the oracle's tie-break).  NaN never wins.
// ----------------------------------------------------------------------------
__device__ __forceinline__ bool pair_before(float sa, int ia, float sb, int ib) {
  // true if (sa, ia) must come before (sb, ib)
  return (sa > sb) || (sa == sb && ia < ib);
}

template <int E>
__device__ __forceinline__ void warp_sort_desc(float (&s)[E], int (&idx)[E]) {
  const uint32_t lane = lane_id();
  constexpr int TOTAL = 32 * E;
#pragma unroll
  for (int k = 2; k <= TOTAL; k <<= 1) {
#pragma unroll
    for (int j = k >> 1; j > 0; j >>= 1) {
      if (j >= 32) {
        // partner lives in the same lane, register e ^ (j / 32)
        const int je = j >> 5;
#pragma unroll
        for (int e = 0; e < E; ++e) {
          const int pe = e ^ je;
          if (pe > e) {
            const int i = e * 32;  // bit positions >= 5 come from e only
            const bool desc_block = ((i & k) == 0);
            // element e has the lower index of the pair
            const bool lower_first = pair_before(s[e], idx[e], s[pe], idx[pe]);
            const bool swap = desc_block ? !lower_first : lower_first;
            if (swap) {
              float ts = s[e]; s[e] = s[pe]; s[pe] = ts;
              int ti = idx[e]; idx[e] = idx[pe]; idx[pe] = ti;
            }
          }
        }
      } else {
#pragma unroll
        for (int e = 0; e < E; ++e) {
          const int i = e * 32 + static_cast<int>(lane);
          const float os = __shfl_xor_sync(kFullMask, s[e], j);
          const int oi = __shfl_xor_sync(kFullMask, idx[e], j);
          const bool desc_block = ((i & k) == 0);
          const bool i_am_lower = ((lane & j) == 0);
          // In a descending block the lower position keeps the element that sorts first.
          const bool mine_first = pair_before(s[e], idx[e], os, oi);
          const bool keep_mine = (desc_block == i_am_lower) ? mine_first : !mine_first;
          if (!keep_mine) { s[e] = os; idx[e] = oi; }
        }
      }
    }
  }
}

// Final phase of the same network: sorts a BITONIC input (slots [0, T/2) descending, slots [T/2, T)
// ascending, in the pair order above) with log2(T) compare-exchange steps instead of the full sort's
// log2(T) (log2(T) + 1) / 2.  Used to merge two sorted lists.
template <int E>
__device__ __forceinline__ void warp_merge_desc(float (&s)[E], int (&idx)[E]) {
  const uint32_t lane = lane_id();
  constexpr int TOTAL = 32 * E;
#pragma unroll
  for (int j = TOTAL >> 1; j > 0; j >>= 1) {
    if (j >= 32) {
      const int je = j >> 5;
#pragma unroll
      for (int e = 0; e < E; ++e) {
        const int pe = e ^ je;
        if (pe > e) {
          if (!pair_before(s[e], idx[e], s[pe], idx[pe])) {
            float ts = s[e]; s[e] = s[pe]; s[pe] = ts;
            int ti = idx[e]; idx[e] = idx[pe]; idx[pe] = ti;
          }
        }
      }
    } else {
#pragma unroll
      for (int e = 0; e < E; ++e) {
        const float os = __shfl_xor_sync(kFullMask, s[e], j);
        const int oi = __shfl_xor_sync(kFullMask, idx[e], j);
        const bool i_am_lower = ((lane & j) == 0);
        const bool mine_first = pair_before(s[e], idx[e], os, oi);
        const bool keep_mine = i_am_lower ? mine_first : !mine_first;
        if (!keep_mine) { s[e] = os; idx[e] = oi; }
      }
    }
  }
}

}  // namespace isx
#endif  // __CUDACC__
