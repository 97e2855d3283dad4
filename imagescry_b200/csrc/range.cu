// Ordering pass of the range search (isx_knn_range): the search kernel appends its hits as unordered
// 12-byte records {query, global row, fp32 score bits}; this pass turns them into CSR, every query's
// hits ordered by (score desc, row asc) like the k-NN search's lists.
//
//   range_hist_kernel     per-query hit counts (records with row < 0 are padding and are skipped)
//   cub::DeviceScan       exclusive sum of the counts -> offsets[q + 1]
//   range_scatter_kernel  every record into its query's segment as one 64-bit key
//                         (~orderable(score) << 32) | (row << 1) | (score is -0), whose ascending order is
//                         (score desc, row asc)
//   cub::DeviceSegmentedSort  one radix sort per query segment
//   range_decode_kernel   keys -> rows, scores
#include "common.cuh"

#include <cub/device/device_scan.cuh>
#include <cub/device/device_segmented_sort.cuh>

namespace isx {
namespace {

// Monotonic float -> uint32 map.  -0 is ordered as +0 (the k-NN search compares scores as floats);
// its sign travels in the key's lowest bit instead, so the decoded score keeps its bits.
__device__ __forceinline__ uint32_t score_order(float f) {
  const uint32_t b = __float_as_uint(f == 0.f ? 0.f : f);
  return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}

__device__ __forceinline__ float score_from_order(uint32_t u) {
  return __uint_as_float((u & 0x80000000u) ? (u & 0x7FFFFFFFu) : ~u);
}

// (~order(score) << 32) | (row << 1) | (score is -0): ascending keys are (score desc, row asc); rows
// are < 2^31, so row << 1 fits the low word
__device__ __forceinline__ unsigned long long range_key(float score, int row) {
  const uint32_t neg_zero = __float_as_uint(score) == 0x80000000u ? 1u : 0u;
  return (static_cast<unsigned long long>(~score_order(score)) << 32) | (static_cast<uint32_t>(row) << 1) | neg_zero;
}

__device__ __forceinline__ bool range_record_valid(const int3& r, int q) { return r.y >= 0 && r.x >= 0 && r.x < q; }

// record i of the N x 3 buffer; 64-bit index: 3 * i exceeds int32 for i > 715 827 882
__device__ __forceinline__ int3 range_record(const int32_t* records, long long i) {
  const int32_t* r = records + 3 * i;
  return make_int3(r[0], r[1], r[2]);
}

__global__ void __launch_bounds__(256)
range_hist_kernel(const int32_t* __restrict__ records, long long total, int q, unsigned long long* __restrict__ counts) {
  const long long stride = static_cast<long long>(gridDim.x) * blockDim.x;
  for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < total; i += stride) {
    const int3 r = range_record(records, i);
    if (range_record_valid(r, q)) atomicAdd(counts + r.x, 1ull);
  }
}

__global__ void __launch_bounds__(256)
range_scatter_kernel(const int32_t* __restrict__ records, long long total, int q, const long long* __restrict__ offsets,
                     unsigned long long* __restrict__ cursor, unsigned long long* __restrict__ keys) {
  const long long stride = static_cast<long long>(gridDim.x) * blockDim.x;
  for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < total; i += stride) {
    const int3 r = range_record(records, i);
    if (!range_record_valid(r, q)) continue;
    const unsigned long long pos = static_cast<unsigned long long>(offsets[r.x]) + atomicAdd(cursor + r.x, 1ull);
    keys[pos] = range_key(__int_as_float(r.z), r.y);
  }
}

__global__ void __launch_bounds__(256)
range_decode_kernel(const unsigned long long* __restrict__ keys, const long long* __restrict__ end, long long total,
                    int32_t* __restrict__ rows, float* __restrict__ scores) {
  const long long m = min(*end, total);
  const long long stride = static_cast<long long>(gridDim.x) * blockDim.x;
  for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < m; i += stride) {
    const unsigned long long key = keys[i];
    const uint32_t lo = static_cast<uint32_t>(key & 0xFFFFFFFFull);
    rows[i] = static_cast<int32_t>(lo >> 1);
    scores[i] = (lo & 1u) ? -0.f : score_from_order(~static_cast<uint32_t>(key >> 32));
  }
}

size_t align256(size_t v) { return (v + 255) / 256 * 256; }

struct RangeSortWorkspace {
  size_t counts_off, keys_in_off, keys_out_off, temp_off, temp_bytes, total;
};

// counts[q + 1] (reused as the scatter cursors), keys in / out [total], CUB's temporary storage
int range_sort_workspace(int total, int q, RangeSortWorkspace* w) {
  size_t scan_bytes = 0, sort_bytes = 0;
  ISX_CHECK_CUDA(cub::DeviceScan::ExclusiveSum(nullptr, scan_bytes, static_cast<unsigned long long*>(nullptr),
                                               static_cast<long long*>(nullptr), q + 1));
  ISX_CHECK_CUDA(cub::DeviceSegmentedSort::SortKeys(nullptr, sort_bytes, static_cast<const unsigned long long*>(nullptr),
                                                    static_cast<unsigned long long*>(nullptr), total, q,
                                                    static_cast<const long long*>(nullptr),
                                                    static_cast<const long long*>(nullptr)));
  size_t off = 0;
  w->counts_off = off;
  off = align256(off + (static_cast<size_t>(q) + 1) * sizeof(unsigned long long));
  w->keys_in_off = off;
  off = align256(off + static_cast<size_t>(total) * sizeof(unsigned long long));
  w->keys_out_off = off;
  off = align256(off + static_cast<size_t>(total) * sizeof(unsigned long long));
  w->temp_off = off;
  w->temp_bytes = std::max<size_t>(std::max(scan_bytes, sort_bytes), 1);
  w->total = off + w->temp_bytes + 256;  // + 256: the caller's pointer is aligned up
  return ISX_OK;
}

int grid_for(long long items, int sms) {
  return static_cast<int>(std::max<long long>(1, std::min<long long>((items + 255) / 256, static_cast<long long>(sms) * 8)));
}

}  // namespace
}  // namespace isx

using namespace isx;

extern "C" {

size_t isx_knn_range_sort_workspace_bytes(int64_t total, int q) {
  if (total < 0 || total >= (1ll << 31) || q <= 0) return 0;
  RangeSortWorkspace w;
  if (range_sort_workspace(static_cast<int>(total), q, &w) != ISX_OK) return 0;
  return w.total;
}

int isx_knn_range_sort(const int32_t* records, int64_t total, int q, int64_t* offsets, int32_t* rows, float* scores,
                       void* workspace, size_t workspace_bytes, isx_stream_t stream_) {
  const char* fn = "isx_knn_range_sort";
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  ISX_REQUIRE(q > 0 && total >= 0 && total < (1ll << 31), "%s: need q > 0 and 0 <= total < 2^31 (q=%d total=%lld)", fn,
              q, (long long)total);
  ISX_REQUIRE(offsets && (total == 0 || (records && rows && scores)), "%s: null pointer", fn);
  ISX_REQUIRE((reinterpret_cast<uintptr_t>(records) & 3u) == 0 && (reinterpret_cast<uintptr_t>(offsets) & 7u) == 0,
              "%s: records must be 4-byte and offsets 8-byte aligned", fn);
  if (total == 0) {
    ISX_CHECK_CUDA(cudaMemsetAsync(offsets, 0, (static_cast<size_t>(q) + 1) * sizeof(int64_t), stream));
    return ISX_OK;
  }
  const int n = static_cast<int>(total);
  RangeSortWorkspace w;
  int rc = range_sort_workspace(n, q, &w);
  if (rc != ISX_OK) return rc;
  ISX_REQUIRE(workspace != nullptr && workspace_bytes >= w.total, "%s: workspace too small (%zu < %zu)", fn,
              workspace_bytes, w.total);
  uint8_t* base = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(workspace) + 255) & ~uintptr_t(255));
  auto* counts = reinterpret_cast<unsigned long long*>(base + w.counts_off);
  auto* keys_in = reinterpret_cast<unsigned long long*>(base + w.keys_in_off);
  auto* keys_out = reinterpret_cast<unsigned long long*>(base + w.keys_out_off);
  void* temp = base + w.temp_off;
  auto* off = reinterpret_cast<long long*>(offsets);
  int sms = 148;
  rc = device_sm_count(&sms);
  if (rc != ISX_OK) return rc;
  const int grid = grid_for(n, sms);
  const size_t count_bytes = (static_cast<size_t>(q) + 1) * sizeof(unsigned long long);

  ISX_CHECK_CUDA(cudaMemsetAsync(counts, 0, count_bytes, stream));
  range_hist_kernel<<<grid, 256, 0, stream>>>(records, n, q, counts);
  ISX_CHECK_CUDA(cudaGetLastError());
  size_t temp_bytes = w.temp_bytes;
  ISX_CHECK_CUDA(cub::DeviceScan::ExclusiveSum(temp, temp_bytes, counts, off, q + 1, stream));
  ISX_CHECK_CUDA(cudaMemsetAsync(counts, 0, count_bytes, stream));
  range_scatter_kernel<<<grid, 256, 0, stream>>>(records, n, q, off, counts, keys_in);
  ISX_CHECK_CUDA(cudaGetLastError());
  temp_bytes = w.temp_bytes;
  ISX_CHECK_CUDA(cub::DeviceSegmentedSort::SortKeys(temp, temp_bytes, keys_in, keys_out, n, q, off, off + 1, stream));
  range_decode_kernel<<<grid, 256, 0, stream>>>(keys_out, off + q, n, rows, scores);
  ISX_CHECK_CUDA(cudaGetLastError());
  return ISX_OK;
}

}  // extern "C"
