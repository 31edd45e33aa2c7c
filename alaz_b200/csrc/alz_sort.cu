// alz_sort.cu — key/value radix sort, prefix scan and unique of sorted keys, used once per window flush
// (canonical edge order, overlapping-rank merge, GNN node list and CSR build). Off the per-event
// hot path; uses the CUDA toolkit's CUB device primitives.
#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>
#include "alz_kernels.cuh"

namespace alz {
size_t sort_pairs_temp_bytes(uint32_t n) {
  size_t bytes = 0;
  cub::DeviceRadixSort::SortPairs(nullptr, bytes, (const uint64_t*)nullptr, (uint64_t*)nullptr,
                                  (const uint32_t*)nullptr, (uint32_t*)nullptr, (int)n);
  return bytes;
}
void sort_pairs(void* temp, size_t temp_bytes, const uint64_t* keys_in, uint64_t* keys_out,
                const uint32_t* vals_in, uint32_t* vals_out, uint32_t n, cudaStream_t s, int end_bit) {
  // end_bit: only key bits [0, end_bit) differ between keys (each 8 bits less is one pass over the data less)
  cub::DeviceRadixSort::SortPairs(temp, temp_bytes, keys_in, keys_out, vals_in, vals_out, (int)n, 0, end_bit, s);
}
size_t scan_temp_bytes(uint32_t n) {
  size_t bytes = 0;
  cub::DeviceScan::ExclusiveSum(nullptr, bytes, (const uint32_t*)nullptr, (uint32_t*)nullptr, (int)n);
  return bytes;
}
void exclusive_scan_u32(void* temp, size_t temp_bytes, const uint32_t* in, uint32_t* out, uint32_t n, cudaStream_t s) {
  cub::DeviceScan::ExclusiveSum(temp, temp_bytes, in, out, (int)n, s);
}

// unique of sorted keys: flag run heads, exclusive-scan the flags, scatter the heads, count
namespace {
__global__ void flag_heads_kernel(const uint64_t* __restrict__ sorted, uint32_t n, uint32_t* __restrict__ flags) {
  const uint32_t stride = gridDim.x * blockDim.x;
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride)
    flags[i] = (i == 0 || sorted[i - 1] != sorted[i]) ? 1u : 0u;
}
__global__ void scatter_heads_kernel(const uint64_t* __restrict__ sorted, const uint32_t* __restrict__ flags,
                                     const uint32_t* __restrict__ pos, uint32_t n, uint64_t* __restrict__ out) {
  const uint32_t stride = gridDim.x * blockDim.x;
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride)
    if (flags[i]) out[pos[i]] = sorted[i];
}
__global__ void unique_count_kernel(const uint32_t* __restrict__ pos, const uint32_t* __restrict__ flags, uint32_t n,
                                    uint32_t* __restrict__ n_unique) {
  if (threadIdx.x == 0 && blockIdx.x == 0) *n_unique = n ? pos[n - 1] + flags[n - 1] : 0u;
}
}  // namespace

void unique_sorted_u64(void* temp, size_t temp_bytes, const uint64_t* sorted, uint32_t n, uint32_t* flags,
                       uint32_t* pos, uint64_t* out, uint32_t* n_unique, int sms, cudaStream_t s) {
  const unsigned grid = (unsigned)sms * 4;
  flag_heads_kernel<<<grid, 256, 0, s>>>(sorted, n, flags);
  exclusive_scan_u32(temp, temp_bytes, flags, pos, n, s);
  scatter_heads_kernel<<<grid, 256, 0, s>>>(sorted, flags, pos, n, out);
  unique_count_kernel<<<1, 32, 0, s>>>(pos, flags, n, n_unique);
}
}  // namespace alz
