// alz_sort.cu — key/value radix sort, prefix scan, unique of sorted keys and the sum of sorted row blocks by
// key, used once per window flush (canonical edge order, overlapping-rank merge, GNN node list and CSR build)
// and once per rollup over the window history. Off the per-event hot path; uses the CUDA toolkit's CUB device
// primitives.
#include <algorithm>
#include <cstddef>
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

// sum of sorted row blocks by key: keys of the live rows, sort, unique, one summed row per key
namespace {
constexpr uint32_t kSumWord = offsetof(alz_edge_out, count) / 8;   // words [kSumWord, kHistWord): u64 sums
constexpr uint32_t kHistWord = offsetof(alz_edge_out, hist) / 8;   // words from kHistWord on: two u32 cells each
static_assert(offsetof(alz_edge_out, lat_sum_ns) + 8 == offsetof(alz_edge_out, hist) && kHistWord * 8 ==
              offsetof(alz_edge_out, hist), "alz_edge_out layout");

__device__ __forceinline__ uint32_t lower_bound_u64(const uint64_t* __restrict__ a, uint32_t n, uint64_t k) {
  uint32_t lo = 0, hi = n;
  while (lo < hi) { const uint32_t mid = (lo + hi) >> 1; if (a[mid] < k) lo = mid + 1; else hi = mid; }
  return lo;
}

// packed key and row index of every live row, in block order. The whole grid walks one block after the other, so
// any number of blocks needs no shared memory and no search.
__global__ void __launch_bounds__(256) live_row_keys_kernel(RowBlocks b, uint64_t* __restrict__ keys,
                                                            uint32_t* __restrict__ rows) {
  const uint32_t stride = gridDim.x * blockDim.x;
  uint32_t off = 0;
  for (uint32_t q = 0; q < b.n; ++q) {
    const uint32_t head = ((b.first + q) % b.ring) * b.stride;
    const uint32_t cnt = reinterpret_cast<const BlockHeader*>(b.base + head)->count;
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < cnt; i += stride) {
      const uint32_t row = head + 1 + i;
      keys[off + i] = row_key_of(b.base + row);
      rows[off + i] = row;
    }
    off += cnt;
  }
}

__device__ __forceinline__ uint64_t add_cells(uint64_t a, uint64_t b) {   // two u32 histogram cells, each modulo 2^32
  return (uint64_t)((uint32_t)a + (uint32_t)b) | ((uint64_t)((uint32_t)(a >> 32) + (uint32_t)(b >> 32)) << 32);
}

// out[u] = the sum of the rows whose key is ukeys[u]; keys/rows: all live rows, sorted by key. The type and id words
// come from the run's first row. count, err5xx and lat_sum add modulo 2^64 and each histogram cell modulo 2^32: the
// bits an element-wise integer sum over the rows gives. Eight lanes per output row.
__global__ void __launch_bounds__(256) sum_runs_kernel(const alz_edge_out* __restrict__ base,
                                                       const uint64_t* __restrict__ keys,
                                                       const uint32_t* __restrict__ rows, uint32_t n,
                                                       const uint64_t* __restrict__ ukeys,
                                                       const uint32_t* __restrict__ n_unique,
                                                       alz_edge_out* __restrict__ out) {
  const uint32_t nu = *n_unique;
  const uint32_t sl = threadIdx.x & 7u;
  const uint32_t groups = (gridDim.x * blockDim.x) >> 3;
  for (uint32_t u = (blockIdx.x * blockDim.x + threadIdx.x) >> 3; u < nu; u += groups) {
    const uint64_t key = ukeys[u];
    const uint32_t first = lower_bound_u64(keys, n, key);
    uint64_t* d64 = reinterpret_cast<uint64_t*>(out + u);
    for (uint32_t w = sl; w < kRowWords64; w += 8u) {
      uint64_t v = reinterpret_cast<const uint64_t*>(base + rows[first])[w];
      for (uint32_t j = first + 1; w >= kSumWord && j < n && keys[j] == key; ++j) {
        const uint64_t x = reinterpret_cast<const uint64_t*>(base + rows[j])[w];
        v = w < kHistWord ? v + x : add_cells(v, x);
      }
      d64[w] = v;
    }
  }
}
}  // namespace

size_t sum_blocks_temp_bytes(uint32_t n_rows) { return std::max(sort_pairs_temp_bytes(n_rows), scan_temp_bytes(n_rows)); }

// keys: [0, n) the rows' keys, then the distinct keys; [n, 2n) sorted. idx: row indices, sorted row indices, head
// flags, unique positions.
void sum_blocks_by_key(const RowBlocks& b, uint32_t n_rows, uint64_t* keys, uint32_t* idx, void* temp,
                       size_t temp_bytes, alz_edge_out* out, uint32_t* n_unique, int sms, cudaStream_t s) {
  const unsigned grid = (unsigned)sms * 4;
  const size_t n = n_rows;
  uint64_t* sorted = keys + n;
  uint32_t* rows = idx;
  uint32_t* rows_sorted = idx + n;
  live_row_keys_kernel<<<grid, 256, 0, s>>>(b, keys, rows);
  sort_pairs(temp, temp_bytes, keys, sorted, rows, rows_sorted, n_rows, s);
  unique_sorted_u64(temp, temp_bytes, sorted, n_rows, idx + 2 * n, idx + 3 * n, keys, n_unique, sms, s);
  sum_runs_kernel<<<grid, 256, 0, s>>>(b.base, sorted, rows_sorted, n_rows, keys, n_unique, out);
}
}  // namespace alz
