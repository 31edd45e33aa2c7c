// alz_comm.cu — multi-GPU window merge (SURVEY.md §8e): one rank per GPU, events
// pre-partitioned by alz_owner_rank(saddr), tables replicated. Every event of an edge
// reaches one rank, so the ranks' edge sets are disjoint and a rank's accumulators are
// already final: what the flush has to do is hand every rank every other rank's rows.
//
// Default path — ONE collective, no host round trip before it:
//   1. each rank writes its sorted live rows behind a one-row header {count, status} in a
//      send buffer; the per-rank block size of the collective comes from the previous
//      window's counts (+25 %), so no count exchange is needed
//   2. ncclAllGather of the blocks                      <- the single exchange step
//   3. every rank merges the R sorted, disjoint lists: a row's place in the canonical
//      (ascending packed key) order is its index in its own list plus its lower bounds
//      in the other lists. The same kernel notices a key present on two ranks, a rank
//      whose rows did not fit its block, or a rank that reported a local error — all
//      ranks see the same headers, so all ranks take the same decision.
//   4. one device->host read of {total, flags}: the only synchronisation, and the one the
//      API needs anyway to return the edge count.
// A block that was too small (traffic grew by more than 25 % in one window) is sent
// again, larger; the local rows are only reset after a successful merge.
//
// General path (a key present on several ranks: the caller did not partition by
// alz_owner_rank): canonical dictionary by all-gather + sort + unique, local rows
// scattered into a zeroed canonical array, ONE ncclAllReduce(sum) on the accumulators.
// Integer sums either way, so bit-exact for any rank count.
//
// NCCL is loaded lazily with dlopen so that single-GPU users (and the Go agent
// on a box without NCCL) never need libnccl.so.2.
#include <dlfcn.h>
#include <nccl.h>

#include <algorithm>
#include <cstdio>
#include <cstring>
#include <mutex>
#include <string>

#include "alz_handle.h"

using namespace alz;

namespace {

struct NcclApi {
  void* lib = nullptr;
  ncclResult_t (*GetUniqueId)(ncclUniqueId*) = nullptr;
  ncclResult_t (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int) = nullptr;
  ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
  ncclResult_t (*AllGather)(const void*, void*, size_t, ncclDataType_t, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*AllReduce)(const void*, void*, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t) = nullptr;
  const char* (*GetErrorString)(ncclResult_t) = nullptr;
};
NcclApi g_nccl;

bool load_nccl_once() {
  void* lib = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
  if (!lib) lib = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
  if (!lib) return false;
#define SYM(field, name)                                             \
  g_nccl.field = reinterpret_cast<decltype(g_nccl.field)>(dlsym(lib, name)); \
  if (!g_nccl.field) return false;
  SYM(GetUniqueId, "ncclGetUniqueId");
  SYM(CommInitRank, "ncclCommInitRank");
  SYM(CommDestroy, "ncclCommDestroy");
  SYM(AllGather, "ncclAllGather");
  SYM(AllReduce, "ncclAllReduce");
  SYM(GetErrorString, "ncclGetErrorString");
#undef SYM
  g_nccl.lib = lib;
  return true;
}
// several rank threads of one process may get here together (tests/test_gpu_multi.py)
bool load_nccl() {
  static std::once_flag once;
  static bool ok = false;
  std::call_once(once, [] { ok = load_nccl_once(); });
  return ok;
}

constexpr int kCanWords = 3 + ALZ_NB;      // u64 words per canonical edge row of the general path: count, err5xx,
                                           // lat_sum and one word per histogram cell (a cell is u32 modulo 2^32: the
                                           // low halves of the sums are taken, nothing can carry between cells)
constexpr uint32_t kRowBytes = sizeof(alz_edge_out);   // 296 = 37 x 8
constexpr uint32_t kRowWords64 = kRowBytes / 8;
constexpr uint32_t kHdrMagic = 0xA1A2C0DEu;
struct BlockHeader {      // first row of a rank's block
  uint32_t magic, count;
  int32_t status;
  uint32_t pad;
};
struct MergeInfo {        // written by the merge kernel, read by the host
  uint32_t total, dup, overflow, max_count;
  int32_t peer_status;
  uint32_t pad[3];
};

// out[i] = keys[i] for i < n, kEmptyKey padding up to n_pad
__global__ void pad_keys_kernel(const uint64_t* __restrict__ keys, uint32_t n, uint64_t* __restrict__ out,
                                uint32_t n_pad) {
  const uint32_t stride = gridDim.x * blockDim.x;
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n_pad; i += stride)
    out[i] = i < n ? keys[i] : kEmptyKey;
}

// unique of the sorted gathered keys: flag run heads, exclusive-scan the flags, scatter the heads
__global__ void flag_heads_kernel(const uint64_t* __restrict__ sorted, uint32_t n, uint32_t* __restrict__ flags) {
  const uint32_t stride = gridDim.x * blockDim.x;
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
    const uint64_t k = sorted[i];
    flags[i] = (k != kEmptyKey && (i == 0 || sorted[i - 1] != k)) ? 1u : 0u;
  }
}
__global__ void scatter_heads_kernel(const uint64_t* __restrict__ sorted, const uint32_t* __restrict__ flags,
                                     const uint32_t* __restrict__ pos, uint32_t n, uint64_t* __restrict__ out) {
  const uint32_t stride = gridDim.x * blockDim.x;
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride)
    if (flags[i]) out[pos[i]] = sorted[i];
}

__device__ __forceinline__ uint32_t lower_bound_u64(const uint64_t* __restrict__ a, uint32_t n, uint64_t k) {
  uint32_t lo = 0, hi = n;
  while (lo < hi) { const uint32_t mid = (lo + hi) >> 1; if (a[mid] < k) lo = mid + 1; else hi = mid; }
  return lo;
}

// union of R sorted, pairwise disjoint key lists (segment r = gathered[r * pad .. + counts[r])):
// out[sum of lower bounds] = key. *dup is set if a key occurs in two lists.
__global__ void __launch_bounds__(256) merge_disjoint_kernel(const uint64_t* __restrict__ gathered, uint32_t pad,
                                                             uint32_t R, const uint32_t* __restrict__ counts,
                                                             uint64_t* __restrict__ out, uint32_t* __restrict__ dup) {
  const uint32_t stride = gridDim.x * blockDim.x;
  for (uint32_t t = blockIdx.x * blockDim.x + threadIdx.x; t < pad * R; t += stride) {
    const uint32_t r = t / pad, i = t - r * pad;
    if (i >= counts[r]) continue;
    const uint64_t k = gathered[t];
    uint32_t pos = i;
    for (uint32_t q = 0; q < R; ++q) {
      if (q == r) continue;
      const uint64_t* seg = gathered + (size_t)q * pad;
      const uint32_t lb = lower_bound_u64(seg, counts[q], k);
      if (lb < counts[q] && seg[lb] == k) *dup = 1u;
      pos += lb;
    }
    out[pos] = k;
  }
}

// local live rows -> canonical array (zeroed beforehand); a warp per local edge; rows are zeroed
__global__ void __launch_bounds__(256) scatter_canonical_kernel(AccTable edges, const uint64_t* __restrict__ keys,
                                                                const uint32_t* __restrict__ rows, uint32_t n_local,
                                                                const uint64_t* __restrict__ can_keys, uint32_t n_can,
                                                                uint64_t* __restrict__ can) {
  const uint32_t lane = threadIdx.x & 31u;
  const uint32_t warps_per_grid = (gridDim.x * blockDim.x) >> 5;
  for (uint32_t i = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; i < n_local; i += warps_per_grid) {
    const uint32_t row = rows[i];
    const uint32_t pos = lower_bound_u64(can_keys, n_can, keys[i]);   // always present
    uint64_t* dst = can + (size_t)pos * kCanWords;
    dst[3 + lane] = edges.hist[(size_t)row * ALZ_NB + lane];
    dst[3 + 32 + lane] = edges.hist[(size_t)row * ALZ_NB + 32 + lane];
    edges.hist[(size_t)row * ALZ_NB + lane] = 0u;
    edges.hist[(size_t)row * ALZ_NB + 32 + lane] = 0u;
    if (lane == 0) {
      dst[0] = edges.count[row]; dst[1] = edges.err5xx[row]; dst[2] = edges.lat_sum[row];
      edges.count[row] = 0ull; edges.err5xx[row] = 0ull; edges.lat_sum[row] = 0ull;
    }
  }
}

__global__ void __launch_bounds__(256) unpack_canonical_kernel(const uint64_t* __restrict__ can_keys,
                                                               const uint64_t* __restrict__ can, uint32_t n_can,
                                                               alz_edge_out* __restrict__ out) {
  const uint32_t lane = threadIdx.x & 31u;
  const uint32_t warps_per_grid = (gridDim.x * blockDim.x) >> 5;
  for (uint32_t i = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; i < n_can; i += warps_per_grid) {
    const uint64_t* src = can + (size_t)i * kCanWords;
    alz_edge_out* o = &out[i];
    o->hist[lane] = (uint32_t)src[3 + lane];
    o->hist[32 + lane] = (uint32_t)src[3 + 32 + lane];
    if (lane == 0) {
      uint8_t ft, tt; uint32_t f, t;
      unpack_edge_key(can_keys[i], &ft, &f, &tt, &t);
      o->from_type = ft; o->to_type = tt;
      for (int k = 0; k < 6; ++k) o->_pad[k] = 0;
      o->from = f; o->to = t;
      o->count = src[0]; o->err5xx = src[1]; o->lat_sum_ns = src[2];
    }
  }
}

// packed edge key of an output row (inverse of unpack_edge_key)
__device__ __forceinline__ uint64_t row_key_of(const alz_edge_out* r) {
  // rows are 296 bytes apart: 8-byte aligned only
  const uint2 ty = reinterpret_cast<const uint2*>(r)[0];   // from_type, to_type, pad | pad
  const uint2 ft_ = reinterpret_cast<const uint2*>(r)[1];  // from | to
  const uint32_t ft = ty.x & 0xFFu, tt = (ty.x >> 8) & 0xFFu;
  if (ft == ALZ_NODE_POD) return ((uint64_t)tt << 61) | ((uint64_t)(ft_.x & 0x1FFFFFFFu) << 32) | ft_.y;
  return (1ull << 63) | ((uint64_t)ft << 61) | ((uint64_t)(ft_.y & 0x1FFFFFFFu) << 32) | ft_.x;
}
__device__ __forceinline__ uint32_t lower_bound_rows(const alz_edge_out* rows, uint32_t n, uint64_t k, bool* equal) {
  uint32_t lo = 0, hi = n;
  while (lo < hi) { const uint32_t mid = (lo + hi) >> 1; if (row_key_of(rows + mid) < k) lo = mid + 1; else hi = mid; }
  *equal = lo < n && row_key_of(rows + lo) == k;
  return lo;
}

// Merge of the gathered blocks: block q = header row + cap rows, of which header.count are live and sorted.
// Eight lanes per row: the lanes split the other ranks' binary searches among them, then copy the row.
__global__ void __launch_bounds__(256) merge_blocks_kernel(const alz_edge_out* __restrict__ recv, uint32_t cap, uint32_t R,
                                                           alz_edge_out* __restrict__ out, uint32_t out_cap,
                                                           MergeInfo* __restrict__ info) {
  __shared__ uint32_t s_cnt[64];
  __shared__ uint32_t s_bad;
  const size_t stride_rows = (size_t)cap + 1;
  if (threadIdx.x == 0) s_bad = 0u;
  __syncthreads();
  if (threadIdx.x < R) {
    const BlockHeader* hd = reinterpret_cast<const BlockHeader*>(recv + threadIdx.x * stride_rows);
    uint32_t cnt = hd->count;
    if (hd->magic != kHdrMagic || hd->status != ALZ_OK) {
      atomicOr(&s_bad, 1u);
      if (blockIdx.x == 0) info->peer_status = hd->magic != kHdrMagic ? (int32_t)ALZ_E_STATE : hd->status;
      cnt = 0;
    }
    if (cnt > cap) { atomicOr(&s_bad, 2u); if (blockIdx.x == 0) { info->overflow = 1u; atomicMax(&info->max_count, cnt); } }
    if (blockIdx.x == 0) atomicMax(&info->max_count, cnt);
    s_cnt[threadIdx.x] = cnt;
  }
  __syncthreads();
  uint32_t total = 0;
  for (uint32_t q = 0; q < R; ++q) total += s_cnt[q];
  if (blockIdx.x == 0 && threadIdx.x == 0) info->total = total;
  if (s_bad != 0u || total > out_cap) { if (blockIdx.x == 0 && threadIdx.x == 0 && total > out_cap) info->overflow = 2u; return; }
  const uint32_t sl = threadIdx.x & 7u;
  const uint32_t groups = (gridDim.x * blockDim.x) >> 3;
  const uint32_t n_iter = (total + groups - 1) / groups;
  uint32_t g = (blockIdx.x * blockDim.x + threadIdx.x) >> 3;
  for (uint32_t it = 0; it < n_iter; ++it, g += groups) {
    const bool valid = g < total;
    // (q, i) of flat index g
    uint32_t q = 0, i = valid ? g : 0u;
    while (valid && i >= s_cnt[q]) { i -= s_cnt[q]; ++q; }
    const alz_edge_out* src = recv + q * stride_rows + 1 + i;
    const uint64_t key = valid ? row_key_of(src) : 0ull;
    uint32_t part = 0;
    bool dup = false;
    for (uint32_t p = sl; p < R; p += 8u) {
      if (!valid || p == q) continue;
      bool eq;
      part += lower_bound_rows(recv + p * stride_rows + 1, s_cnt[p], key, &eq);
      dup |= eq;
    }
    part += __shfl_xor_sync(0xFFFFFFFFu, part, 1);
    part += __shfl_xor_sync(0xFFFFFFFFu, part, 2);
    part += __shfl_xor_sync(0xFFFFFFFFu, part, 4);
    if (dup) info->dup = 1u;
    if (!valid) continue;
    const uint64_t* s64 = reinterpret_cast<const uint64_t*>(src);
    uint64_t* d64 = reinterpret_cast<uint64_t*>(out + (i + part));
    for (uint32_t w = sl; w < kRowWords64; w += 8u) d64[w] = s64[w];
  }
}

// a successful merge consumes the window: zero the local edge rows that were sent, empty the edge dictionary, reset
// the row allocator. Decided on the device from the merge kernel's verdict, so the host reads that verdict once, at
// the end, instead of synchronising in the middle of the flush to decide whether to launch this.
__global__ void __launch_bounds__(256) consume_window_kernel(const MergeInfo* __restrict__ info, AccTable edges,
                                                             const uint32_t* __restrict__ rows, uint32_t n) {
  if (info->peer_status != ALZ_OK || info->overflow != 0u || info->dup != 0u) return;
  const uint32_t sl = threadIdx.x & 7u;
  const uint32_t groups = (gridDim.x * blockDim.x) >> 3;
  const size_t dict_words = ((size_t)edges.dict_mask + 1u) * (sizeof(DictEnt) / 16u);
  uint4* dict = reinterpret_cast<uint4*>(edges.dict);
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < dict_words; i += (size_t)gridDim.x * blockDim.x)
    dict[i] = make_uint4(0xFFFFFFFFu, 0xFFFFFFFFu, 0xFFFFFFFFu, 0xFFFFFFFFu);
  if (blockIdx.x == 0 && threadIdx.x == 0) *edges.n_rows = 0u;
  for (uint32_t i = (blockIdx.x * blockDim.x + threadIdx.x) >> 3; i < n; i += groups) {
    const uint32_t row = rows[i];
    uint4* cells = reinterpret_cast<uint4*>(edges.hist + (size_t)row * ALZ_NB + sl * 8u);
    cells[0] = make_uint4(0u, 0u, 0u, 0u);
    cells[1] = make_uint4(0u, 0u, 0u, 0u);
    if (sl == 0) { edges.count[row] = 0ull; edges.err5xx[row] = 0ull; edges.lat_sum[row] = 0ull; }
  }
}

}  // namespace

struct alz_comm_state {
  ~alz_comm_state() { if (comm && g_nccl.CommDestroy) g_nccl.CommDestroy(comm); }   // before the buffers below go
  Owned mem;
  ncclComm_t comm = nullptr;
  uint32_t* d_counts = nullptr;   // [nranks]
  uint32_t* h_counts = nullptr;   // pinned
  uint64_t* d_gather = nullptr;   // [nranks * pad] gathered keys, then sorted copy behind it
  uint64_t* d_sorted = nullptr;
  uint32_t* d_flags = nullptr;
  uint32_t* d_pos = nullptr;
  uint64_t* d_can_keys = nullptr; // [max_edges]
  uint64_t* d_can = nullptr;      // [max_edges * kCanWords]
  uint32_t* d_iota = nullptr;
  uint32_t* d_vals = nullptr;
  void* d_tmp = nullptr;
  size_t tmp_bytes = 0;
  size_t gather_cap = 0;          // keys
  // default path
  alz_edge_out* d_send = nullptr; // [1 + block_rows_for(max_edges)]: header row + local sorted rows (+ head room)
  GrowBuf<alz_edge_out> d_recv;   // [R * (1 + cap_r)]
  uint32_t cap_r = 0;             // rows per rank block of the next collective (0 = not known yet)
  BlockHeader* h_hdr = nullptr;   // pinned
  MergeInfo* d_info = nullptr;
  MergeInfo* h_info = nullptr;    // pinned
};
void StateDelete::operator()(alz_comm_state* c) const { delete c; }

#define NK(expr)                                                                       \
  do {                                                                                 \
    const ncclResult_t _r = (expr);                                                    \
    if (_r != ncclSuccess) return alz_error(h, ALZ_E_NCCL, #expr, g_nccl.GetErrorString(_r)); \
  } while (0)

extern "C" int alz_comm_unique_id(void* out_id) {
  if (!out_id) return ALZ_E_INVAL;
  if (!load_nccl()) return ALZ_E_NCCL;
  static_assert(sizeof(ncclUniqueId) <= ALZ_COMM_ID_BYTES, "ncclUniqueId larger than ALZ_COMM_ID_BYTES");
  ncclUniqueId id;
  if (g_nccl.GetUniqueId(&id) != ncclSuccess) return ALZ_E_NCCL;
  memset(out_id, 0, ALZ_COMM_ID_BYTES);
  memcpy(out_id, &id, sizeof(id));
  return ALZ_OK;
}

static uint32_t block_rows_for(uint64_t max_count) {   // +25 % head room, in steps of 1024 rows
  const uint64_t want = max_count + max_count / 4 + 1024;
  return (uint32_t)((want + 1023) / 1024 * 1024);
}

extern "C" int alz_comm_init(alz_handle* h, int nranks, int rank, const void* id_bytes) {
  if (!h || !id_bytes || nranks < 1 || rank < 0 || rank >= nranks) return ALZ_E_INVAL;
  std::lock_guard<std::mutex> g(h->mu);
  if (h->comm) return ALZ_E_STATE;
  if (!load_nccl()) return alz_error(h, ALZ_E_NCCL, nullptr, "dlopen(libnccl.so.2) failed");
  CK(cudaSetDevice(h->device));
  // built here and published only when complete: a failure leaves the handle single-rank, and the caller may retry
  StatePtr<alz_comm_state> c(new alz_comm_state());
  ncclUniqueId id;
  memcpy(&id, id_bytes, sizeof(id));
  ncclComm_t comm = nullptr;
  NK(g_nccl.CommInitRank(&comm, nranks, id, rank));
  c->comm = comm;
  const size_t me = h->cfg.max_edges;
  c->gather_cap = me;  // every rank holds the merged graph, so max_edges bounds the gathered keys too
  Owned& m = c->mem;
  CK(m.dev(&c->d_counts, sizeof(uint32_t) * nranks));
  CK(m.pinned(&c->h_counts, sizeof(uint32_t) * nranks));
  CK(m.dev(&c->d_gather, me * 8 * 2));
  c->d_sorted = c->d_gather + me;
  CK(m.dev(&c->d_flags, me * 4));
  CK(m.dev(&c->d_pos, me * 4));
  CK(m.dev(&c->d_can_keys, me * 8));
  CK(m.dev(&c->d_can, me * kCanWords * 8));
  CK(m.dev(&c->d_iota, me * 4));
  CK(m.dev(&c->d_vals, me * 4));
  c->tmp_bytes = std::max(sort_pairs_temp_bytes((uint32_t)me), scan_temp_bytes((uint32_t)me));
  CK(m.dev(&c->d_tmp, c->tmp_bytes));
  // a block is sized from the largest rank's count plus head room: up to block_rows_for(max_edges) rows are SENT
  // from here even when this rank has fewer (max_edges must be the same on every rank)
  const size_t send_rows = (size_t)block_rows_for(me) + 1;
  CK(m.dev(&c->d_send, send_rows * sizeof(alz_edge_out)));
  CK(cudaMemset(c->d_send, 0, send_rows * sizeof(alz_edge_out)));
  CK(m.pinned(&c->h_hdr, sizeof(alz_edge_out)));
  CK(m.dev(&c->d_info, sizeof(MergeInfo)));
  CK(m.pinned(&c->h_info, sizeof(MergeInfo)));
  h->comm = std::move(c);
  h->comm_nranks = nranks;
  h->comm_rank = rank;
  return ALZ_OK;
}

// General path: keys may live on several ranks. Local live edges are sorted in d_keys[1] / d_rows[1].
static int merge_allreduce(alz_handle* h) {
  alz_comm_state* c = h->comm.get();
  const int R = h->comm_nranks;
  cudaStream_t s = h->stream;
  const unsigned grid = (unsigned)h->sms * 4;

  // 1. counts
  CK(cudaMemcpyAsync(c->d_counts + h->comm_rank, &h->n_live, 4, cudaMemcpyHostToDevice, s));
  NK(g_nccl.AllGather(c->d_counts + h->comm_rank, c->d_counts, 1, ncclUint32, c->comm, s));
  CK(cudaMemcpyAsync(c->h_counts, c->d_counts, 4 * R, cudaMemcpyDeviceToHost, s));
  CK(cudaStreamSynchronize(s));
  uint32_t pad = 0;
  uint64_t total = 0;
  for (int r = 0; r < R; ++r) { pad = std::max(pad, c->h_counts[r]); total += c->h_counts[r]; }
  if (total == 0) {
    h->last_n_edges = 0;
    h->windows++;
    CK(cudaMemsetAsync(h->edges.dict, 0xFF, ((size_t)h->edges.dict_mask + 1) * sizeof(DictEnt), s));
    CK(cudaMemsetAsync(h->edges.n_rows, 0, 4, s));
    return ALZ_OK;
  }
  if ((uint64_t)pad * R > c->gather_cap) return ALZ_E_CAPACITY;
  const uint32_t n_g = pad * (uint32_t)R;

  // 2. keys: pad, all-gather, merge. Each rank's list is sorted and, when the caller partitioned by
  //    alz_owner_rank, the lists are disjoint: a key's place in the union is then the sum of its lower
  //    bounds in the R lists - no sort. A key found on two ranks (caller routed one source to two ranks)
  //    raises a flag and the general path (sort + unique) runs instead; the sums are right either way.
  pad_keys_kernel<<<grid, 256, 0, s>>>(h->d_keys[1], h->n_live, c->d_sorted, pad);
  NK(g_nccl.AllGather(c->d_sorted, c->d_gather, pad, ncclUint64, c->comm, s));
  CK(cudaMemsetAsync(c->d_flags, 0, 4, s));
  merge_disjoint_kernel<<<grid, 256, 0, s>>>(c->d_gather, pad, (uint32_t)R, c->d_counts, c->d_can_keys, c->d_flags);
  uint32_t dup = 0;
  CK(cudaMemcpyAsync(&dup, c->d_flags, 4, cudaMemcpyDeviceToHost, s));
  CK(cudaStreamSynchronize(s));
  uint32_t n_can = (uint32_t)total;
  if (dup) {
    launch_iota(c->d_iota, n_g, h->sms, s);
    sort_pairs(c->d_tmp, c->tmp_bytes, c->d_gather, c->d_sorted, c->d_iota, c->d_vals, n_g, s);
    flag_heads_kernel<<<grid, 256, 0, s>>>(c->d_sorted, n_g, c->d_flags);
    exclusive_scan_u32(c->d_tmp, c->tmp_bytes, c->d_flags, c->d_pos, n_g, s);
    scatter_heads_kernel<<<grid, 256, 0, s>>>(c->d_sorted, c->d_flags, c->d_pos, n_g, c->d_can_keys);
    uint32_t last[2];
    CK(cudaMemcpyAsync(&last[0], c->d_pos + (n_g - 1), 4, cudaMemcpyDeviceToHost, s));
    CK(cudaMemcpyAsync(&last[1], c->d_flags + (n_g - 1), 4, cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    n_can = last[0] + last[1];
  }
  if (n_can > h->cfg.max_edges) return ALZ_E_CAPACITY;

  // 3. scatter local rows into the zeroed canonical array
  const size_t can_bytes = (size_t)n_can * kCanWords * 8;
  CK(cudaMemsetAsync(c->d_can, 0, can_bytes, s));
  if (h->n_live)
    scatter_canonical_kernel<<<grid * 2, 256, 0, s>>>(h->edges, h->d_keys[1], h->d_rows[1], h->n_live,
                                                      c->d_can_keys, n_can, c->d_can);
  // 4. the single exchange step
  NK(g_nccl.AllReduce(c->d_can, c->d_can, (size_t)n_can * kCanWords, ncclUint64, ncclSum, c->comm, s));
  h->collective_bytes_last += can_bytes;
  h->launches += 5;
  // 5. unpack; local edge table back to empty
  unpack_canonical_kernel<<<grid * 2, 256, 0, s>>>(c->d_can_keys, c->d_can, n_can, h->d_out);
  CK(cudaGetLastError());
  CK(cudaMemsetAsync(h->edges.dict, 0xFF, ((size_t)h->edges.dict_mask + 1) * sizeof(DictEnt), s));
  CK(cudaMemsetAsync(h->edges.n_rows, 0, 4, s));
  h->last_n_edges = n_can;
  h->windows++;
  return ALZ_OK;
}

// Called by the flush after prepare_flush(): local live edges are sorted in d_keys[1] (keys) / d_rows[1]
// (rows), h->n_live of them; local_rc is this rank's status so far. Every rank enters the collective whatever
// its own status, so nobody is left waiting in NCCL, and all ranks return the same failure.
int alz_internal_merge_ranks(alz_handle* h, int local_rc) {
  alz_comm_state* c = h->comm.get();
  if (!c || h->comm_nranks <= 1) return ALZ_E_UNSUPPORTED;
  const int R = h->comm_nranks;
  if (R > 64) return ALZ_E_UNSUPPORTED;
  cudaStream_t s = h->stream;
  const unsigned grid = (unsigned)h->sms * 4;
  const uint32_t n_local = local_rc == ALZ_OK ? h->n_live : 0u;
  h->collective_bytes_last = 0;

  if (c->cap_r == 0) {   // first window: nothing to size the blocks from, exchange the counts once
    CK(cudaMemcpyAsync(c->d_counts + h->comm_rank, &n_local, 4, cudaMemcpyHostToDevice, s));
    NK(g_nccl.AllGather(c->d_counts + h->comm_rank, c->d_counts, 1, ncclUint32, c->comm, s));
    CK(cudaMemcpyAsync(c->h_counts, c->d_counts, 4 * R, cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    uint32_t mx = 0;
    for (int r = 0; r < R; ++r) mx = std::max(mx, c->h_counts[r]);
    c->cap_r = block_rows_for(mx);
  }
  // local rows behind the header, in canonical order; the window is NOT reset yet
  if (n_local) {
    launch_gather_edges(h->edges, h->d_keys[1], h->d_rows[1], n_local, c->d_send + 1, false, h->sms, s);
    h->launches += 1;
  }
  for (int attempt = 0; attempt < 4; ++attempt) {
    memset(c->h_hdr, 0, sizeof(alz_edge_out));
    c->h_hdr->magic = kHdrMagic; c->h_hdr->count = n_local; c->h_hdr->status = local_rc;
    CK(cudaMemcpyAsync(c->d_send, c->h_hdr, sizeof(alz_edge_out), cudaMemcpyHostToDevice, s));
    const size_t block_rows = (size_t)c->cap_r + 1;
    CK(c->d_recv.ensure(block_rows * R, s));
    CK(cudaMemsetAsync(c->d_info, 0, sizeof(MergeInfo), s));
    // the single exchange step: every rank's header + its first cap_r rows
    NK(g_nccl.AllGather(c->d_send, c->d_recv.get(), block_rows * kRowWords64, ncclUint64, c->comm, s));
    h->collective_bytes_last += (uint64_t)block_rows * R * kRowBytes;
    merge_blocks_kernel<<<grid, 256, 0, s>>>(c->d_recv.get(), c->cap_r, (uint32_t)R, h->d_out, h->cfg.max_edges, c->d_info);
    consume_window_kernel<<<grid, 256, 0, s>>>(c->d_info, h->edges, h->d_rows[1], n_local);
    h->launches += 2;
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(c->h_info, c->d_info, sizeof(MergeInfo), cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));   // the flush's one synchronisation: the caller needs the edge count
    const MergeInfo inf = *c->h_info;
    if (inf.peer_status != ALZ_OK) return local_rc != ALZ_OK ? local_rc : inf.peer_status;   // the window stays intact
    if (inf.overflow == 1u) { c->cap_r = block_rows_for(inf.max_count); continue; }   // every rank sees the same headers
    if (inf.overflow == 2u) return ALZ_E_CAPACITY;                                    // merged graph larger than max_edges
    c->cap_r = block_rows_for(inf.max_count);                                         // next window's block size
    if (inf.dup) return merge_allreduce(h);                                           // not partitioned by owner: general path
    // success: consume_window_kernel has consumed the window
    h->last_n_edges = inf.total;
    h->windows++;
    return ALZ_OK;
  }
  return ALZ_E_CAPACITY;
}
