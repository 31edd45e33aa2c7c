// alz_comm.cu — multi-GPU window merge (SURVEY.md §8e): one rank per GPU, events
// pre-partitioned by alz_owner_rank(saddr), tables replicated. Every event of an edge
// reaches one rank, so the ranks' edge sets are disjoint and a rank's accumulators are
// already final: what the flush has to do is hand every rank every other rank's rows.
//
// ONE collective, no host round trip before it:
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
// Overlapping ranks (a key present on several ranks: the caller did not partition by
// alz_owner_rank): after the all-gather every rank holds every rank's complete rows, the
// same bytes on every rank, so each rank merges them locally with no further exchange:
// sort the live rows by key, then one row per distinct key with the sums of its rows.
// Integer sums either way, so bit-exact for any rank count.
//
// NCCL is loaded lazily with dlopen so that single-GPU users (and the Go agent
// on a box without NCCL) never need libnccl.so.2.
#include <dlfcn.h>
#include <nccl.h>

#include <algorithm>
#include <cstddef>
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

constexpr uint32_t kMaxRanks = 64;                     // merge_blocks_kernel keeps one count per rank in shared memory
constexpr uint32_t kRowBytes = sizeof(alz_edge_out);   // 296 = 37 x 8
struct MergeInfo {        // written by the merge kernels, read by the host
  uint32_t total, dup, overflow, max_count;
  int32_t peer_status;
  uint32_t n_unique;      // overlapping ranks: rows after the merge
  uint32_t pad[2];
};

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
  __shared__ uint32_t s_cnt[kMaxRanks];
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

// a merge without a failed peer or an overflow consumes the window: zero the local edge rows that were sent, empty
// the edge dictionary, reset the row allocator. Decided on the device from the merge kernel's verdict, so the host
// reads that verdict once, at the end, instead of synchronising in the middle of the flush to decide whether to
// launch this. Overlapping ranks are merged from the gathered blocks alone, so they consume the window too.
__global__ void __launch_bounds__(256) consume_window_kernel(const MergeInfo* __restrict__ info, AccTable edges,
                                                             const uint32_t* __restrict__ rows, uint32_t n) {
  if (info->peer_status != ALZ_OK || info->overflow != 0u) return;
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
  uint32_t* d_counts = nullptr;   // [nranks]: the first window's count exchange
  uint32_t* h_counts = nullptr;   // pinned
  alz_edge_out* d_send = nullptr; // [1 + block_rows_for(max_edges)]: header row + local sorted rows (+ head room)
  GrowBuf<alz_edge_out> d_recv;   // [R * (1 + cap_r)]
  uint32_t cap_r = 0;             // rows per rank block of the next collective (0 = not known yet)
  BlockHeader* h_hdr = nullptr;   // pinned
  MergeInfo* d_info = nullptr;
  MergeInfo* h_info = nullptr;    // pinned
  // overlapping ranks only, grown on first use (n = live rows of all blocks): sum_blocks_by_key's scratch
  GrowBuf<uint64_t> ov_keys;
  GrowBuf<uint32_t> ov_idx;
  GrowBuf<uint8_t> ov_tmp;
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

// the merge verdict on the device and its pinned copy
static int alloc_info(alz_handle* h, alz_comm_state* c) {
  CK(c->mem.dev(&c->d_info, sizeof(MergeInfo)));
  CK(c->mem.pinned(&c->h_info, sizeof(MergeInfo)));
  return ALZ_OK;
}

extern "C" int alz_comm_init(alz_handle* h, int nranks, int rank, const void* id_bytes) {
  if (!h || !id_bytes || nranks < 1 || rank < 0 || rank >= nranks) return ALZ_E_INVAL;
  if (nranks > (int)kMaxRanks) return ALZ_E_UNSUPPORTED;
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
  Owned& m = c->mem;
  CK(m.dev(&c->d_counts, sizeof(uint32_t) * nranks));
  CK(m.pinned(&c->h_counts, sizeof(uint32_t) * nranks));
  // a block is sized from the largest rank's count plus head room: up to block_rows_for(max_edges) rows are SENT
  // from here even when this rank has fewer (max_edges must be the same on every rank)
  const size_t send_rows = (size_t)block_rows_for(h->cfg.max_edges) + 1;
  CK(m.dev(&c->d_send, send_rows * sizeof(alz_edge_out)));
  CK(cudaMemset(c->d_send, 0, send_rows * sizeof(alz_edge_out)));
  CK(m.pinned(&c->h_hdr, sizeof(alz_edge_out)));
  const int rc = alloc_info(h, c.get());
  if (rc != ALZ_OK) return rc;
  h->comm = std::move(c);
  h->comm_nranks = nranks;
  h->comm_rank = rank;
  return ALZ_OK;
}

// Overlapping ranks: all n live rows of the R gathered blocks, sorted by key, summed per key into h->d_out.
// *n_unique: rows written, read back in this path's one synchronisation.
static int merge_overlap(alz_handle* h, alz_comm_state* c, const alz_edge_out* recv, uint32_t cap, uint32_t R,
                         uint32_t n, uint32_t* n_unique) {
  cudaStream_t s = h->stream;
  const size_t tmp_bytes = sum_blocks_temp_bytes(n);
  CK(c->ov_keys.ensure(2 * (size_t)n, s));
  CK(c->ov_idx.ensure(4 * (size_t)n, s));
  CK(c->ov_tmp.ensure(tmp_bytes, s));
  sum_blocks_by_key(RowBlocks{recv, cap + 1, 0, R, R}, n, c->ov_keys.get(), c->ov_idx.get(), c->ov_tmp.get(),
                    tmp_bytes, h->d_out, &c->d_info->n_unique, h->sms, s);
  h->launches += 5;
  CK(cudaGetLastError());
  CK(cudaMemcpyAsync(&c->h_info->n_unique, &c->d_info->n_unique, 4, cudaMemcpyDeviceToHost, s));
  CK(cudaStreamSynchronize(s));
  *n_unique = c->h_info->n_unique;
  return ALZ_OK;
}

// What the flush runs after the all-gather: merge the R blocks of recv (header row + cap rows each) into h->d_out
// and read the verdict back into *inf. consume: also reset the local window (n_local rows in h->d_rows[1]) unless a
// peer failed or something overflowed; the caller handles those. Otherwise the window is complete: overlapping
// blocks go through merge_overlap, and last_n_edges is set.
static int merge_gathered(alz_handle* h, alz_comm_state* c, const alz_edge_out* recv, uint32_t cap, uint32_t R,
                          bool consume, uint32_t n_local, MergeInfo* inf) {
  cudaStream_t s = h->stream;
  const unsigned grid = (unsigned)h->sms * 4;
  CK(cudaMemsetAsync(c->d_info, 0, sizeof(MergeInfo), s));
  merge_blocks_kernel<<<grid, 256, 0, s>>>(recv, cap, R, h->d_out, h->cfg.max_edges, c->d_info);
  h->launches += 1;
  if (consume) {
    consume_window_kernel<<<grid, 256, 0, s>>>(c->d_info, h->edges, h->d_rows[1], n_local);
    h->launches += 1;
  }
  CK(cudaGetLastError());
  CK(cudaMemcpyAsync(c->h_info, c->d_info, sizeof(MergeInfo), cudaMemcpyDeviceToHost, s));
  CK(cudaStreamSynchronize(s));   // the flush's one synchronisation: the caller needs the edge count
  *inf = *c->h_info;
  if (inf->peer_status != ALZ_OK || inf->overflow != 0u) return ALZ_OK;
  uint32_t n = inf->total;
  if (inf->dup) {                 // not partitioned by owner
    const int rc = merge_overlap(h, c, recv, cap, R, inf->total, &n);
    if (rc != ALZ_OK) return rc;
  }
  h->last_n_edges = n;
  h->windows++;
  return ALZ_OK;
}

// Called by the flush after prepare_flush(): local live edges are sorted in d_keys (keys) / d_rows[1]
// (rows), h->n_live of them; local_rc is this rank's status so far. Every rank enters the collective whatever
// its own status, so nobody is left waiting in NCCL, and all ranks return the same failure.
int alz_internal_merge_ranks(alz_handle* h, int local_rc) {
  alz_comm_state* c = h->comm.get();
  const int R = h->comm_nranks;
  cudaStream_t s = h->stream;
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
    launch_gather_edges(h->edges, h->d_keys, h->d_rows[1], n_local, c->d_send + 1, false, h->sms, s);
    h->launches += 1;
  }
  for (int attempt = 0; attempt < 4; ++attempt) {
    memset(c->h_hdr, 0, sizeof(alz_edge_out));
    c->h_hdr->magic = kHdrMagic; c->h_hdr->count = n_local; c->h_hdr->status = local_rc;
    CK(cudaMemcpyAsync(c->d_send, c->h_hdr, sizeof(alz_edge_out), cudaMemcpyHostToDevice, s));
    const size_t block_rows = (size_t)c->cap_r + 1;
    CK(c->d_recv.ensure(block_rows * R, s));
    // the single exchange step: every rank's header + its first cap_r rows
    NK(g_nccl.AllGather(c->d_send, c->d_recv.get(), block_rows * kRowWords64, ncclUint64, c->comm, s));
    h->collective_bytes_last += (uint64_t)block_rows * R * kRowBytes;
    MergeInfo inf;
    const int rc = merge_gathered(h, c, c->d_recv.get(), c->cap_r, (uint32_t)R, true, n_local, &inf);
    if (rc != ALZ_OK) return rc;
    if (inf.peer_status != ALZ_OK) return local_rc != ALZ_OK ? local_rc : inf.peer_status;   // the window stays intact
    if (inf.overflow == 1u) { c->cap_r = block_rows_for(inf.max_count); continue; }   // every rank sees the same headers
    if (inf.overflow == 2u) return ALZ_E_CAPACITY;                                    // merged graph larger than max_edges
    c->cap_r = block_rows_for(inf.max_count);                                         // next window's block size
    return alz_internal_history_append(h);
  }
  return ALZ_E_CAPACITY;
}

// test entry (alazgpu_synth.h): merge_gathered on blocks the caller gathered, with a verdict of this call's own
extern "C" int alz_merge_blocks_device(alz_handle* h, const alz_edge_out* dev_blocks, uint32_t nranks,
                                       uint32_t block_rows, const alz_edge_out** dev_out, size_t* n_out) {
  if (!h || !dev_blocks || nranks < 1 || !n_out) return ALZ_E_INVAL;
  if (nranks > kMaxRanks) return ALZ_E_UNSUPPORTED;
  std::lock_guard<std::mutex> g(h->mu);
  CK(cudaSetDevice(h->device));
  *n_out = 0;
  StatePtr<alz_comm_state> c(new alz_comm_state());
  int rc = alloc_info(h, c.get());
  MergeInfo inf;
  if (rc == ALZ_OK) rc = merge_gathered(h, c.get(), dev_blocks, block_rows, nranks, false, 0, &inf);
  if (rc != ALZ_OK) return rc;
  if (inf.peer_status != ALZ_OK) return inf.peer_status;
  if (inf.overflow != 0u) return ALZ_E_CAPACITY;
  *n_out = h->last_n_edges;
  if (dev_out) *dev_out = h->d_out;
  return ALZ_OK;
}
