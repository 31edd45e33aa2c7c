// alz_history.cu — the edge rows of the last `depth` flushed windows, kept on the device, and their rollup over
// any k of them (docs/SPEC.md §12).
//
// The history is a ring of `depth` slots in the layout of the gathered blocks of a multi-rank flush: a header row
// with the count, then up to max_edges rows in ascending packed-key order. A flush that counts a window appends it
// with one device-to-device copy of its output rows; a rollup sums the newest k slots by key with the same kernels
// as the overlapping-rank merge (sum_blocks_by_key, alz_sort.cu), into buffers of its own, so the flush output, the
// GNN pass and the open window never see it. Every rank of a multi-rank handle appends the same merged rows, so a
// rollup needs no communication and gives the same bytes on every rank.
#include <algorithm>
#include <mutex>
#include <vector>

#include "alz_handle.h"

using namespace alz;

struct alz_history_state {
  Owned mem;
  uint32_t depth = 0;
  uint32_t stride = 0;              // rows per slot: max_edges + 1
  alz_edge_out* ring = nullptr;     // [depth * stride]
  BlockHeader* h_hdr = nullptr;     // pinned, one per slot: the source of the slot's header copy
  std::vector<uint32_t> counts;     // rows per slot, as in the device headers
  uint32_t next = 0, held = 0;      // slot of the next append; slots in use
  uint64_t newest = 0;              // alz_stats.windows ordinal of the newest slot
  uint32_t* d_n = nullptr;          // rollup: distinct keys, on the device
  uint32_t* h_n = nullptr;          // pinned
  // rollup scratch, grown to the rows of the windows summed
  GrowBuf<uint64_t> keys;
  GrowBuf<uint32_t> idx;
  GrowBuf<uint8_t> tmp;
  GrowBuf<alz_edge_out> out;
};
void StateDelete::operator()(alz_history_state* y) const { delete y; }

// an allocation that failed is reported as ALZ_E_NOMEM and is not left behind as the thread's last CUDA error, where
// the next kernel launch check of a flush would find it
#define CKM(expr)                                                                      \
  do {                                                                                 \
    const cudaError_t _e = (expr);                                                     \
    if (_e != cudaSuccess) {                                                           \
      cudaGetLastError();                                                              \
      return alz_error(h, _e == cudaErrorMemoryAllocation ? ALZ_E_NOMEM : ALZ_E_CUDA, #expr, cudaGetErrorString(_e)); \
    }                                                                                  \
  } while (0)

extern "C" int alz_history_init(alz_handle* h, uint32_t depth) {
  if (!h || depth == 0) return ALZ_E_INVAL;
  const uint64_t stride = (uint64_t)h->cfg.max_edges + 1;
  if ((uint64_t)depth * stride >= (1ull << 32)) return ALZ_E_INVAL;   // row indices of the sum kernels are u32
  std::lock_guard<std::mutex> g(h->mu);
  if (h->hist) return ALZ_E_STATE;
  CK(cudaSetDevice(h->device));
  // built here and published only when complete: a failure leaves the handle without history
  StatePtr<alz_history_state> y(new alz_history_state());
  y->depth = depth;
  y->stride = (uint32_t)stride;
  y->counts.assign(depth, 0u);
  Owned& m = y->mem;
  CKM(m.dev(&y->ring, (size_t)depth * stride * sizeof(alz_edge_out)));
  CKM(m.pinned(&y->h_hdr, (size_t)depth * sizeof(BlockHeader)));
  CKM(m.dev(&y->d_n, 4));
  CKM(m.pinned(&y->h_n, 4));
  h->hist = std::move(y);
  return ALZ_OK;
}

int alz_internal_history_append(alz_handle* h) {
  alz_history_state* y = h->hist.get();
  if (!y) return ALZ_OK;
  const uint32_t slot = y->next, n = h->last_n_edges;
  alz_edge_out* dst = y->ring + (size_t)slot * y->stride;
  // h_hdr[slot] is written again only `depth` appends later; every flush in between waits for the stream past
  // this copy before it appends
  y->h_hdr[slot] = BlockHeader{kHdrMagic, n, ALZ_OK, 0u};
  CK(cudaMemcpyAsync(dst, &y->h_hdr[slot], sizeof(BlockHeader), cudaMemcpyHostToDevice, h->stream));
  if (n) CK(cudaMemcpyAsync(dst + 1, h->d_out, (size_t)n * sizeof(alz_edge_out), cudaMemcpyDeviceToDevice, h->stream));
  y->counts[slot] = n;
  y->next = (slot + 1) % y->depth;
  y->held = std::min(y->held + 1, y->depth);
  y->newest = h->windows;
  return ALZ_OK;
}

extern "C" int alz_history_info(alz_handle* h, uint32_t* held, uint64_t* newest) {
  if (!h || !held || !newest) return ALZ_E_INVAL;
  std::lock_guard<std::mutex> g(h->mu);
  const alz_history_state* y = h->hist.get();
  if (!y) return ALZ_E_STATE;
  *held = y->held;
  *newest = y->newest;
  return ALZ_OK;
}

// the newest min(k, held) slots summed by key into y->out; *n_out: rows written (the call's one synchronisation)
static int rollup_locked(alz_handle* h, uint32_t k, size_t* n_out) {
  alz_history_state* y = h->hist.get();
  if (!y) return ALZ_E_STATE;
  CK(cudaSetDevice(h->device));
  const uint32_t m = std::min(k, y->held);
  const uint32_t first = (y->next + y->depth - m) % y->depth;   // oldest of the m slots
  uint64_t n_rows = 0;
  for (uint32_t q = 0; q < m; ++q) n_rows += y->counts[(first + q) % y->depth];
  if (n_rows == 0) return ALZ_OK;   // < depth * max_edges < 2^32 from here on
  cudaStream_t s = h->stream;
  const uint32_t n = (uint32_t)n_rows;
  const size_t tmp_bytes = sum_blocks_temp_bytes(n);
  CKM(y->keys.ensure(2 * n_rows, s));
  CKM(y->idx.ensure(4 * n_rows, s));
  CKM(y->tmp.ensure(tmp_bytes, s));
  CKM(y->out.ensure(n_rows, s));
  sum_blocks_by_key(RowBlocks{y->ring, y->stride, first, m, y->depth}, n, y->keys.get(), y->idx.get(), y->tmp.get(),
                    tmp_bytes, y->out.get(), y->d_n, h->sms, s);
  h->launches += 5;
  CK(cudaGetLastError());
  CK(cudaMemcpyAsync(y->h_n, y->d_n, 4, cudaMemcpyDeviceToHost, s));
  CK(cudaStreamSynchronize(s));
  *n_out = *y->h_n;
  return ALZ_OK;
}

extern "C" int alz_rollup_device(alz_handle* h, uint32_t k, const alz_edge_out** dev_edges, size_t* n_out) {
  if (!h || !n_out || k == 0) return ALZ_E_INVAL;
  std::lock_guard<std::mutex> g(h->mu);
  *n_out = 0;
  const int rc = rollup_locked(h, k, n_out);
  if (rc != ALZ_OK) return rc;
  if (dev_edges) *dev_edges = h->hist->out.get();
  return ALZ_OK;
}

extern "C" int alz_rollup(alz_handle* h, uint32_t k, alz_edge_out* out, size_t cap, size_t* n_out) {
  if (!h || !n_out || (!out && cap) || k == 0) return ALZ_E_INVAL;
  std::lock_guard<std::mutex> g(h->mu);
  *n_out = 0;
  const int rc = rollup_locked(h, k, n_out);
  if (rc != ALZ_OK) return rc;
  if (*n_out > cap) return ALZ_E_CAPACITY;
  if (*n_out) {
    CK(cudaMemcpyAsync(out, h->hist->out.get(), *n_out * sizeof(alz_edge_out), cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
  }
  return ALZ_OK;
}
