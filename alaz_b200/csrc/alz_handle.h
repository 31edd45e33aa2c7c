// alz_handle.h — the handle behind the C ABI: everything one GPU owns.
#pragma once
#include <algorithm>
#include <cstdint>
#include <memory>
#include <mutex>
#include <string>
#include <unordered_map>
#include <vector>
#include <cuda_runtime.h>

#include "../../include/alazgpu.h"
#include "../../include/alazgpu_synth.h"
#include "alz_kernels.cuh"

struct alz_handle;

// ---- errors ------------------------------------------------------------------------------------------
// Records "what: why" as the handle's last error and returns rc. The only writer of last_err: it takes
// err_mu, because submitting threads may fail at the same time.
int alz_error(alz_handle* h, int rc, const char* what, const char* why);

#define CK(expr)                                                                       \
  do {                                                                                 \
    const cudaError_t _e = (expr);                                                     \
    if (_e != cudaSuccess) return alz_error(h, ALZ_E_CUDA, #expr, cudaGetErrorString(_e)); \
  } while (0)

// ---- ownership ---------------------------------------------------------------------------------------
// What the library takes from CUDA is held by owners. The structs handed to kernels by value (AccTable,
// HotState, Counters, alz_synth_view, ...) keep raw pointers; the memory behind them belongs to an owner
// beside them. An owner is destroyed only while its handle's device is current: one process may drive
// several GPUs from several threads.
enum class Res { kDev, kPinned, kEvent, kStream };
struct ResFree {
  Res kind = Res::kDev;
  void operator()(void* p) const {
    switch (kind) {
      case Res::kDev: cudaFree(p); break;
      case Res::kPinned: cudaFreeHost(p); break;
      case Res::kEvent: cudaEventDestroy(static_cast<cudaEvent_t>(p)); break;
      case Res::kStream: cudaStreamDestroy(static_cast<cudaStream_t>(p)); break;
    }
  }
};
using Owner = std::unique_ptr<void, ResFree>;

// cudaMalloc / cudaMallocHost into o; o is left untouched on failure
inline cudaError_t alz_alloc(Owner& o, Res kind, size_t bytes) {
  void* p = nullptr;
  const cudaError_t e = kind == Res::kPinned ? cudaMallocHost(&p, bytes) : cudaMalloc(&p, bytes);
  if (e == cudaSuccess) o = Owner(p, ResFree{kind});
  return e;
}

// A buffer of T that grows on demand (device or pinned)
template <class T>
struct GrowBuf {
  explicit GrowBuf(Res kind = Res::kDev) : p(nullptr, ResFree{kind}) {}
  T* get() const { return static_cast<T*>(p.get()); }
  // at least n elements; a growth allocates max(n, grow) of them. Work in flight on `stream` may still use the
  // old buffer, so it waits for the stream before freeing it; cap changes only once the allocation succeeded.
  cudaError_t ensure(size_t n, cudaStream_t stream, size_t grow = 0) {
    if (n <= cap) return cudaSuccess;
    if (p) {
      const cudaError_t e = cudaStreamSynchronize(stream);
      if (e != cudaSuccess) return e;
      p.reset();
      cap = 0;
    }
    const size_t want = std::max(n, grow);
    const cudaError_t e = alz_alloc(p, p.get_deleter().kind, want * sizeof(T));
    if (e == cudaSuccess) cap = want;
    return e;
  }
  Owner p;
  size_t cap = 0;   // elements
};

// Everything a state allocated once, for its whole life. Released in reverse order of allocation, so a
// handle's streams (created first) outlive its buffers and events.
struct Owned {
  ~Owned() { while (!items.empty()) items.pop_back(); }
  template <class T> cudaError_t dev(T** out, size_t bytes) { return add(Res::kDev, reinterpret_cast<void**>(out), bytes); }
  template <class T> cudaError_t pinned(T** out, size_t bytes) { return add(Res::kPinned, reinterpret_cast<void**>(out), bytes); }
  cudaError_t event(cudaEvent_t* out, unsigned flags) {
    cudaEvent_t e = nullptr;
    const cudaError_t r = cudaEventCreateWithFlags(&e, flags);
    if (r == cudaSuccess) { items.emplace_back(e, ResFree{Res::kEvent}); *out = e; }
    return r;
  }
  cudaError_t stream(cudaStream_t* out) {
    cudaStream_t s = nullptr;
    const cudaError_t r = cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking);
    if (r == cudaSuccess) { items.emplace_back(s, ResFree{Res::kStream}); *out = s; }
    return r;
  }

 private:
  cudaError_t add(Res kind, void** out, size_t bytes) {
    Owner o;
    const cudaError_t e = alz_alloc(o, kind, bytes);
    if (e == cudaSuccess) { *out = o.get(); items.push_back(std::move(o)); }
    return e;
  }
  std::vector<Owner> items;
};

struct HostEp {
  uint32_t state = 0;  // kEpPod | kEpSvc
  uint32_t pod = 0, svc = 0;
};

struct EpPatch { uint32_t slot, pad[3]; alz::EpEntry e; };
static_assert(sizeof(EpPatch) == 32, "EpPatch layout");

struct alz_gnn_state;   // alz_gnn.cu
struct alz_sock_state;  // alz_sock.cu
struct alz_comm_state;  // alz_comm.cu
struct StateDelete {    // each defined beside its state
  void operator()(alz_comm_state* c) const;
  void operator()(alz_gnn_state* g) const;
  void operator()(alz_sock_state* s) const;
};
template <class T> using StatePtr = std::unique_ptr<T, StateDelete>;

// One host->device staging slot: pinned host buffer + device buffer. A submitting thread owns the slot
// (mu) from the copy into the pinned buffer until its H2D and kernel are enqueued. The buffers are
// published together (h last), so a slot with h is whole.
struct StageSlot {
  std::mutex mu;
  Owner h, d;
  Owner d_aux;                            // raw path: compacted 32-B records
  cudaEvent_t copied = nullptr;           // H2D out of h done -> h may be rewritten
  cudaEvent_t consumed = nullptr;         // kernel that read d (and d_aux) done -> d may be rewritten
};
constexpr int kStageSlots = 4;
constexpr int kRawSlots = 2;

struct alz_handle {
  alz_config cfg{};
  int device = 0, sms = 0;
  // streams, events and the fixed buffers of alz_create / alz_window_clock. Declared before every other
  // owner, so destroyed after them: the streams go last.
  Owned mem;
  cudaStream_t own_stream = nullptr, stream = nullptr, copy_stream = nullptr;
  cudaEvent_t ev_count = nullptr;
  std::mutex err_mu;
  std::string last_err;                   // written only by alz_error

  // Serialises everything that enqueues on `stream` or touches the bookkeeping below. Submitting threads
  // take it only around their enqueue; flush / commit / stats hold it for the whole call.
  std::mutex mu;
  std::mutex turn_mu;                     // staging slot hand-out
  uint64_t stage_turn = 0, raw_turn = 0;
  StageSlot stage[kStageSlots];
  StageSlot raw[kRawSlots];

  // join build side: host mirror of the ClusterInfo maps and of the device's open-addressed table;
  // a commit patches only the slots that changed (alz_table_commit)
  std::unordered_map<uint32_t, HostEp> ep_host;
  std::vector<uint32_t> ep_dirty_ips;
  std::vector<alz::EpEntry> ep_tab;       // host mirror, ep_cap entries
  std::vector<uint8_t> ep_touched;        // per slot: changed since the last upload
  std::vector<uint32_t> ep_touched_list;
  alz::EpEntry* d_ep = nullptr;
  uint32_t ep_cap = 0;
  std::vector<uint8_t> bloom_cnt;         // per filter bit: how many pod addresses set it (saturating at 255)
  bool bloom_dirty = false;
  uint32_t* d_bloom = nullptr;            // ALZ_BLOOM_WORDS words
  uint32_t* h_bloom = nullptr;            // pinned staging
  GrowBuf<EpPatch> h_patch{Res::kPinned}; // (slot, entry) records of one commit
  GrowBuf<EpPatch> d_patch;
  cudaEvent_t ev_patch = nullptr;

  // accumulators
  alz::AccTable pairs{}, edges{};
  alz::Counters* d_ctr = nullptr;
  alz::Counters* h_ctr = nullptr;  // pinned
  alz::HotState* d_hot = nullptr;

  // flush scratch
  uint64_t* d_keys = nullptr;             // sorted live edge keys
  uint32_t* d_rows[2] = {nullptr, nullptr};
  void* d_sort_tmp = nullptr;
  size_t sort_tmp_bytes = 0;
  alz_edge_out* d_out = nullptr;
  uint32_t n_live = 0, last_n_edges = 0;
  uint64_t lost_reported = 0;             // capacity_events already reported by an earlier flush

  // time-cut windows (alz_window_clock)
  bool win_on = false;
  uint64_t win_off = 0;                   // first_user - first_kernel (mod 2^64)
  uint64_t* d_win = nullptr;              // device WinClock {lo, len, ready}
  alz_l7_rec* d_defer[2] = {nullptr, nullptr};   // records of later windows (ping-pong)
  uint32_t defer_cap = 0;
  int defer_cur = 0;

  uint64_t events_in = 0, pending_since_fold = 0, windows = 0;
  uint64_t launches = 0;                  // own kernels launched (stats)
  cudaEvent_t ev_t[3] = {nullptr, nullptr, nullptr};   // flush start / local part done / merge done (timing events)
  bool ev_t_valid = false;
  uint64_t collective_bytes_last = 0;
  uint64_t tcp_events_in = 0, tcp_localhost_dropped = 0;

  int comm_nranks = 1, comm_rank = 0;
  StatePtr<alz_comm_state> comm;          // optional state: published only when complete
  StatePtr<alz_gnn_state> gnn;
  StatePtr<alz_sock_state> sock;
};

int alz_internal_fold(alz_handle* h);
// device records -> the ingest kernel of the current mode; caller holds h->mu and has set the device
int alz_internal_ingest(alz_handle* h, const alz_l7_rec* d_recs, size_t n);
// multi-GPU merge of the prepared (sorted) live edges, for a handle with comm_nranks > 1.
// local_rc: this rank's own status so far (every rank enters the collective even when its local
// preparation failed, and all ranks return the same failure)
int alz_internal_merge_ranks(alz_handle* h, int local_rc);
