// alz_api.cu — the C ABI of libalazgpu (include/alazgpu.h): handle, HBM layout,
// host staging and the launch sequence of each entry point. Host side C++; the
// reference's Go caller reaches it through cgo (INTEGRATION.md).
//
// There is no CPU fallback anywhere in this file: without a CUDA device
// alz_create fails with ALZ_E_NODEVICE.
//
// Threading (SURVEY.md §8b; the reference calls this seam from 4*NumCPU goroutines,
// aggregator/data.go:230-232): alz_submit_* may be called from many OS threads. Each call
// takes a staging slot, copies into the slot's pinned buffer outside any shared lock, and
// holds h->mu only while it enqueues its H2D copy and kernel. Flush / commit / stats take
// h->mu for the whole call, so they are ordered after every submit that has returned.
#include <sched.h>

#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <new>
#include <string>
#include <unordered_map>
#include <vector>

#include "alz_handle.h"

using namespace alz;

int alz_error(alz_handle* h, int rc, const char* what, const char* why) {
  std::lock_guard<std::mutex> g(h->err_mu);
  h->last_err = what ? std::string(what) + ": " + why : std::string(why);
  return rc;
}

static uint32_t next_pow2(uint64_t x) {
  uint64_t p = 1;
  while (p < x) p <<= 1;
  return (uint32_t)std::min<uint64_t>(p, 1ull << 31);
}

// pinned buffers handed to callers (alz_pinned_alloc): submits from these skip
// the staging memcpy
static std::mutex g_pin_mu;
static std::vector<std::pair<const char*, size_t>> g_pinned;
static bool is_lib_pinned(const void* p, size_t bytes) {
  std::lock_guard<std::mutex> g(g_pin_mu);
  const char* c = (const char*)p;
  for (auto& r : g_pinned)
    if (c >= r.first && c + bytes <= r.first + r.second) return true;
  return false;
}

static int alloc_table(alz_handle* h, AccTable* t, uint32_t max_rows, uint32_t* n_rows_dev, bool pair_table) {
  memset(t, 0, sizeof(*t));
  t->max_rows = max_rows;
  t->n_rows = n_rows_dev;
  const uint32_t dict_cap = next_pow2(2ull * max_rows);
  t->dict_mask = dict_cap - 1;
  const size_t rows = (size_t)max_rows + kPairKinds;
  Owned& m = h->mem;
  CK(m.dev(&t->dict, (size_t)dict_cap * sizeof(DictEnt)));
  CK(m.dev(&t->row_key, rows * 8));
  if (!pair_table) {
    CK(m.dev(&t->lat_sum, rows * 8));
    CK(m.dev(&t->err5xx, rows * 8));
    CK(m.dev(&t->count, rows * 8));
    CK(m.dev(&t->hist, rows * ALZ_NB * 4));
    CK(cudaMemsetAsync(t->count, 0, rows * 8, h->stream));
    CK(cudaMemsetAsync(t->lat_sum, 0, rows * 8, h->stream));
    CK(cudaMemsetAsync(t->err5xx, 0, rows * 8, h->stream));
    CK(cudaMemsetAsync(t->hist, 0, rows * ALZ_NB * 4, h->stream));
  } else {
    CK(m.dev(&t->sect, rows * kSectPerRow * 32));
    CK(cudaMemsetAsync(t->sect, 0, rows * kSectPerRow * 32, h->stream));
    // reversed rows are a few per cent of the traffic: a quarter-size dictionary is ample, and both
    // dictionaries draw rows from the one pool
    const uint32_t rev_cap = std::max<uint32_t>(1024u, dict_cap >> 2);
    t->dict_rev_mask = rev_cap - 1;
    CK(m.dev(&t->dict_rev, (size_t)rev_cap * sizeof(DictEnt)));
    CK(cudaMemsetAsync(t->dict_rev, 0xFF, (size_t)rev_cap * sizeof(DictEnt), h->stream));
    const uint32_t host_cap = std::max<uint32_t>(1024u, dict_cap >> 3);   // host-keyed outbound pairs: rarer still
    t->dict_host_mask = host_cap - 1;
    CK(m.dev(&t->dict_host, (size_t)host_cap * sizeof(DictEnt)));
    CK(cudaMemsetAsync(t->dict_host, 0xFF, (size_t)host_cap * sizeof(DictEnt), h->stream));
    CK(m.dev(&t->row_kind, rows));
    CK(cudaMemsetAsync(t->row_kind, 0, rows, h->stream));
    CK(cudaMemsetAsync(t->row_kind + max_rows + kPairRev, (int)kPairRev, 1, h->stream));   // sentinel rows of the free-marker key
    CK(cudaMemsetAsync(t->row_kind + max_rows + kPairHost, (int)kPairHost, 1, h->stream));
    CK(m.dev(&t->row_cnt, rows * 4)); CK(cudaMemsetAsync(t->row_cnt, 0, rows * 4, h->stream));
    CK(m.dev(&t->row_base, rows)); CK(cudaMemsetAsync(t->row_base, 0, rows, h->stream));
    CK(m.dev(&t->row_aux, rows * 4));
  }
  CK(cudaMemsetAsync(t->dict, 0xFF, (size_t)dict_cap * sizeof(DictEnt), h->stream));
  return ALZ_OK;
}
// all keys out of the dictionaries, row allocator back to zero (rows were zeroed by fold / gather)
static int clear_dict(alz_handle* h, AccTable* t) {
  CK(cudaMemsetAsync(t->dict, 0xFF, ((size_t)t->dict_mask + 1) * sizeof(DictEnt), h->stream));
  if (t->dict_rev) CK(cudaMemsetAsync(t->dict_rev, 0xFF, ((size_t)t->dict_rev_mask + 1) * sizeof(DictEnt), h->stream));
  if (t->dict_host) CK(cudaMemsetAsync(t->dict_host, 0xFF, ((size_t)t->dict_host_mask + 1) * sizeof(DictEnt), h->stream));
  CK(cudaMemsetAsync(t->n_rows, 0, 4, h->stream));
  return ALZ_OK;
}

extern "C" const char* alz_strerror(int s) {
  switch (s) {
    case ALZ_OK: return "ok";
    case ALZ_E_INVAL: return "invalid argument";
    case ALZ_E_NOMEM: return "out of memory";
    case ALZ_E_CUDA: return "CUDA error";
    case ALZ_E_NODEVICE: return "no CUDA device (libalazgpu has no CPU fallback)";
    case ALZ_E_CAPACITY: return "capacity exceeded";
    case ALZ_E_STATE: return "invalid state";
    case ALZ_E_NCCL: return "NCCL error";
    case ALZ_E_UNSUPPORTED: return "unsupported";
    default: return "unknown status";
  }
}

// a copy taken under the lock: another thread may record a new error while the caller reads this one
extern "C" const char* alz_last_cuda_error(alz_handle* h) {
  if (!h) return "";
  thread_local std::string copy;
  std::lock_guard<std::mutex> g(h->err_mu);
  copy = h->last_err;
  return copy.c_str();
}

extern "C" int alz_create(const alz_config* cfg, alz_handle** out) {
  if (!cfg || !out || cfg->abi_version != ALZ_ABI_VERSION) return ALZ_E_INVAL;
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) return ALZ_E_NODEVICE;
  if (cfg->device < 0 || cfg->device >= ndev) return ALZ_E_INVAL;
  alz_handle* h = new (std::nothrow) alz_handle();
  if (!h) return ALZ_E_NOMEM;
  h->cfg = *cfg;
  if (h->cfg.max_endpoints == 0) h->cfg.max_endpoints = 1u << 16;
  if (h->cfg.max_pairs == 0) h->cfg.max_pairs = 1u << 20;
  if (h->cfg.max_edges == 0) h->cfg.max_edges = h->cfg.max_pairs;
  if (h->cfg.max_batch == 0) h->cfg.max_batch = 1u << 22;
  h->device = cfg->device;
  auto fail = [&](int rc) { alz_destroy(h); return rc; };
#define CKC(expr)                                                                      \
  do {                                                                                 \
    cudaError_t _e = (expr);                                                           \
    if (_e != cudaSuccess) {                                                           \
      fprintf(stderr, "libalazgpu: %s: %s\n", #expr, cudaGetErrorString(_e));          \
      return fail(_e == cudaErrorMemoryAllocation ? ALZ_E_NOMEM : ALZ_E_CUDA);         \
    }                                                                                  \
  } while (0)
  CKC(cudaSetDevice(h->device));
  cudaDeviceProp prop;
  CKC(cudaGetDeviceProperties(&prop, h->device));
  h->sms = prop.multiProcessorCount;
  Owned& m = h->mem;
  CKC(m.stream(&h->own_stream));
  CKC(m.stream(&h->copy_stream));
  h->stream = h->own_stream;
  for (int b = 0; b < kStageSlots + kRawSlots; ++b) {
    StageSlot& s = b < kStageSlots ? h->stage[b] : h->raw[b - kStageSlots];
    CKC(m.event(&s.copied, cudaEventDisableTiming));
    CKC(m.event(&s.consumed, cudaEventDisableTiming));
  }
  CKC(m.event(&h->ev_count, cudaEventDisableTiming));
  CKC(m.event(&h->ev_patch, cudaEventDisableTiming));
  for (int i = 0; i < 3; ++i) CKC(m.event(&h->ev_t[i], cudaEventDefault));

  h->ep_cap = next_pow2(2ull * h->cfg.max_endpoints);
  h->ep_tab.assign(h->ep_cap, EpEntry{0u, 0u, 0u, 0u});
  h->ep_touched.assign(h->ep_cap, 0);
  CKC(m.dev(&h->d_ep, (size_t)h->ep_cap * sizeof(EpEntry)));
  CKC(cudaMemsetAsync(h->d_ep, 0, (size_t)h->ep_cap * sizeof(EpEntry), h->stream));
  h->bloom_cnt.assign(ALZ_BLOOM_WORDS * 32u, 0);
  CKC(m.dev(&h->d_bloom, ALZ_BLOOM_WORDS * 4u));
  CKC(cudaMemsetAsync(h->d_bloom, 0, ALZ_BLOOM_WORDS * 4u, h->stream));   // no pods yet: every source is unresolvable
  CKC(m.pinned(&h->h_bloom, ALZ_BLOOM_WORDS * 4u));
  CKC(m.dev(&h->d_ctr, sizeof(Counters)));
  CKC(cudaMemsetAsync(h->d_ctr, 0, sizeof(Counters), h->stream));
  CKC(m.dev(&h->d_hot, sizeof(HotState)));
  CKC(cudaMemsetAsync(h->d_hot, 0, sizeof(HotState), h->stream));
  int rc;
  if (!(h->cfg.flags & ALZ_CFG_EAGER_JOIN)) {
    if ((rc = alloc_table(h, &h->pairs, h->cfg.max_pairs, &h->d_ctr->pair_rows, true)) != ALZ_OK) return fail(rc);
  }
  if ((rc = alloc_table(h, &h->edges, h->cfg.max_edges, &h->d_ctr->edge_rows, false)) != ALZ_OK) return fail(rc);
  CKC(m.pinned(&h->h_ctr, sizeof(Counters)));
  memset(h->h_ctr, 0, sizeof(Counters));
  CKC(m.dev(&h->d_keys, (size_t)h->cfg.max_edges * 8));
  for (int b = 0; b < 2; ++b) CKC(m.dev(&h->d_rows[b], (size_t)h->cfg.max_edges * 4));
  h->sort_tmp_bytes = sort_pairs_temp_bytes(h->cfg.max_edges);
  CKC(m.dev(&h->d_sort_tmp, h->sort_tmp_bytes));
  CKC(m.dev(&h->d_out, (size_t)h->cfg.max_edges * sizeof(alz_edge_out)));
  CKC(cudaStreamSynchronize(h->stream));
#undef CKC
  *out = h;
  return ALZ_OK;
}

extern "C" int alz_destroy(alz_handle* h) {
  if (!h) return ALZ_E_INVAL;
  cudaSetDevice(h->device);
  cudaDeviceSynchronize();
  // owners go in reverse declaration order (alz_handle.h): the optional states (the NCCL communicator before
  // the comm buffers), the grown buffers and the staging slots, then h->mem, whose streams are released last
  delete h;
  return ALZ_OK;
}

extern "C" int alz_set_stream(alz_handle* h, void* s) {
  if (!h) return ALZ_E_INVAL;
  std::lock_guard<std::mutex> g(h->mu);
  CK(cudaSetDevice(h->device));
  CK(cudaStreamSynchronize(h->stream));
  h->stream = s ? (cudaStream_t)s : h->own_stream;
  return ALZ_OK;
}

extern "C" int alz_sync(alz_handle* h) {
  if (!h) return ALZ_E_INVAL;
  std::lock_guard<std::mutex> g(h->mu);
  CK(cudaSetDevice(h->device));
  CK(cudaStreamSynchronize(h->copy_stream));
  CK(cudaStreamSynchronize(h->stream));
  return ALZ_OK;
}

// ---- pinned host memory for callers ----------------------------------------------
extern "C" int alz_pinned_alloc(size_t bytes, void** out) {
  if (!out || bytes == 0) return ALZ_E_INVAL;
  void* p = nullptr;
  if (cudaMallocHost(&p, bytes) != cudaSuccess) return ALZ_E_NOMEM;
  std::lock_guard<std::mutex> g(g_pin_mu);
  g_pinned.emplace_back((const char*)p, bytes);
  *out = p;
  return ALZ_OK;
}
extern "C" int alz_pinned_free(void* p) {
  if (!p) return ALZ_E_INVAL;
  {
    std::lock_guard<std::mutex> g(g_pin_mu);
    for (size_t i = 0; i < g_pinned.size(); ++i)
      if (g_pinned[i].first == (const char*)p) { g_pinned.erase(g_pinned.begin() + i); break; }
  }
  return cudaFreeHost(p) == cudaSuccess ? ALZ_OK : ALZ_E_CUDA;
}

// Run f() with the calling thread bound to the CPUs next to this handle's GPU (sysfs local_cpulist of
// the PCI device), so that pages it allocates and pins land on the GPU's NUMA node: with 8 ranks feeding
// 8 GPUs through host buffers, remote-socket staging memory halves the achievable H2D rate (r1: 80 ms
// per step at 8 ranks against 59 ms at 1-4). Best effort: without sysfs it just runs f().
template <class F>
static void with_gpu_local_cpus(int device, F f) {
  cpu_set_t old, want;
  CPU_ZERO(&want);
  bool bound = false;
  char bus[32] = {0};
  if (sched_getaffinity(0, sizeof(old), &old) == 0 && cudaDeviceGetPCIBusId(bus, sizeof(bus), device) == cudaSuccess) {
    for (char* c = bus; *c; ++c) *c = (char)tolower(*c);
    std::string path = std::string("/sys/bus/pci/devices/") + bus + "/local_cpulist";
    if (FILE* fp = fopen(path.c_str(), "r")) {
      char line[4096] = {0};
      if (fgets(line, sizeof(line), fp)) {
        for (char* tok = strtok(line, ",\n"); tok; tok = strtok(nullptr, ",\n")) {
          int a = 0, b = 0;
          if (sscanf(tok, "%d-%d", &a, &b) == 2) { for (int c = a; c <= b && c < CPU_SETSIZE; ++c) CPU_SET(c, &want); }
          else if (sscanf(tok, "%d", &a) == 1 && a < CPU_SETSIZE) CPU_SET(a, &want);
        }
        cpu_set_t both;
        CPU_AND(&both, &want, &old);
        if (CPU_COUNT(&both) > 0 && sched_setaffinity(0, sizeof(both), &both) == 0) bound = true;
      }
      fclose(fp);
    }
  }
  f();
  if (bound) sched_setaffinity(0, sizeof(old), &old);
}

// pinned memory on the NUMA node of `device`: allocated and first touched from the CPUs next to it
static cudaError_t pinned_alloc_local(int device, size_t bytes, void** out) {
  cudaError_t e = cudaSuccess;
  with_gpu_local_cpus(device, [&] {
    cudaSetDevice(device);
    e = cudaMallocHost(out, bytes);
    if (e == cudaSuccess) for (size_t o = 0; o < bytes; o += 4096) ((volatile char*)*out)[o] = 0;
  });
  return e;
}

extern "C" int alz_pinned_alloc_local(alz_handle* h, size_t bytes, void** out) {
  if (!h || !out || bytes == 0) return ALZ_E_INVAL;
  void* p = nullptr;
  if (pinned_alloc_local(h->device, bytes, &p) != cudaSuccess) return ALZ_E_NOMEM;
  std::lock_guard<std::mutex> g(g_pin_mu);
  g_pinned.emplace_back((const char*)p, bytes);
  *out = p;
  return ALZ_OK;
}

// ---- join build side -----------------------------------------------------------------
static int upsert_locked(alz_handle* h, int table, uint32_t ip, uint32_t id);
extern "C" int alz_table_upsert(alz_handle* h, int table, uint32_t ip, uint32_t id) {
  if (!h || (table != ALZ_TABLE_POD && table != ALZ_TABLE_SVC) || id >= (1u << 29)) return ALZ_E_INVAL;
  std::lock_guard<std::mutex> g(h->mu);
  return upsert_locked(h, table, ip, id);
}
extern "C" int alz_table_upsert_batch(alz_handle* h, int table, const uint32_t* ips, const uint32_t* ids, size_t n) {
  if (!h || (table != ALZ_TABLE_POD && table != ALZ_TABLE_SVC) || ((!ips || !ids) && n)) return ALZ_E_INVAL;
  std::lock_guard<std::mutex> g(h->mu);
  for (size_t i = 0; i < n; ++i) {
    if (ids[i] >= (1u << 29)) return ALZ_E_INVAL;
    const int rc = upsert_locked(h, table, ips[i], ids[i]);
    if (rc != ALZ_OK) return rc;
  }
  return ALZ_OK;
}
// the pod-address filter follows the pod table: counters per bit, so that a delete takes back exactly what the add set
static void bloom_update(alz_handle* h, uint32_t ip, int delta) {
  const uint32_t hh = hash32(ip);
  const uint32_t bits[2] = {hh & (ALZ_BLOOM_WORDS * 32u - 1u), (hh >> 15) & (ALZ_BLOOM_WORDS * 32u - 1u)};
  for (int k = 0; k < 2; ++k) {
    uint8_t& c = h->bloom_cnt[bits[k]];
    if (delta > 0) { if (c != 255) ++c; }
    else if (c != 255 && c != 0) --c;      // a saturated counter stays set: the filter may only err towards "maybe"
  }
  h->bloom_dirty = true;
}
static int upsert_locked(alz_handle* h, int table, uint32_t ip, uint32_t id) {
  auto it = h->ep_host.find(ip);
  if (it == h->ep_host.end()) {
    if (h->ep_host.size() >= h->cfg.max_endpoints) return ALZ_E_CAPACITY;
    it = h->ep_host.emplace(ip, HostEp{}).first;
  }
  HostEp& e = it->second;
  if (table == ALZ_TABLE_POD && !(e.state & kEpPod)) bloom_update(h, ip, +1);
  if (table == ALZ_TABLE_POD) { e.state |= kEpPod; e.pod = id; }   // persist.go:55-65
  else { e.state |= kEpSvc; e.svc = id; }                          // persist.go:114-124
  h->ep_dirty_ips.push_back(ip);
  return ALZ_OK;
}
extern "C" int alz_table_erase(alz_handle* h, int table, uint32_t ip) {
  if (!h || (table != ALZ_TABLE_POD && table != ALZ_TABLE_SVC)) return ALZ_E_INVAL;
  std::lock_guard<std::mutex> g(h->mu);
  auto it = h->ep_host.find(ip);
  if (it == h->ep_host.end()) return ALZ_OK;                       // delete of a missing key: no-op
  if (table == ALZ_TABLE_POD && (it->second.state & kEpPod)) bloom_update(h, ip, -1);
  it->second.state &= ~(table == ALZ_TABLE_POD ? kEpPod : kEpSvc); // persist.go:66-70, :125-129
  if (it->second.state == 0) h->ep_host.erase(it);
  h->ep_dirty_ips.push_back(ip);
  return ALZ_OK;
}

// host mirror of the open-addressed endpoint table: linear probing, deletion by backward shift (no
// tombstones, so the device's probe loop keeps its "stop at the first free slot" rule)
static void ep_touch(alz_handle* h, uint32_t slot) {
  if (!h->ep_touched[slot]) { h->ep_touched[slot] = 1; h->ep_touched_list.push_back(slot); }
}
static void ep_mirror_put(alz_handle* h, uint32_t ip, const HostEp& v) {
  const uint32_t mask = h->ep_cap - 1;
  uint32_t slot = hash32(ip) & mask;
  while ((h->ep_tab[slot].state & kEpOcc) && h->ep_tab[slot].ip != ip) slot = (slot + 1) & mask;
  h->ep_tab[slot] = EpEntry{ip, kEpOcc | v.state, v.pod, v.svc};
  ep_touch(h, slot);
}
static void ep_mirror_del(alz_handle* h, uint32_t ip) {
  const uint32_t mask = h->ep_cap - 1;
  uint32_t i = hash32(ip) & mask;
  while ((h->ep_tab[i].state & kEpOcc) && h->ep_tab[i].ip != ip) i = (i + 1) & mask;
  if (!(h->ep_tab[i].state & kEpOcc)) return;
  uint32_t j = i;
  for (;;) {
    j = (j + 1) & mask;
    if (!(h->ep_tab[j].state & kEpOcc)) break;
    const uint32_t k = hash32(h->ep_tab[j].ip) & mask;            // home of the entry at j
    const bool stays = (i <= j) ? (i < k && k <= j) : (i < k || k <= j);
    if (stays) continue;
    h->ep_tab[i] = h->ep_tab[j];
    ep_touch(h, i);
    i = j;
  }
  h->ep_tab[i] = EpEntry{0u, 0u, 0u, 0u};
  ep_touch(h, i);
}

static int fold_locked(alz_handle* h);

extern "C" int alz_table_commit(alz_handle* h) {
  if (!h) return ALZ_E_INVAL;
  std::lock_guard<std::mutex> g(h->mu);
  CK(cudaSetDevice(h->device));
  if (h->ep_dirty_ips.empty()) return ALZ_OK;
  // events already submitted are joined through the tables they arrived under
  int rc = fold_locked(h);
  if (rc != ALZ_OK) return rc;
  for (uint32_t ip : h->ep_dirty_ips) {
    auto it = h->ep_host.find(ip);
    if (it == h->ep_host.end()) ep_mirror_del(h, ip); else ep_mirror_put(h, ip, it->second);
  }
  h->ep_dirty_ips.clear();
  if (h->bloom_dirty) {   // 16 KB, through the pinned staging buffer, in stream order behind the fold above
    CK(cudaEventSynchronize(h->ev_patch));
    for (uint32_t w = 0; w < ALZ_BLOOM_WORDS; ++w) {
      uint32_t v = 0;
      for (uint32_t b = 0; b < 32; ++b) v |= (h->bloom_cnt[w * 32u + b] ? 1u : 0u) << b;
      h->h_bloom[w] = v;
    }
    CK(cudaMemcpyAsync(h->d_bloom, h->h_bloom, ALZ_BLOOM_WORDS * 4u, cudaMemcpyHostToDevice, h->stream));
    CK(cudaEventRecord(h->ev_patch, h->stream));
    h->bloom_dirty = false;
  }
  // only the slots that changed travel: (slot, entry) records through a pinned buffer, scattered on the
  // device in stream order (an informer burst under churn touches a handful of slots of a table that
  // may hold millions)
  const size_t n = h->ep_touched_list.size();
  if (n == 0) return ALZ_OK;
  CK(h->h_patch.ensure(n, h->stream, std::max<size_t>(1024, n * 2)));
  CK(h->d_patch.ensure(n, h->stream, std::max<size_t>(1024, n * 2)));
  CK(cudaEventSynchronize(h->ev_patch));   // the previous commit's upload has left the pinned buffer
  EpPatch* p = h->h_patch.get();
  for (size_t i = 0; i < n; ++i) {
    const uint32_t slot = h->ep_touched_list[i];
    p[i].slot = slot; p[i].pad[0] = p[i].pad[1] = p[i].pad[2] = 0;
    p[i].e = h->ep_tab[slot];
    h->ep_touched[slot] = 0;
  }
  h->ep_touched_list.clear();
  CK(cudaMemcpyAsync(h->d_patch.get(), p, n * sizeof(EpPatch), cudaMemcpyHostToDevice, h->stream));
  CK(cudaEventRecord(h->ev_patch, h->stream));
  launch_ep_patch(h->d_ep, h->d_patch.get(), (uint32_t)n, h->sms, h->stream);
  h->launches += 1;
  CK(cudaGetLastError());
  return ALZ_OK;
}

// ---- fold: the join on distinct pairs ------------------------------------------------------
// It also leaves per-pair counts behind, from which the next ingest launches learn which pairs are hot
// (alz_ingest.cu). Split in two so that a flush can read the edge count between the halves.
static int fold_first_half(alz_handle* h) {
  launch_fold_resolve(h->pairs, h->d_ep, h->ep_cap - 1, h->edges, h->d_ctr, h->d_hot, h->sms, h->stream);
  h->launches += 1;
  CK(cudaGetLastError());
  return ALZ_OK;
}
static int fold_second_half(alz_handle* h) {
  launch_fold_add(h->pairs, h->edges, h->d_ctr, h->d_hot, h->sms, h->stream);
  launch_hot_select(h->pairs, h->d_hot, h->sms, h->stream);
  h->launches += 2;
  CK(cudaGetLastError());
  int rc = clear_dict(h, &h->pairs);
  h->pending_since_fold = 0;
  return rc;
}
static int fold_locked(alz_handle* h) {
  if (h->cfg.flags & ALZ_CFG_EAGER_JOIN) return ALZ_OK;
  if (h->pending_since_fold == 0) return ALZ_OK;
  int rc = fold_first_half(h);
  if (rc != ALZ_OK) return rc;
  return fold_second_half(h);
}
int alz_internal_fold(alz_handle* h) { return fold_locked(h); }

// ---- ingest ------------------------------------------------------------------------------
// requires h->mu
static int ingest_device(alz_handle* h, const void* d, uint64_t n, bool rec16, const uint64_t* d_ovf) {
  if (h->win_on && (rec16 || (h->cfg.flags & (ALZ_CFG_EAGER_JOIN | ALZ_CFG_NO_SMEM_CACHE)))) return ALZ_E_STATE;
  if (rec16) {
    if (h->cfg.flags & (ALZ_CFG_EAGER_JOIN | ALZ_CFG_NO_SMEM_CACHE)) return ALZ_E_UNSUPPORTED;
    launch_ingest_pairs_rec16((const alz_l7_rec16*)d, n, d_ovf, h->pairs, h->d_ctr, h->d_hot, h->d_ep, h->ep_cap - 1,
                              h->d_bloom, h->sms, h->stream);
  } else if (h->cfg.flags & ALZ_CFG_EAGER_JOIN) {
    launch_ingest_eager((const alz_l7_rec*)d, n, h->d_ep, h->ep_cap - 1, h->edges, h->d_ctr, h->sms, h->stream);
  } else if (h->cfg.flags & ALZ_CFG_NO_SMEM_CACHE) {
    launch_ingest_pairs_v1((const alz_l7_rec*)d, n, h->pairs, h->d_ctr, h->d_ep, h->ep_cap - 1, h->sms, h->stream);
  } else if (h->win_on) {
    launch_ingest_pairs_windowed((const alz_l7_rec*)d, n, h->pairs, h->d_ctr, h->d_hot, h->d_ep, h->ep_cap - 1, h->d_bloom,
                                 h->d_win, h->win_off, h->d_defer[h->defer_cur], h->defer_cap, h->sms, h->stream);
    h->launches += 1;
  } else {
    launch_ingest_pairs((const alz_l7_rec*)d, n, h->pairs, h->d_ctr, h->d_hot, h->d_ep, h->ep_cap - 1, h->d_bloom, h->sms,
                        h->stream);
  }
  CK(cudaGetLastError());
  h->launches += n ? 1 : 0;
  h->events_in += n;
  h->pending_since_fold += n;
  // pair histograms are u32: fold before any bucket could wrap
  if (h->pending_since_fold >= (1ull << 31)) return fold_locked(h);
  return ALZ_OK;
}

int alz_internal_ingest(alz_handle* h, const alz_l7_rec* d_recs, size_t n) { return ingest_device(h, d_recs, n, false, nullptr); }

extern "C" int alz_submit_l7_device(alz_handle* h, const alz_l7_rec* d, size_t n) {
  if (!h || (!d && n)) return ALZ_E_INVAL;
  if (((uintptr_t)d & 31u) != 0) return ALZ_E_INVAL;  // 32-B records, bulk copies
  std::lock_guard<std::mutex> g(h->mu);
  CK(cudaSetDevice(h->device));
  return ingest_device(h, d, n, false, nullptr);
}

extern "C" int alz_submit_l7_packed_device(alz_handle* h, const alz_l7_rec16* d, size_t n, const uint64_t* d_ovf) {
  if (!h || (!d && n)) return ALZ_E_INVAL;
  if (((uintptr_t)d & 15u) != 0) return ALZ_E_INVAL;
  std::lock_guard<std::mutex> g(h->mu);
  CK(cudaSetDevice(h->device));
  return ingest_device(h, d, n, true, d_ovf);
}

// staging slot s ready for `bytes` (allocated on first use, pinned memory next to the GPU); published only
// once every buffer exists
static int ensure_slot(alz_handle* h, StageSlot& s, size_t bytes, size_t aux_bytes) {
  if (s.h) return ALZ_OK;
  void* p = nullptr;
  const cudaError_t e = pinned_alloc_local(h->device, bytes, &p);
  if (e != cudaSuccess) return alz_error(h, ALZ_E_NOMEM, nullptr, cudaGetErrorString(e));
  Owner hb(p, ResFree{Res::kPinned}), d, aux;
  CK(alz_alloc(d, Res::kDev, bytes));
  if (aux_bytes) CK(alz_alloc(aux, Res::kDev, aux_bytes));
  s.d = std::move(d);
  s.d_aux = std::move(aux);
  s.h = std::move(hb);
  return ALZ_OK;
}

// Host records -> device -> ingest, in chunks through the staging slots. rec_bytes = 32 (alz_l7_rec) or
// 16 (alz_l7_rec16); raw: ALZ_BPF_L7_EVENT_SIZE-byte samples through the raw slots, compacted into 32-B
// records on the device before the ingest. A chunk is as many records as fit the byte size of max_batch
// 32-B records.
static int submit_staged(alz_handle* h, const void* recs, size_t n, size_t rec_bytes, bool raw, const uint64_t* d_ovf) {
  StageSlot* slots = raw ? h->raw : h->stage;
  const int n_slots = raw ? kRawSlots : kStageSlots;
  uint64_t& next_turn = raw ? h->raw_turn : h->stage_turn;
  const bool direct = is_lib_pinned(recs, n * rec_bytes);
  const size_t per = std::max<size_t>(1, (size_t)h->cfg.max_batch * sizeof(alz_l7_rec) / rec_bytes);
  size_t done = 0;
  while (done < n) {
    const size_t m = std::min(per, n - done);
    uint64_t turn;
    { std::lock_guard<std::mutex> t(h->turn_mu); turn = next_turn++; }
    StageSlot& s = slots[turn % n_slots];
    std::lock_guard<std::mutex> own(s.mu);
    int rc = ensure_slot(h, s, per * rec_bytes, raw ? per * sizeof(alz_l7_rec) : 0);
    if (rc != ALZ_OK) return rc;
    const void* src = (const char*)recs + done * rec_bytes;
    if (!direct) {
      CK(cudaEventSynchronize(s.copied));      // the previous H2D out of this pinned buffer is done
      memcpy(s.h.get(), src, m * rec_bytes);   // in parallel with other submitting threads
      src = s.h.get();
    }
    {
      std::lock_guard<std::mutex> g(h->mu);
      // the copy of chunk k+1 overlaps the (compaction +) ingest of chunk k (two slots or more, two streams)
      CK(cudaStreamWaitEvent(h->copy_stream, s.consumed, 0));   // the kernel that read s.d
      CK(cudaMemcpyAsync(s.d.get(), src, m * rec_bytes, cudaMemcpyHostToDevice, h->copy_stream));
      CK(cudaEventRecord(s.copied, h->copy_stream));
      CK(cudaStreamWaitEvent(h->stream, s.copied, 0));
      const void* d = s.d.get();
      if (raw) {
        launch_compact_raw((const uint8_t*)d, m, (alz_l7_rec*)s.d_aux.get(), h->sms, h->stream);
        h->launches += 1;
        d = s.d_aux.get();
      }
      rc = ingest_device(h, d, m, rec_bytes == sizeof(alz_l7_rec16), d_ovf);
      if (rc != ALZ_OK) return rc;
      CK(cudaEventRecord(s.consumed, h->stream));
    }
    done += m;
  }
  if (direct) CK(cudaStreamSynchronize(h->copy_stream));   // the caller may reuse its pinned buffer once we return
  return ALZ_OK;
}

extern "C" int alz_submit_l7(alz_handle* h, const alz_l7_rec* recs, size_t n) {
  if (!h || (!recs && n)) return ALZ_E_INVAL;
  CK(cudaSetDevice(h->device));
  return submit_staged(h, recs, n, sizeof(alz_l7_rec), false, nullptr);
}

extern "C" int alz_submit_l7_packed(alz_handle* h, const alz_l7_rec16* recs, size_t n, const uint64_t* ovf, size_t n_ovf) {
  if (!h || (!recs && n) || (!ovf && n_ovf)) return ALZ_E_INVAL;
  CK(cudaSetDevice(h->device));
  uint64_t* d_ovf = nullptr;
  if (n_ovf) {   // rare (durations >= 4.29 s): a stream-ordered allocation that lives until the kernels have run
    std::lock_guard<std::mutex> g(h->mu);
    CK(cudaMallocAsync(&d_ovf, n_ovf * 8, h->stream));
    CK(cudaMemcpyAsync(d_ovf, ovf, n_ovf * 8, cudaMemcpyHostToDevice, h->stream));
    CK(cudaStreamSynchronize(h->stream));   // ovf is caller memory (possibly pageable): done with it before returning
  }
  int rc = submit_staged(h, recs, n, sizeof(alz_l7_rec16), false, d_ovf);
  if (d_ovf) { std::lock_guard<std::mutex> g(h->mu); cudaFreeAsync(d_ovf, h->stream); }
  return rc;
}

extern "C" long alz_pack_l7(const alz_l7_rec* recs, size_t n, alz_l7_rec16* out, uint64_t* ovf, size_t cap_ovf) {
  if ((!recs || !out) && n) return -1;
  size_t k = 0;
  for (size_t i = 0; i < n; ++i) {
    const alz_l7_rec& r = recs[i];
    alz_l7_rec16 o;
    o.saddr = r.saddr; o.daddr = r.daddr; o.status = r.status;
    o.protocol = r.protocol & 0x7Fu; o.method_flags = r.method_flags;   // keeps ALZ_PROTO_F_HOSTKEY
    if (r.protocol & 0x80u) o.protocol = 0x3Fu;   // no such protocol either way: stays "not a request row"
    if (r.duration_ns >> 32) {
      if (k >= cap_ovf || !ovf) return -1;
      ovf[k] = r.duration_ns;
      o.duration_ns = (uint32_t)k++;
      o.protocol |= ALZ_REC16_DUR_OVERFLOW;
    } else {
      o.duration_ns = (uint32_t)r.duration_ns;
    }
    out[i] = o;
  }
  return (long)k;
}

extern "C" int alz_submit_l7_raw(alz_handle* h, const void* raw, size_t n) {
  if (!h || (!raw && n)) return ALZ_E_INVAL;
  CK(cudaSetDevice(h->device));
  return submit_staged(h, raw, n, ALZ_BPF_L7_EVENT_SIZE, true, nullptr);
}

// ---- window result ---------------------------------------------------------------------------
// Fold + sort of the live edge keys (no reset). After it h->n_live edges sit in d_keys/d_rows[1].
// The edge count is final once the first half of the fold has run, so the counters are copied out right
// there and the host waits on an event for THAT copy only: the second half of the fold is still
// running on the GPU while the host sizes and enqueues the sort (r1 stalled the whole stream here).
// *overflow: the window lost rows (pair or edge table full); the flush still emits what it has.
static int prepare_flush(alz_handle* h, bool* overflow) {
  *overflow = false;
  const bool fold = !(h->cfg.flags & ALZ_CFG_EAGER_JOIN) && h->pending_since_fold != 0;
  int rc = ALZ_OK;
  if (fold && (rc = fold_first_half(h)) != ALZ_OK) return rc;
  CK(cudaMemcpyAsync(h->h_ctr, h->d_ctr, sizeof(Counters), cudaMemcpyDeviceToHost, h->stream));
  CK(cudaEventRecord(h->ev_count, h->stream));
  if (fold && (rc = fold_second_half(h)) != ALZ_OK) return rc;
  CK(cudaEventSynchronize(h->ev_count));
  h->n_live = h->h_ctr->edge_rows;
  if (h->n_live > h->cfg.max_edges) { h->n_live = h->cfg.max_edges; *overflow = true; }
  // events the pair table could not take during this window's ingest launches
  if (h->h_ctr->capacity_events != h->lost_reported) { h->lost_reported = h->h_ctr->capacity_events; *overflow = true; }
  if (h->n_live) {
    launch_iota(h->d_rows[0], h->n_live, h->sms, h->stream);
    h->launches += 1;
    sort_pairs(h->d_sort_tmp, h->sort_tmp_bytes, h->edges.row_key, h->d_keys, h->d_rows[0], h->d_rows[1],
               h->n_live, h->stream);
    CK(cudaGetLastError());
  }
  return ALZ_OK;
}

static int finish_flush(alz_handle* h) {
  launch_gather_edges(h->edges, h->d_keys, h->d_rows[1], h->n_live, h->d_out, true, h->sms, h->stream);
  h->launches += h->n_live ? 1 : 0;
  CK(cudaGetLastError());
  int rc = clear_dict(h, &h->edges);
  if (rc != ALZ_OK) return rc;
  h->last_n_edges = h->n_live;
  h->windows++;
  return alz_internal_history_append(h);
}

// time-cut windows: the flushed epoch is closed; open the next one and submit the records that waited for it
// (those of still later epochs are deferred again, into the other buffer)
static int window_roll(alz_handle* h) {
  if (!h->win_on) return ALZ_OK;
  launch_window_advance(h->d_win, h->stream);
  h->launches += 1;
  const uint32_t n_def = std::min<uint32_t>(h->h_ctr->defer_count, h->defer_cap);   // read with the edge count
  CK(cudaMemsetAsync(&h->d_ctr->defer_count, 0, 4, h->stream));
  if (n_def == 0) return ALZ_OK;
  const alz_l7_rec* src = h->d_defer[h->defer_cur];
  h->defer_cur ^= 1;
  const uint64_t before = h->events_in;
  const int rc = ingest_device(h, src, n_def, false, nullptr);
  h->events_in = before;   // they were counted when they were first submitted
  return rc;
}

static int flush_device_locked(alz_handle* h, const alz_edge_out** dev_edges, size_t* n_out) {
  bool overflow = false;
  CK(cudaEventRecord(h->ev_t[0], h->stream));
  int rc = prepare_flush(h, &overflow);
  *n_out = h->n_live;
  CK(cudaEventRecord(h->ev_t[1], h->stream));
  int mrc;
  if (h->comm_nranks > 1) {
    mrc = alz_internal_merge_ranks(h, rc);  // one collective over the ranks' edge rows (alz_comm.cu)
  } else {
    if (rc != ALZ_OK) return rc;
    mrc = finish_flush(h);
  }
  CK(cudaEventRecord(h->ev_t[2], h->stream));
  h->ev_t_valid = true;
  if (mrc != ALZ_OK) return mrc;
  if ((mrc = window_roll(h)) != ALZ_OK) return mrc;
  *n_out = h->last_n_edges;
  if (dev_edges) *dev_edges = h->d_out;
  return overflow ? ALZ_E_CAPACITY : ALZ_OK;
}

extern "C" int alz_window_flush_device(alz_handle* h, const alz_edge_out** dev_edges, size_t* n_out) {
  if (!h || !n_out) return ALZ_E_INVAL;
  std::lock_guard<std::mutex> g(h->mu);
  CK(cudaSetDevice(h->device));
  return flush_device_locked(h, dev_edges, n_out);
}

extern "C" int alz_window_flush(alz_handle* h, alz_edge_out* out, size_t cap, size_t* n_out) {
  if (!h || !n_out || (!out && cap)) return ALZ_E_INVAL;
  std::lock_guard<std::mutex> g(h->mu);
  CK(cudaSetDevice(h->device));
  if (h->comm_nranks <= 1) {
    // size check first so that a too-small buffer keeps the window intact
    bool overflow = false;
    int rc = prepare_flush(h, &overflow);
    *n_out = h->n_live;
    if (rc != ALZ_OK) return rc;
    if (h->n_live > cap) { if (overflow) h->lost_reported = ~0ull; return ALZ_E_CAPACITY; }   // report the loss again next time
    rc = finish_flush(h);
    if (rc != ALZ_OK) return rc;
    if (h->n_live) CK(cudaMemcpyAsync(out, h->d_out, (size_t)h->n_live * sizeof(alz_edge_out),
                                      cudaMemcpyDeviceToHost, h->stream));
    if ((rc = window_roll(h)) != ALZ_OK) return rc;
    CK(cudaStreamSynchronize(h->stream));
    return overflow ? ALZ_E_CAPACITY : ALZ_OK;
  }
  // several ranks: the merge consumes the window on every rank, so a too-small buffer cannot keep it.
  // The merged rows stay on the device (alz_window_fetch) and *n_out says how many there are.
  const alz_edge_out* d = nullptr;
  int rc = flush_device_locked(h, &d, n_out);
  if (rc != ALZ_OK && rc != ALZ_E_CAPACITY) return rc;
  if (*n_out > cap) return ALZ_E_CAPACITY;
  if (*n_out) CK(cudaMemcpyAsync(out, d, *n_out * sizeof(alz_edge_out), cudaMemcpyDeviceToHost, h->stream));
  CK(cudaStreamSynchronize(h->stream));
  return rc;
}

// the rows of the last flushed window again (e.g. after a flush that returned ALZ_E_CAPACITY because the
// caller's buffer was too small on a multi-rank handle)
extern "C" int alz_window_fetch(alz_handle* h, alz_edge_out* out, size_t cap, size_t* n_out) {
  if (!h || !n_out || (!out && cap)) return ALZ_E_INVAL;
  std::lock_guard<std::mutex> g(h->mu);
  CK(cudaSetDevice(h->device));
  *n_out = h->last_n_edges;
  if (h->last_n_edges > cap) return ALZ_E_CAPACITY;
  if (h->last_n_edges) CK(cudaMemcpyAsync(out, h->d_out, (size_t)h->last_n_edges * sizeof(alz_edge_out),
                                          cudaMemcpyDeviceToHost, h->stream));
  CK(cudaStreamSynchronize(h->stream));
  return ALZ_OK;
}

extern "C" int alz_get_stats(alz_handle* h, alz_stats* st) {
  if (!h || !st) return ALZ_E_INVAL;
  std::lock_guard<std::mutex> g(h->mu);
  CK(cudaSetDevice(h->device));
  CK(cudaMemcpyAsync(h->h_ctr, h->d_ctr, sizeof(Counters), cudaMemcpyDeviceToHost, h->stream));
  CK(cudaStreamSynchronize(h->stream));
  memset(st, 0, sizeof(*st));
  const uint64_t lost = h->h_ctr->capacity_events + h->h_ctr->fold_lost_events;
  st->events_in = h->events_in;
  st->not_request = h->h_ctr->not_request;
  st->src_unresolved = h->h_ctr->src_unresolved;   // complete once pending pairs are folded
  st->rows_emitted = h->events_in - st->not_request - st->src_unresolved - lost - h->h_ctr->defer_count;   // waiting records are not rows yet
  st->pairs_live = h->h_ctr->pair_rows;
  st->edges_live = h->h_ctr->edge_rows;
  st->tcp_events_in = h->tcp_events_in;
  st->tcp_localhost_dropped = h->tcp_localhost_dropped;
  st->capacity_events = lost;
  st->windows = h->windows;
  st->late_events = h->h_ctr->late_events;
  st->deferred_events = h->h_ctr->defer_count;
  st->kernel_launches = h->launches;
  st->collective_bytes_last = h->collective_bytes_last;
  if (h->ev_t_valid) {   // the stream was synchronised above, so the events have completed
    float a = 0.f, b = 0.f;
    if (cudaEventElapsedTime(&a, h->ev_t[0], h->ev_t[1]) == cudaSuccess) st->flush_local_us_last = (uint64_t)(a * 1000.f);
    if (cudaEventElapsedTime(&b, h->ev_t[1], h->ev_t[2]) == cudaSuccess) st->merge_us_last = (uint64_t)(b * 1000.f);
  }
  return ALZ_OK;
}

extern "C" int alz_window_clock(alz_handle* h, uint64_t first_kernel_ns, uint64_t first_user_ns, uint64_t window_ns) {
  if (!h) return ALZ_E_INVAL;
  std::lock_guard<std::mutex> g(h->mu);
  CK(cudaSetDevice(h->device));
  if (h->pending_since_fold != 0 || h->h_ctr->defer_count != 0) return ALZ_E_STATE;   // only between windows
  if (window_ns == 0) { h->win_on = false; return ALZ_OK; }
  h->defer_cap = 2u * h->cfg.max_batch;
  for (int b = 0; b < 2; ++b)   // each allocated once; a retry after a failure allocates only what is missing
    if (!h->d_defer[b]) CK(h->mem.dev(&h->d_defer[b], (size_t)h->defer_cap * sizeof(alz_l7_rec)));
  if (!h->d_win) CK(h->mem.dev(&h->d_win, 3 * sizeof(uint64_t)));
  const uint64_t init[3] = {0ull, window_ns, 0ull};
  CK(cudaMemcpyAsync(h->d_win, init, sizeof(init), cudaMemcpyHostToDevice, h->stream));
  CK(cudaStreamSynchronize(h->stream));
  h->win_off = first_user_ns - first_kernel_ns;
  h->win_on = true;
  return ALZ_OK;
}
extern "C" int alz_window_epoch(alz_handle* h, uint64_t* epoch) {
  if (!h || !epoch) return ALZ_E_INVAL;
  std::lock_guard<std::mutex> g(h->mu);
  CK(cudaSetDevice(h->device));
  if (!h->win_on) return ALZ_E_STATE;
  uint64_t w[3];
  CK(cudaMemcpyAsync(w, h->d_win, sizeof(w), cudaMemcpyDeviceToHost, h->stream));
  CK(cudaStreamSynchronize(h->stream));
  if (!w[2]) return ALZ_E_STATE;
  *epoch = (w[0] + h->win_off) / w[1];
  return ALZ_OK;
}

// make pending pairs visible in the edge accumulators (and in src_unresolved)
extern "C" int alz_fold(alz_handle* h) {
  if (!h) return ALZ_E_INVAL;
  std::lock_guard<std::mutex> g(h->mu);
  CK(cudaSetDevice(h->device));
  return fold_locked(h);
}

extern "C" uint32_t alz_owner_rank(uint32_t saddr, uint32_t nranks) { return owner_rank(saddr, nranks); }

// ---- device memory helpers + synthetic stream (include/alazgpu_synth.h) ---------------------------
extern "C" int alz_dev_alloc(alz_handle* h, size_t bytes, void** out) {
  if (!h || !out) return ALZ_E_INVAL;
  CK(cudaSetDevice(h->device));
  const cudaError_t e = cudaMalloc(out, bytes);   // the caller's: freed with alz_dev_free
  if (e != cudaSuccess) return alz_error(h, ALZ_E_NOMEM, nullptr, cudaGetErrorString(e));
  return ALZ_OK;
}
extern "C" int alz_dev_free(alz_handle* h, void* p) {
  if (!h) return ALZ_E_INVAL;
  CK(cudaSetDevice(h->device));
  CK(cudaFree(p));
  return ALZ_OK;
}
extern "C" int alz_memcpy_h2d(alz_handle* h, void* dst, const void* src, size_t bytes) {
  if (!h) return ALZ_E_INVAL;
  std::lock_guard<std::mutex> g(h->mu);
  CK(cudaSetDevice(h->device));
  CK(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, h->stream));
  CK(cudaStreamSynchronize(h->stream));
  return ALZ_OK;
}
extern "C" int alz_memcpy_d2h(alz_handle* h, void* dst, const void* src, size_t bytes) {
  if (!h) return ALZ_E_INVAL;
  std::lock_guard<std::mutex> g(h->mu);
  CK(cudaSetDevice(h->device));
  CK(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, h->stream));
  CK(cudaStreamSynchronize(h->stream));
  return ALZ_OK;
}

struct alz_synth_dev {
  alz_synth_view view;  // device pointers into mem
  Owned mem;
};

extern "C" int alz_synth_dev_create(alz_handle* h, const alz_synth_topo* t, alz_synth_dev** out) {
  if (!h || !t || !out) return ALZ_E_INVAL;
  std::lock_guard<std::mutex> g(h->mu);
  CK(cudaSetDevice(h->device));
  std::unique_ptr<alz_synth_dev> d(new (std::nothrow) alz_synth_dev());
  if (!d) return ALZ_E_NOMEM;
  d->view = t->view;
  const size_t E = t->n_edges;
  const void* src[6] = {t->edge_saddr, t->edge_daddr, t->edge_flags, t->alias_thresh, t->alias_idx, t->lat_q};
  const size_t bytes[6] = {E * 4, E * 4, E, E * 4, E * 4, (ALZ_SYNTH_LATQ + 1) * 8};
  void* bufs[6];
  for (int i = 0; i < 6; ++i) {
    CK(d->mem.dev(&bufs[i], bytes[i]));
    CK(cudaMemcpyAsync(bufs[i], src[i], bytes[i], cudaMemcpyHostToDevice, h->stream));
  }
  CK(cudaStreamSynchronize(h->stream));   // the sources are pageable caller memory
  d->view.edge_saddr = (const uint32_t*)bufs[0];
  d->view.edge_daddr = (const uint32_t*)bufs[1];
  d->view.edge_flags = (const uint8_t*)bufs[2];
  d->view.alias_thresh = (const uint32_t*)bufs[3];
  d->view.alias_idx = (const uint32_t*)bufs[4];
  d->view.lat_q = (const uint64_t*)bufs[5];
  *out = d.release();
  return ALZ_OK;
}
extern "C" int alz_synth_dev_fill(alz_handle* h, alz_synth_dev* d, uint64_t first, uint64_t n, alz_l7_rec* dev_out) {
  if (!h || !d || (!dev_out && n)) return ALZ_E_INVAL;
  std::lock_guard<std::mutex> g(h->mu);
  CK(cudaSetDevice(h->device));
  launch_synth(d->view, first, n, dev_out, h->sms, h->stream);
  CK(cudaGetLastError());
  return ALZ_OK;
}
// First `want` events of the global stream (indices first, first+1, ...) that rank `rank` of `nranks` owns,
// scanning in chunks; *n_scanned = how many global events were looked at. Order within dev_out is arbitrary.
extern "C" int alz_synth_dev_fill_owned(alz_handle* h, alz_synth_dev* d, uint64_t first, uint32_t nranks, uint32_t rank,
                                        alz_l7_rec* dev_out, uint64_t want, uint64_t* n_written, uint64_t* n_scanned) {
  if (!h || !d || !dev_out || !n_written || !n_scanned || nranks == 0 || rank >= nranks) return ALZ_E_INVAL;
  std::lock_guard<std::mutex> g(h->mu);
  CK(cudaSetDevice(h->device));
  Owned scratch;   // freed on every return, with the device still current
  unsigned long long* d_cnt = nullptr;
  CK(scratch.dev(&d_cnt, 8));
  CK(cudaMemsetAsync(d_cnt, 0, 8, h->stream));
  const uint64_t chunk = std::max<uint64_t>(1u << 20, want / 4);
  unsigned long long got = 0;
  uint64_t scanned = 0;
  while (got < want && scanned < want * (uint64_t)nranks * 64ull) {
    launch_synth_owned(d->view, first + scanned, chunk, nranks, rank, dev_out, want, d_cnt, h->sms, h->stream);
    scanned += chunk;
    CK(cudaMemcpyAsync(&got, d_cnt, 8, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
  }
  *n_written = got < want ? got : want;
  *n_scanned = scanned;
  return ALZ_OK;
}
extern "C" int alz_synth_dev_destroy(alz_handle* h, alz_synth_dev* d) {
  if (!h || !d) return ALZ_E_INVAL;
  cudaSetDevice(h->device);
  delete d;
  return ALZ_OK;
}
