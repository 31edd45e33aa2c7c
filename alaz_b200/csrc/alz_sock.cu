// alz_sock.cu — tcp_state sink and the temporal socket join (SURVEY.md §8 rows R11/R12, f.2).
//
// Replaces, for events whose in-event 5-tuple is empty (get_sock miss, ebpf/c/l7.c:313-314):
//   processTcpConnect      aggregator/data.go:404-506   -> alz_submit_tcp   (host, exact order semantics)
//   SocketLine.AddValue    aggregator/sock_num_line.go:62-80, 311-322
//   SocketLine.GetValue    aggregator/sock_num_line.go:82-158 -> alz_sock_lookup (device, one thread per query)
//
// tcp_state events are two per connection and AddValue's dedupe depends on arrival order ("equal to the LAST
// element"), so the host keeps each line's timestamps and 5-tuples and decides, sequentially as the reference does,
// WHERE every new value goes. The lines themselves live in HBM: a record pool with one segment per (pid, fd) and an
// open-addressed index. A sync sends only the inserts since the last one (48 B each) and one warp per changed line
// applies them on the device (shift the tail, move a grown segment), so the LastMatch stamps the lookups write stay
// with their records. Consumers, all one thread per query / line on the device:
//   alz_sock_lookup      GetValue for a batch of (pid, fd, timestamp)
//   alz_submit_l7_join   findRelatedSocket (data.go:1407-1429) for L7 events with an empty 5-tuple, then ingest
//   alz_sock_alive       sendOpenConnection (data.go:1628-1679) for every line
//   alz_sock_gc          clearSocketLines / DeleteUnused (data.go:1681-1716, sock_num_line.go:160-209)
#include <algorithm>
#include <cstring>
#include <ctime>
#include <mutex>
#include <string>
#include <unordered_map>
#include <vector>

#include "alz_handle.h"

using namespace alz;

namespace {

struct SockRec {       // one TimestampedSocket (sock_num_line.go:23-27)
  uint64_t ts;
  uint64_t lm;         // LastMatch: written by the lookups on the device, read back by the GC
  uint32_t saddr, daddr;
  uint16_t sport, dport;
  uint32_t open;       // SockInfo != nil
};
static_assert(sizeof(SockRec) == 32, "SockRec layout");

struct LineEnt {       // index entry: (pid, fd) -> segment of the record pool
  uint64_t fd;
  uint32_t pid;
  uint32_t used;
  uint32_t off, len;
  uint64_t pad;
};
static_assert(sizeof(LineEnt) == 32, "LineEnt layout");

// One changed line of a sync: copy len_before records from src_off to dst_off (segment moved or pool
// replaced), then apply n_ops sorted inserts, then publish the index entry.
struct LineDesc {
  uint64_t fd;
  uint32_t pid, slot;
  uint32_t src_off, dst_off;
  uint32_t len_before, op_begin, n_ops, pad;
};
static_assert(sizeof(LineDesc) == 40, "LineDesc layout");
struct LineOp {        // insertIntoSortedSlice at `pos` of the line as it is when the op is applied
  SockRec rec;
  uint32_t pos, pad[3];
};
static_assert(sizeof(LineOp) == 48, "LineOp layout");

struct LineKey {
  uint32_t pid;
  uint64_t fd;
  bool operator==(const LineKey& o) const { return pid == o.pid && fd == o.fd; }
};
struct LineKeyHash {
  size_t operator()(const LineKey& k) const { return (size_t)hash64(((uint64_t)k.pid << 40) ^ k.fd ^ 0x9E3779B97F4A7C15ull); }
};

__host__ __device__ inline uint32_t line_slot(uint32_t pid, uint64_t fd, uint32_t mask) {
  return (uint32_t)hash64(((uint64_t)pid << 40) ^ fd ^ 0x9E3779B97F4A7C15ull) & mask;
}

constexpr uint64_t kOneMinuteNs = 60ull * 1000000000ull;
constexpr uint64_t kFiveMinutesNs = 5ull * kOneMinuteNs;
constexpr uint32_t kLocalhost = 0x7F000001u;   // "127.0.0.1" (data.go:409, :455)

__device__ __forceinline__ const SockRec* find_line(const LineEnt* __restrict__ index, uint32_t mask,
                                                    SockRec* recs, uint32_t pid, uint64_t fd, uint32_t* len) {
  uint32_t slot = line_slot(pid, fd, mask);
  for (;;) {
    const LineEnt e = index[slot];
    if (!e.used) { *len = 0; return nullptr; }
    if (e.pid == pid && e.fd == fd) { *len = e.len; return recs + e.off; }
    slot = (slot + 1u) & mask;
  }
}

// SocketLine.GetValue on one line of the pool; stamps LastMatch where the reference does (:96, :156)
__device__ __forceinline__ const SockRec* get_value(SockRec* v, uint32_t len, uint64_t ts, uint64_t now) {
  if (v == nullptr || len == 0u) return nullptr;                       // :86-88 empty line -> error
  uint32_t lo = 0, hi = len;                                           // sort.Search(!(Timestamp < ts)) :90-92
  while (lo < hi) { const uint32_t mid = (lo + hi) >> 1; if (!(v[mid].ts < ts)) hi = mid; else lo = mid + 1; }
  const uint32_t idx = lo;
  if (idx == len) {                                                    // after the last entry, :94-105
    atomicMax((unsigned long long*)&v[len - 1].lm, (unsigned long long)now);
    if (!v[len - 1].open) {
      if (idx >= 2u && v[idx - 2].open && (ts - v[idx - 2].ts) < kOneMinuteNs) return &v[idx - 2];
      return nullptr;
    }
    return &v[len - 1];
  }
  if (idx == 0u) return v[0].open ? &v[0] : nullptr;                   // before the first entry, :107-119
  if (!v[idx - 1].open) {                                              // matched a close, :123-153
    if (idx >= 2u && v[idx - 2].open && v[idx].open && v[idx - 2].daddr == v[idx].daddr &&
        v[idx - 2].dport == v[idx].dport)
      return (ts - v[idx - 2].ts < v[idx].ts - ts) ? &v[idx - 2] : &v[idx];
    return nullptr;
  }
  atomicMax((unsigned long long*)&v[idx - 1].lm, (unsigned long long)now);   // :155-157
  return &v[idx - 1];
}

__global__ void __launch_bounds__(256) sock_lookup_kernel(const LineEnt* __restrict__ index, uint32_t mask,
                                                          SockRec* recs, const alz_sock_query* __restrict__ q,
                                                          uint32_t n, uint64_t now, alz_sock_result* __restrict__ out) {
  const uint32_t stride = gridDim.x * blockDim.x;
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
    alz_sock_result r;
    r.found = 0; r.saddr = 0; r.daddr = 0; r.sport = 0; r.dport = 0;
    uint32_t len;
    SockRec* v = const_cast<SockRec*>(find_line(index, mask, recs, q[i].pid, q[i].fd, &len));   // data.go:1407-1429
    const SockRec* hit = get_value(v, len, q[i].timestamp_ns, now);
    if (hit != nullptr) {
      r.found = 1; r.saddr = hit->saddr; r.daddr = hit->daddr; r.sport = hit->sport; r.dport = hit->dport;
    }
    out[i] = r;
  }
}

// L7 records whose in-event 5-tuple is empty (get_sock miss, ebpf/c/l7.c:313-314) take their addresses from
// the timeline of their (pid, fd) at their write time; a miss leaves the zeros, and 0.0.0.0 is no pod, so the
// ingest kernel drops the event the way setFromToV2 would (data.go:829-832)
__global__ void __launch_bounds__(256) sock_join_kernel(const LineEnt* __restrict__ index, uint32_t mask,
                                                        SockRec* recs, const alz_sock_query* __restrict__ keys,
                                                        uint32_t n, uint64_t now, alz_l7_rec* __restrict__ l7,
                                                        unsigned long long* __restrict__ joined) {
  const uint32_t stride = gridDim.x * blockDim.x;
  uint32_t mine = 0;
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
    if (l7[i].saddr != 0u || l7[i].daddr != 0u) continue;
    uint32_t len;
    SockRec* v = const_cast<SockRec*>(find_line(index, mask, recs, keys[i].pid, keys[i].fd, &len));
    const SockRec* hit = get_value(v, len, keys[i].timestamp_ns, now);
    if (hit == nullptr) continue;
    l7[i].saddr = hit->saddr; l7[i].daddr = hit->daddr; l7[i].sport = hit->sport; l7[i].dport = hit->dport;
    ++mine;
  }
  if (mine) atomicAdd(joined, (unsigned long long)mine);
}

__device__ __forceinline__ void copy_rec(SockRec* dst, const SockRec* src) {
  const uint4 a = reinterpret_cast<const uint4*>(src)[0], b = reinterpret_cast<const uint4*>(src)[1];
  reinterpret_cast<uint4*>(dst)[0] = a; reinterpret_cast<uint4*>(dst)[1] = b;
}

// One warp per changed line: optional move of the segment, then the sorted inserts in arrival order (the
// tail of the line shifts up by one, top chunk first), then the index entry. LastMatch stamps stay with
// their records because the records are moved on the device, never re-uploaded.
__global__ void __launch_bounds__(128) sock_apply_kernel(const SockRec* __restrict__ src_pool, SockRec* dst_pool,
                                                         LineEnt* index, const LineDesc* __restrict__ descs,
                                                         const LineOp* __restrict__ ops, uint32_t n_desc) {
  const uint32_t lane = threadIdx.x & 31u;
  const uint32_t warps = (gridDim.x * blockDim.x) >> 5;
  for (uint32_t d = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; d < n_desc; d += warps) {
    const LineDesc L = descs[d];
    SockRec* v = dst_pool + L.dst_off;
    if (src_pool != dst_pool || L.src_off != L.dst_off) {
      const SockRec* from = src_pool + L.src_off;
      for (uint32_t i = lane; i < L.len_before; i += 32u) copy_rec(&v[i], &from[i]);
      __syncwarp();
    }
    uint32_t len = L.len_before;
    for (uint32_t k = 0; k < L.n_ops; ++k) {
      const LineOp* op = &ops[L.op_begin + k];
      const uint32_t pos = op->pos;
      for (uint32_t hi = len; hi > pos;) {
        const uint32_t span = min(32u, hi - pos);
        SockRec tmp;
        const bool on = lane < span;
        if (on) copy_rec(&tmp, &v[hi - 1u - lane]);
        __syncwarp();
        if (on) copy_rec(&v[hi - lane], &tmp);
        __syncwarp();
        hi -= span;
      }
      if (lane == 0) copy_rec(&v[pos], &op->rec);
      ++len;
      __syncwarp();
    }
    if (lane == 0) {
      LineEnt e;
      e.fd = L.fd; e.pid = L.pid; e.used = 1u; e.off = L.dst_off; e.len = len; e.pad = 0;
      index[L.slot] = e;
    }
  }
}

// sendOpenConnection (data.go:1628-1679) for every line: last value open, source a pod -> one row
__global__ void __launch_bounds__(256) sock_alive_kernel(const LineEnt* __restrict__ index, uint32_t cap,
                                                         const SockRec* __restrict__ recs,
                                                         const EpEntry* __restrict__ ep, uint32_t ep_mask,
                                                         alz_alive_conn* __restrict__ out, uint32_t out_cap,
                                                         uint32_t* __restrict__ n_out) {
  const uint32_t stride = gridDim.x * blockDim.x;
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < cap; i += stride) {
    const LineEnt e = index[i];
    if (!e.used || e.len == 0u) continue;                               // :1632-1634
    const SockRec t = recs[e.off + e.len - 1u];                         // values are sorted: the last one
    if (!t.open) continue;                                              // a close: ignored
    uint32_t pod, svc;
    if ((ep_lookup(ep, ep_mask, t.saddr, &pod, &svc) & kEpPod) == 0u) continue;   // :1643-1647
    alz_alive_conn c;
    c.from_ip = t.saddr; c.from_id = pod; c.from_port = t.sport;
    c.to_ip = t.daddr; c.to_port = t.dport;
    c._pad[0] = c._pad[1] = c._pad[2] = 0;
    const uint32_t d = ep_lookup(ep, ep_mask, t.daddr, &pod, &svc);
    if (d & kEpSvc) { c.to_type = ALZ_NODE_SVC; c.to_id = svc; }        // :1662-1665
    else if (d & kEpPod) { c.to_type = ALZ_NODE_POD; c.to_id = pod; }   // :1667-1670
    else { c.to_type = ALZ_NODE_OUTBOUND; c.to_id = t.daddr; }          // :1671-1674
    const uint32_t k = atomicAdd(n_out, 1u);
    if (k < out_cap) out[k] = c;
  }
}

struct Line {
  std::vector<SockRec> v;        // host mirror: timestamps and 5-tuples (AddValue's dedupe and insert position)
  std::vector<LineOp> ops;       // inserts since the last sync
  uint32_t off = 0, cap = 0;     // segment in the device pool
  uint32_t dev_len = 0;          // records the device has
  uint32_t slot = UINT32_MAX;    // index slot
  bool queued = false;
};
using LineMap = std::unordered_map<LineKey, Line, LineKeyHash>;

}  // namespace

struct alz_sock_state {
  Owned mem;                                 // ev_stage, d_joined, d_alive_n
  LineMap lines;
  std::vector<LineMap::value_type*> dirty;   // lines with pending ops (node addresses are stable)
  std::vector<LineEnt> h_index;              // host mirror of the index (keys and slots only)
  GrowBuf<LineEnt> d_index;
  uint32_t index_cap = 0;
  Owner d_pool;
  size_t pool_cap = 0, pool_used = 0, pool_garbage = 0;
  GrowBuf<char> h_stage{Res::kPinned};      // descs then ops of one sync
  GrowBuf<char> d_stage;
  cudaEvent_t ev_stage = nullptr;            // the H2D out of h_stage is done
  GrowBuf<alz_sock_query> d_q;
  GrowBuf<alz_sock_result> d_out;
  GrowBuf<alz_l7_rec> d_jrec;                // alz_submit_l7_join scratch
  GrowBuf<alz_sock_query> d_jkey;
  unsigned long long* d_joined = nullptr;
  GrowBuf<alz_alive_conn> d_alive;
  uint32_t* d_alive_n = nullptr;
  uint64_t syncs = 0, sync_ops = 0, sync_bytes = 0, repools = 0;
  SockRec* pool() const { return static_cast<SockRec*>(d_pool.get()); }
};
void StateDelete::operator()(alz_sock_state* s) const { delete s; }

static alz_sock_state* state_of(alz_handle* h) {
  if (!h->sock) h->sock.reset(new alz_sock_state());
  return h->sock.get();
}

static void enqueue(alz_sock_state* s, LineMap::value_type* node) {
  if (!node->second.queued) { node->second.queued = true; s->dirty.push_back(node); }
}

// SocketLine.AddValue: skip when equal to the last element's open socket, else sorted insert
static void add_value(alz_sock_state* s, LineMap::value_type* node, uint64_t ts, const alz_tcp_rec* si) {
  std::vector<SockRec>& v = node->second.v;
  if (!v.empty() && si != nullptr) {
    const SockRec& last = v.back();
    if (last.open && last.saddr == si->saddr && last.sport == si->sport && last.daddr == si->daddr &&
        last.dport == si->dport)
      return;                                                            // sock_num_line.go:70-78
  }
  size_t lo = 0, hi = v.size();                                          // insertIntoSortedSlice :311-322
  while (lo < hi) { const size_t mid = (lo + hi) / 2; if (v[mid].ts >= ts) hi = mid; else lo = mid + 1; }
  SockRec r;
  memset(&r, 0, sizeof r);
  r.ts = ts;
  if (si != nullptr) { r.open = 1; r.saddr = si->saddr; r.daddr = si->daddr; r.sport = si->sport; r.dport = si->dport; }
  v.insert(v.begin() + (ptrdiff_t)lo, r);
  LineOp op;
  memset(&op, 0, sizeof op);
  op.rec = r; op.pos = (uint32_t)lo;
  node->second.ops.push_back(op);
  enqueue(s, node);
}

extern "C" int alz_submit_tcp(alz_handle* h, const alz_tcp_rec* recs, size_t n) {
  if (!h || (!recs && n)) return ALZ_E_INVAL;
  std::lock_guard<std::mutex> g(h->mu);
  alz_sock_state* s = state_of(h);
  for (size_t i = 0; i < n; ++i) {
    const alz_tcp_rec& d = recs[i];
    h->tcp_events_in++;
    if (d.type != 1u && d.type != 5u) continue;                          // only ESTABLISHED / CLOSED are handled
    if (d.saddr == kLocalhost || d.daddr == kLocalhost) { h->tcp_localhost_dropped++; continue; }
    const LineKey k{d.pid, d.fd};
    if (d.type == 1u) {                                                  // EVENT_TCP_ESTABLISHED, data.go:406-449
      auto it = s->lines.try_emplace(k).first;                           // line created on first use (:417-437)
      add_value(s, &*it, d.timestamp_ns, &d);
    } else {                                                             // EVENT_TCP_CLOSED, :450-478
      auto it = s->lines.find(k);
      if (it == s->lines.end()) continue;                                // no line: ignored (:471-473)
      add_value(s, &*it, d.timestamp_ns, nullptr);
    }
  }
  return ALZ_OK;
}

// struct tcp_event (ebpf/c/struct.h:2-12): fd u64 @0, timestamp u64 @8, type u32 @16, pid u32 @20, sport u16 @24,
// dport u16 @26, saddr[16] @28, daddr[16] @44, padded to 64
extern "C" int alz_submit_tcp_raw(alz_handle* h, const void* raw, size_t n) {
  if (!h || (!raw && n)) return ALZ_E_INVAL;
  const uint8_t* p = static_cast<const uint8_t*>(raw);
  alz_tcp_rec buf[256];
  for (size_t done = 0; done < n;) {
    const size_t m = std::min<size_t>(256, n - done);
    for (size_t i = 0; i < m; ++i, p += ALZ_BPF_TCP_EVENT_SIZE) {
      alz_tcp_rec& r = buf[i];
      memset(&r, 0, sizeof r);
      memcpy(&r.fd, p, 8); memcpy(&r.timestamp_ns, p + 8, 8); memcpy(&r.type, p + 16, 4); memcpy(&r.pid, p + 20, 4);
      memcpy(&r.sport, p + 24, 2); memcpy(&r.dport, p + 26, 2);
      r.saddr = ((uint32_t)p[28] << 24) | ((uint32_t)p[29] << 16) | ((uint32_t)p[30] << 8) | p[31];   // tcp.go:241
      r.daddr = ((uint32_t)p[44] << 24) | ((uint32_t)p[45] << 16) | ((uint32_t)p[46] << 8) | p[47];   // tcp.go:242
    }
    const int rc = alz_submit_tcp(h, buf, m);
    if (rc != ALZ_OK) return rc;
    done += m;
  }
  return ALZ_OK;
}

static uint32_t pow2_at_least(size_t x) { uint32_t p = 16; while (p < x) p <<= 1; return p; }

static uint32_t seg_cap_for(size_t len) { return std::max<uint32_t>(8u, pow2_at_least(len + len / 2)); }

// Brings the device pool and index up to the host's lines. Work and bytes are proportional to the inserts
// since the last sync (the apply kernel shifts and moves on the device); the index is re-sent whole only
// when it doubles, the pool is re-laid only when it is full or half garbage.
static int sync_lines(alz_handle* h) {
  alz_sock_state* s = h->sock.get();
  if (s->dirty.empty()) return ALZ_OK;
  if (!s->ev_stage) CK(s->mem.event(&s->ev_stage, cudaEventDisableTiming));
  if (!s->d_joined) { CK(s->mem.dev(&s->d_joined, 8)); CK(cudaMemsetAsync(s->d_joined, 0, 8, h->stream)); }

  // 1. index: a slot for every new line; doubling rebuilds the mirror and re-sends it
  bool index_resend = false;
  if (s->lines.size() * 2 > s->index_cap) {
    const uint32_t cap = pow2_at_least(4 * s->lines.size() + 1);
    s->h_index.assign(cap, LineEnt{});
    for (auto& kv : s->lines) {
      Line& L = kv.second;
      uint32_t slot = line_slot(kv.first.pid, kv.first.fd, cap - 1);
      while (s->h_index[slot].used) slot = (slot + 1) & (cap - 1);
      LineEnt& e = s->h_index[slot];
      e.used = 1; e.pid = kv.first.pid; e.fd = kv.first.fd; e.off = L.off; e.len = L.dev_len;
      L.slot = slot;
    }
    CK(s->d_index.ensure(cap, h->stream));
    s->index_cap = cap;
    index_resend = true;
  } else {
    for (auto* node : s->dirty) {
      Line& L = node->second;
      if (L.slot != UINT32_MAX) continue;
      uint32_t slot = line_slot(node->first.pid, node->first.fd, s->index_cap - 1);
      while (s->h_index[slot].used) slot = (slot + 1) & (s->index_cap - 1);
      LineEnt& e = s->h_index[slot];
      e.used = 1; e.pid = node->first.pid; e.fd = node->first.fd;      // off/len live on the device
      L.slot = slot;
    }
  }

  // 2. segments: a line that outgrew its segment moves to a new one at the pool's tail
  size_t need = 0;
  for (auto* node : s->dirty) {
    Line& L = node->second;
    if (L.v.size() > L.cap) need += seg_cap_for(L.v.size());
  }
  const bool repool = s->pool_used + need > s->pool_cap ||
                      (s->pool_garbage > (1u << 16) && s->pool_garbage * 2 > s->pool_used);
  Owner old_pool;   // a repool's source: freed on return, after the apply kernel has read it
  std::vector<LineDesc> descs;
  std::vector<LineOp> ops;
  auto add_desc = [&](LineMap::value_type* node, uint32_t src_off) {
    Line& L = node->second;
    LineDesc d;
    d.fd = node->first.fd; d.pid = node->first.pid; d.slot = L.slot;
    d.src_off = src_off; d.dst_off = L.off; d.len_before = L.dev_len;
    d.op_begin = (uint32_t)ops.size(); d.n_ops = (uint32_t)L.ops.size(); d.pad = 0;
    ops.insert(ops.end(), L.ops.begin(), L.ops.end());
    descs.push_back(d);
    L.dev_len = (uint32_t)L.v.size();
    L.ops.clear(); L.ops.shrink_to_fit();
    L.queued = false;
  };
  if (repool) {
    size_t total = 0;
    for (auto& kv : s->lines) total += seg_cap_for(kv.second.v.size());
    const size_t cap = std::max<size_t>(1u << 16, total * 2);
    if (cap > 0xFFFFFFF0ull) return alz_error(h, ALZ_E_CAPACITY, "socket timelines", "more than 2^32 records");
    Owner fresh;
    CK(alz_alloc(fresh, Res::kDev, cap * sizeof(SockRec)));
    old_pool = std::move(s->d_pool);
    s->d_pool = std::move(fresh); s->pool_cap = cap; s->pool_used = 0; s->pool_garbage = 0;
    for (auto& kv : s->lines) {                                        // every line moves, on the device
      Line& L = kv.second;
      const uint32_t old_off = L.off;
      L.cap = seg_cap_for(L.v.size());
      L.off = (uint32_t)s->pool_used;
      s->pool_used += L.cap;
      add_desc(&kv, old_off);
    }
    s->repools++;
  } else {
    for (auto* node : s->dirty) {
      Line& L = node->second;
      const uint32_t old_off = L.off;
      if (L.v.size() > L.cap) {
        s->pool_garbage += L.cap;
        L.cap = seg_cap_for(L.v.size());
        L.off = (uint32_t)s->pool_used;
        s->pool_used += L.cap;
      }
      add_desc(node, old_off);
    }
  }
  s->dirty.clear();

  // 3. one staged copy, one kernel
  const size_t desc_bytes = (descs.size() * sizeof(LineDesc) + 15u) & ~(size_t)15u;
  const size_t bytes = desc_bytes + ops.size() * sizeof(LineOp);
  CK(s->h_stage.ensure(bytes, h->stream, bytes * 2));
  CK(s->d_stage.ensure(bytes, h->stream, bytes * 2));
  CK(cudaEventSynchronize(s->ev_stage));
  char* stage = s->h_stage.get();
  memcpy(stage, descs.data(), descs.size() * sizeof(LineDesc));
  if (!ops.empty()) memcpy(stage + desc_bytes, ops.data(), ops.size() * sizeof(LineOp));
  if (index_resend)
    CK(cudaMemcpyAsync(s->d_index.get(), s->h_index.data(), (size_t)s->index_cap * sizeof(LineEnt), cudaMemcpyHostToDevice,
                       h->stream));
  CK(cudaMemcpyAsync(s->d_stage.get(), stage, bytes, cudaMemcpyHostToDevice, h->stream));
  CK(cudaEventRecord(s->ev_stage, h->stream));
  const unsigned blocks = (unsigned)std::min<size_t>((descs.size() + 3) / 4, (size_t)h->sms * 8);
  sock_apply_kernel<<<std::max(1u, blocks), 128, 0, h->stream>>>(
      old_pool ? static_cast<SockRec*>(old_pool.get()) : s->pool(), s->pool(), s->d_index.get(),
      (const LineDesc*)s->d_stage.get(), (const LineOp*)(s->d_stage.get() + desc_bytes), (uint32_t)descs.size());
  CK(cudaGetLastError());
  h->launches++;
  s->syncs++; s->sync_ops += ops.size();
  s->sync_bytes += bytes + (index_resend ? (size_t)s->index_cap * sizeof(LineEnt) : 0);
  if (index_resend) CK(cudaStreamSynchronize(h->stream));   // h_index is pageable
  if (old_pool) CK(cudaStreamSynchronize(h->stream));
  return ALZ_OK;
}

static uint64_t wall_ns() {
  timespec ts;
  clock_gettime(CLOCK_REALTIME, &ts);
  return (uint64_t)ts.tv_sec * 1000000000ull + (uint64_t)ts.tv_nsec;
}

extern "C" int alz_sock_lookup_at(alz_handle* h, const alz_sock_query* q, size_t n, alz_sock_result* out,
                                  uint64_t now_ns) {
  if (!h || (!q && n) || (!out && n)) return ALZ_E_INVAL;
  if (n == 0) return ALZ_OK;
  if (n > 0xFFFFFFFFull) return ALZ_E_INVAL;
  std::lock_guard<std::mutex> g(h->mu);
  CK(cudaSetDevice(h->device));
  alz_sock_state* s = state_of(h);
  int rc = sync_lines(h);
  if (rc != ALZ_OK) return rc;
  if (s->index_cap == 0) { memset(out, 0, n * sizeof(alz_sock_result)); return ALZ_OK; }   // no line yet
  CK(s->d_q.ensure(n, h->stream));
  CK(s->d_out.ensure(n, h->stream));
  CK(cudaMemcpyAsync(s->d_q.get(), q, n * sizeof(alz_sock_query), cudaMemcpyHostToDevice, h->stream));
  sock_lookup_kernel<<<(unsigned)h->sms * 4, 256, 0, h->stream>>>(s->d_index.get(), s->index_cap - 1, s->pool(),
                                                                s->d_q.get(), (uint32_t)n, now_ns, s->d_out.get());
  CK(cudaGetLastError());
  h->launches++;
  CK(cudaMemcpyAsync(out, s->d_out.get(), n * sizeof(alz_sock_result), cudaMemcpyDeviceToHost, h->stream));
  CK(cudaStreamSynchronize(h->stream));
  return ALZ_OK;
}

extern "C" int alz_sock_lookup(alz_handle* h, const alz_sock_query* q, size_t n, alz_sock_result* out) {
  return alz_sock_lookup_at(h, q, n, out, wall_ns());   // LastMatch = time.Now() (sock_num_line.go:96, :156)
}

// L7 events with (pid, fd) keys: the zero 5-tuples are filled from the timelines on the device, then the
// batch takes the normal ingest path. host_keys[i].timestamp_ns = the event's WriteTimeNs (data.go:1424).
extern "C" int alz_submit_l7_join(alz_handle* h, const alz_l7_rec* recs, const alz_sock_query* keys, size_t n,
                                  uint64_t now_ns) {
  if (!h || ((!recs || !keys) && n)) return ALZ_E_INVAL;
  if (n == 0) return ALZ_OK;
  std::lock_guard<std::mutex> g(h->mu);
  CK(cudaSetDevice(h->device));
  alz_sock_state* s = state_of(h);
  int rc = sync_lines(h);
  if (rc != ALZ_OK) return rc;
  if (!s->d_joined) { CK(s->mem.dev(&s->d_joined, 8)); CK(cudaMemsetAsync(s->d_joined, 0, 8, h->stream)); }
  const size_t per = h->cfg.max_batch;
  CK(s->d_jrec.ensure(per, h->stream));
  CK(s->d_jkey.ensure(per, h->stream));
  if (now_ns == 0) now_ns = wall_ns();
  for (size_t done = 0; done < n; done += per) {
    const size_t m = std::min(per, n - done);
    CK(cudaMemcpyAsync(s->d_jrec.get(), recs + done, m * sizeof(alz_l7_rec), cudaMemcpyHostToDevice, h->stream));
    CK(cudaMemcpyAsync(s->d_jkey.get(), keys + done, m * sizeof(alz_sock_query), cudaMemcpyHostToDevice, h->stream));
    if (s->index_cap != 0) {
      sock_join_kernel<<<(unsigned)h->sms * 4, 256, 0, h->stream>>>(s->d_index.get(), s->index_cap - 1, s->pool(),
                                                                  s->d_jkey.get(), (uint32_t)m, now_ns, s->d_jrec.get(),
                                                                  s->d_joined);
      CK(cudaGetLastError());
      h->launches++;
    }
    rc = alz_internal_ingest(h, s->d_jrec.get(), m);
    if (rc != ALZ_OK) return rc;
    CK(cudaStreamSynchronize(h->stream));   // one scratch buffer; the caller's arrays may be pageable
  }
  return ALZ_OK;
}

// SocketLine.DeleteUnused (sock_num_line.go:160-209) on one line, restated as written — including that its
// first loop stops before the last element, so a line that does not end in two opens loses its last value.
static bool delete_unused(std::vector<SockRec>& v) {
  if (v.size() <= 1) return false;                                       // :165-167
  std::vector<SockRec> res;
  res.reserve(v.size());
  size_t i = 0;
  while (i < v.size() - 1) {                                             // :172-181
    if (v[i].open && v[i + 1].open) { res.push_back(v[i + 1]); i += 2; }
    else { res.push_back(v[i]); i += 1; }
  }
  uint64_t last_matched = 0;                                             // :184-190
  for (const SockRec& r : res) if (r.lm != 0 && r.lm > last_matched) last_matched = r.lm;
  for (ptrdiff_t k = (ptrdiff_t)res.size() - 1; k >= 1; --k) {           // :197-208
    if (!res[k].open && res[k - 1].open && res[k - 1].lm + kFiveMinutesNs < last_matched) {
      res.erase(res.begin() + (k - 1), res.begin() + (k + 1));
      --k;
    }
  }
  v.swap(res);
  return true;
}

// One tick of clearSocketLines (data.go:1681-1716): DeleteUnused on every line. The LastMatch stamps live on
// the device (the lookups write them), so the pool is read back once; changed lines are re-sent whole.
extern "C" int alz_sock_gc(alz_handle* h) {
  if (!h) return ALZ_E_INVAL;
  std::lock_guard<std::mutex> g(h->mu);
  CK(cudaSetDevice(h->device));
  alz_sock_state* s = state_of(h);
  int rc = sync_lines(h);
  if (rc != ALZ_OK) return rc;
  if (s->pool_used == 0) return ALZ_OK;
  std::vector<SockRec> pool(s->pool_used);
  CK(cudaMemcpyAsync(pool.data(), s->pool(), s->pool_used * sizeof(SockRec), cudaMemcpyDeviceToHost, h->stream));
  CK(cudaStreamSynchronize(h->stream));
  for (auto& kv : s->lines) {
    Line& L = kv.second;
    for (size_t i = 0; i < L.v.size(); ++i) L.v[i].lm = pool[L.off + i].lm;
    if (!delete_unused(L.v)) continue;
    // re-send: the line restarts empty on the device and its records arrive as appends (with their stamps)
    L.dev_len = 0;
    L.ops.clear();
    for (size_t i = 0; i < L.v.size(); ++i) {
      LineOp op;
      memset(&op, 0, sizeof op);
      op.rec = L.v[i]; op.pos = (uint32_t)i;
      L.ops.push_back(op);
    }
    enqueue(s, &kv);
  }
  return sync_lines(h);
}

extern "C" int alz_sock_alive(alz_handle* h, alz_alive_conn* out, size_t cap, size_t* n_out) {
  if (!h || !n_out || (!out && cap)) return ALZ_E_INVAL;
  std::lock_guard<std::mutex> g(h->mu);
  CK(cudaSetDevice(h->device));
  alz_sock_state* s = state_of(h);
  int rc = sync_lines(h);
  if (rc != ALZ_OK) return rc;
  *n_out = 0;
  if (s->index_cap == 0) return ALZ_OK;
  if (!s->d_alive_n) CK(s->mem.dev(&s->d_alive_n, 4));
  CK(s->d_alive.ensure(cap, h->stream));
  CK(cudaMemsetAsync(s->d_alive_n, 0, 4, h->stream));
  sock_alive_kernel<<<(unsigned)h->sms * 4, 256, 0, h->stream>>>(s->d_index.get(), s->index_cap, s->pool(), h->d_ep,
                                                               h->ep_cap - 1, s->d_alive.get(),
                                                               (uint32_t)std::min<size_t>(cap, 0xFFFFFFFFu), s->d_alive_n);
  CK(cudaGetLastError());
  h->launches++;
  uint32_t cnt = 0;
  CK(cudaMemcpyAsync(&cnt, s->d_alive_n, 4, cudaMemcpyDeviceToHost, h->stream));
  CK(cudaStreamSynchronize(h->stream));
  *n_out = cnt;                                                          // the number there are
  const size_t take = std::min<size_t>(cnt, cap);
  if (take) CK(cudaMemcpy(out, s->d_alive.get(), take * sizeof(alz_alive_conn), cudaMemcpyDeviceToHost));
  return cnt > cap ? ALZ_E_CAPACITY : ALZ_OK;
}

extern "C" int alz_sock_stats(alz_handle* h, alz_sock_stats_t* st) {
  if (!h || !st) return ALZ_E_INVAL;
  std::lock_guard<std::mutex> g(h->mu);
  memset(st, 0, sizeof *st);
  alz_sock_state* s = h->sock.get();
  if (!s) return ALZ_OK;
  CK(cudaSetDevice(h->device));
  st->lines = s->lines.size();
  st->pool_records = s->pool_used;
  st->pool_garbage = s->pool_garbage;
  st->syncs = s->syncs;
  st->sync_ops = s->sync_ops;
  st->sync_bytes = s->sync_bytes;
  st->repools = s->repools;
  if (s->d_joined) {
    unsigned long long j = 0;
    CK(cudaMemcpyAsync(&j, s->d_joined, 8, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    st->joined_events = j;
  }
  return ALZ_OK;
}
