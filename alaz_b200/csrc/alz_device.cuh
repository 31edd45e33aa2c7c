// alz_device.cuh — device-side building blocks of libalazgpu (sm_100a).
//
// Semantics restated from the reference (file:line = getanteon/alaz @ 828b997f):
//   row-emit rule      aggregator/data.go:1364-1383 (processL7 switch), :1252-1255,
//                      :1288-1292, :1328-1332 (payload parse failure => no row)
//   direction reversal aggregator/data.go:1110-1112 (AMQP DELIVER), :1151-1153
//                      (REDIS PUSHED_EVENT); datastore/dto.go:246-251
//   resolve            aggregator/data.go:827-870 (setFromToV2)
// Everything else (edge key, buckets, accumulators) is docs/SPEC.md.
#pragma once
#include <cstdint>
#include <cuda_runtime.h>
#include "../../include/alazgpu.h"

namespace alz {

constexpr uint64_t kEmptyKey = ~0ull;   // open-addressing empty marker (u64 tables)
constexpr uint32_t kMaxProbe = 4096;    // linear-probe bound before "capacity"

// ---- endpoint table: the join's build side, one entry per IPv4 ---------------
// (ClusterInfo.PodIPToPodUid + ServiceIPToServiceUid, aggregator/cluster.go:15-16,
// merged: one probe answers "is it a pod" and "is it a service")
struct __align__(16) EpEntry {
  uint32_t ip;
  uint32_t state;  // bit0 occupied, bit1 has pod id, bit2 has service id
  uint32_t pod;
  uint32_t svc;
};
constexpr uint32_t kEpOcc = 1u, kEpPod = 2u, kEpSvc = 4u;

// Filter of the pod addresses (two bits per address out of hash32): the ingest kernel keeps a copy in shared memory
// and drops an event whose source cannot be a pod without touching the dictionary (alz_ingest.cu). The host keeps
// counters per bit so that deletes are exact (alz_api.cu). A cluster far larger than the filter just saturates it.
#define ALZ_BLOOM_WORDS 4096u   /* 128 Kbit */

__host__ __device__ __forceinline__ uint32_t hash32(uint32_t x) {
  x ^= x >> 16; x *= 0x85EBCA6Bu; x ^= x >> 13; x *= 0xC2B2AE35u; x ^= x >> 16;
  return x;
}
__host__ __device__ __forceinline__ uint64_t hash64(uint64_t x) {
  x ^= x >> 33; x *= 0xFF51AFD7ED558CCDull; x ^= x >> 33; x *= 0xC4CEB9FE1A85EC53ull; x ^= x >> 33;
  return x;
}

// rank that owns an event (alz_owner_rank): a function of the source address only
__host__ __device__ __forceinline__ uint32_t owner_rank(uint32_t saddr, uint32_t nranks) {
  if (nranks <= 1u) return 0u;
  return (uint32_t)(((uint64_t)hash32(saddr ^ 0xA1A2B200u) * nranks) >> 32);
}

// Socket-pair key of the pair dictionaries: daddr in the high word, saddr in the low word — the order the two
// words have in a record, so a record's first 8 bytes ARE its key (no shuffling in the per-event path).
__host__ __device__ __forceinline__ uint64_t make_pair_key(uint32_t saddr, uint32_t daddr) { return ((uint64_t)daddr << 32) | saddr; }
__host__ __device__ __forceinline__ uint32_t pair_saddr(uint64_t key) { return (uint32_t)key; }
__host__ __device__ __forceinline__ uint32_t pair_daddr(uint64_t key) { return (uint32_t)(key >> 32); }

// cheap 32-bit hash of a socket pair for the pair dictionaries and the per-CTA table (the per-event
// path pays for this once; hash64 costs two 64-bit multiplies)
__host__ __device__ __forceinline__ uint32_t pair_hash(uint64_t key) {
  uint32_t h = (uint32_t)(key >> 32) * 0x9E3779B1u ^ (uint32_t)key * 0x85EBCA6Bu;
  h ^= h >> 15; h *= 0x2C1B3C6Du; h ^= h >> 13;
  return h;
}

// ---- packed edge key (docs/SPEC.md §3) -----------------------------------------
// One end of every edge is the pod that setFromToV2 resolved from saddr.
//   bit 63      rev: 0 = pod is From, 1 = pod is To (row was reversed)
//   bits 62..61 type of the other end (ALZ_NODE_*)
//   bits 60..32 pod id (< 2^29)
//   bits 31..0  other end: pod/service id, or raw IPv4 for outbound
// Canonical form: a reversed pod<->pod row is stored with rev = 0 and the ends
// swapped, so equal (From,To) always give equal keys.
__host__ __device__ __forceinline__ uint64_t make_edge_key(uint32_t pod_id, uint32_t other_type,
                                                           uint32_t other, bool rev) {
  if (rev && other_type == ALZ_NODE_POD) { uint32_t t = pod_id; pod_id = other; other = t; rev = false; }
  return ((uint64_t)(rev ? 1u : 0u) << 63) | ((uint64_t)other_type << 61) |
         ((uint64_t)(pod_id & 0x1FFFFFFFu) << 32) | (uint64_t)other;
}
__host__ __device__ __forceinline__ void unpack_edge_key(uint64_t k, uint8_t* from_type, uint32_t* from,
                                                         uint8_t* to_type, uint32_t* to) {
  const bool rev = (k >> 63) != 0;
  const uint8_t ot = (uint8_t)((k >> 61) & 3u);
  const uint32_t pod = (uint32_t)((k >> 32) & 0x1FFFFFFFu);
  const uint32_t other = (uint32_t)k;
  if (!rev) { *from_type = ALZ_NODE_POD; *from = pod; *to_type = ot; *to = other; }
  else      { *from_type = ot; *from = other; *to_type = ALZ_NODE_POD; *to = pod; }
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

// ---- per-record rules ------------------------------------------------------------
// Does processL7 hand a row to PersistRequest for this record (before resolve)?
__host__ __device__ __forceinline__ bool emits_request_row(uint32_t protocol, uint32_t method_flags) {
  switch (protocol) {
    case ALZ_PROTO_HTTP: case ALZ_PROTO_AMQP: case ALZ_PROTO_REDIS:
      return true;
    case ALZ_PROTO_POSTGRES: case ALZ_PROTO_MYSQL: case ALZ_PROTO_MONGO:
      return (method_flags & ALZ_MF_PAYLOAD_REJECT) == 0;
    default:  // HTTP2 (frame pairing), KAFKA (PersistKafkaEvent), UNKNOWN
      return false;
  }
}
__host__ __device__ __forceinline__ bool is_reversed(uint32_t protocol, uint32_t method_flags) {
  const uint32_t m = method_flags & ALZ_MF_METHOD_MASK;
  return (protocol == ALZ_PROTO_AMQP && m == ALZ_AMQP_DELIVER) ||
         (protocol == ALZ_PROTO_REDIS && m == ALZ_REDIS_PUSHED_EVENT);
}
// Protocol is "HTTP" or "HTTPS" (HTTPS = HTTP && tls, data.go:1240-1242)
__host__ __device__ __forceinline__ bool is_5xx(uint32_t protocol, uint32_t status) {
  return protocol == ALZ_PROTO_HTTP && status >= 500u && status < 600u;
}
// docs/SPEC.md §4: two sub-buckets per octave over [2^8, 2^40), clamped
__device__ __forceinline__ uint32_t latency_bucket(uint64_t d) {
  if (d < 256ull) return 0u;
  const uint32_t o = 63u - (uint32_t)__clzll((long long)d);
  if (o >= 40u) return ALZ_NB - 1u;
  return 2u * (o - 8u) + (uint32_t)((d >> (o - 1u)) & 1ull);
}

// ---- open-addressed u64 dictionary -> dense accumulator rows ---------------------------
// The dictionary only maps a key to a row number; rows are handed out densely
// by an atomic counter, so the accumulators of the live keys stay contiguous
// (190k live pairs x 280 B = 53 MB: L2-resident) however large the dictionary
// was sized. v1 indexed the accumulators by dictionary slot and every
// reduction missed L2 (profiles/r1_v2_ingest_ncu.txt: 11 GB DRAM reads for a
// 3.2 GB stream).
struct __align__(16) DictEnt {
  uint64_t key;   // kEmptyKey = free
  uint32_t row;   // kNoRow until the inserting thread has published it
  uint32_t pad;
};
constexpr uint32_t kNoRow = 0xFFFFFFFFu;
constexpr uint32_t kLostRow = 0xFFFFFFFEu;  // dictionary or row pool exhausted

constexpr uint32_t kPairFwd = 0u, kPairRev = 1u, kPairHost = 2u, kPairKinds = 3u;

struct AccTable {
  DictEnt* dict;      // [dict_mask + 1]   (= dicts[kPairFwd])
  uint32_t dict_mask;
  // pair table only: further dictionaries for the socket pairs of reversed rows (kind 1: AMQP DELIVER, REDIS
  // PUSHED_EVENT) and for host-keyed outbound events (kind 2: the key's high word is a Host-header id, not a
  // daddr; ALZ_PROTO_F_HOSTKEY). All dictionaries hand out rows of the same pool; row_kind[row] says which one.
  DictEnt* dict_rev;
  uint32_t dict_rev_mask;
  DictEnt* dict_host;
  uint32_t dict_host_mask;
  __device__ __forceinline__ DictEnt* dict_of(uint32_t kind) const {
    return kind == kPairFwd ? dict : kind == kPairRev ? dict_rev : dict_host;
  }
  __device__ __forceinline__ uint32_t mask_of(uint32_t kind) const {
    return kind == kPairFwd ? dict_mask : kind == kPairRev ? dict_rev_mask : dict_host_mask;
  }
  uint32_t max_rows;  // rows [0, max_rows) are allocatable; rows max_rows + kind are the sentinel rows of the key that
                      // equals the free marker (one per kind); every per-row array has max_rows + kPairKinds entries
  uint32_t* n_rows;   // device counter of allocated rows
  uint64_t* row_key;  // [max_rows + 3]
  uint8_t* row_kind;  // [max_rows + 3] (pair table only) kPairFwd / kPairRev / kPairHost
  uint64_t* lat_sum;  // [max_rows + 3]
  uint64_t* err5xx;   // [max_rows + 3]
  uint64_t* count;    // [max_rows + 3] (edge table only; the pair table derives it from hist)
  uint32_t* row_cnt;  // [max_rows + 3] (pair table only) events of the row at the last fold, saturated
  uint8_t* row_base;  // [max_rows + 3] (pair table only) first bucket / 4 of the 16-bucket window that held most of
                      // the row's events at the last fold (the per-CTA table keeps only such a window per pair)
  uint32_t* row_aux;  // [max_rows + 3] (pair table only) edge row found by fold_resolve_kernel
  uint32_t* hist;     // [(max_rows + 3) * ALZ_NB] (edge table only)
  // Pair table rows are kept in 32-byte SECTORS, 16 per row (512 B): sector g = { cells 4g, 4g+1 | cells 4g+2, 4g+3 |
  // latency partial u64 | 5xx partial u64 }. A global reduction costs the SM one LSU pass per distinct sector an
  // instruction touches, not per lane (scripts/micro/red_merge.cu on B200: a histogram increment and a latency add as
  // two instructions = 93 G events/s chip-wide whether or not they share a sector; as ONE red.u64 instruction with two
  // lanes on the same sector = 172 G/s, the price of a single reduction, 188 G/s). So an event's cell and latency live
  // in one sector and are added by a lane pair of one instruction; a row's latency / 5xx totals are the sums of its 16
  // partials (fold_pairs_kernel). A cell pair is added to as a u64: cells are u32 and a fold runs before any cell
  // could reach 2^31 (alz_api.cu), so nothing carries from the low cell into the high one.
  uint64_t* sect;     // [(max_rows + 3) * kSectPerRow * 4] (pair table only; hist / lat_sum / err5xx are null there)
};
constexpr uint32_t kSectPerRow = 16;
__device__ __forceinline__ uint64_t* pair_sect(const AccTable& t, uint32_t row, uint32_t bucket) {
  return t.sect + ((size_t)row * kSectPerRow + (bucket >> 2)) * 4u;
}
__device__ __forceinline__ uint32_t* pair_cell(const AccTable& t, uint32_t row, uint32_t bucket) {
  return reinterpret_cast<uint32_t*>(pair_sect(t, row, bucket)) + (bucket & 3u);
}

// row of `key`, inserting it if absent; >= kLostRow when capacity is exhausted
__device__ __forceinline__ uint32_t find_or_insert(const AccTable& t, uint64_t key) {
  if (key == kEmptyKey) return t.max_rows;  // the one key that collides with the free marker
  uint32_t slot = (uint32_t)hash64(key) & t.dict_mask;
#pragma unroll 1
  for (uint32_t p = 0; p < kMaxProbe; ++p) {
    const uint4 e = __ldcg(reinterpret_cast<const uint4*>(&t.dict[slot]));
    uint64_t k = ((uint64_t)e.y << 32) | e.x;
    uint32_t row = e.z;
    if (k == kEmptyKey) {
      const uint64_t old = atomicCAS((unsigned long long*)&t.dict[slot].key, (unsigned long long)kEmptyKey,
                                     (unsigned long long)key);
      if (old == kEmptyKey) {
        row = atomicAdd(t.n_rows, 1u);
        if (row >= t.max_rows) row = kLostRow; else t.row_key[row] = key;
        *reinterpret_cast<volatile uint32_t*>(&t.dict[slot].row) = row;
        return row;
      }
      k = old;
      row = kNoRow;
    }
    if (k == key) {
      while (row == kNoRow) row = *reinterpret_cast<volatile uint32_t*>(&t.dict[slot].row);
      return row;
    }
    slot = (slot + 1u) & t.dict_mask;
  }
  return kLostRow;
}

// probe the endpoint table; returns state bits (0 = absent) and ids
__device__ __forceinline__ uint32_t ep_lookup(const EpEntry* __restrict__ tab, uint32_t mask, uint32_t ip,
                                              uint32_t* pod, uint32_t* svc) {
  uint32_t slot = hash32(ip) & mask;
  for (;;) {
    const uint4 e = __ldg(reinterpret_cast<const uint4*>(&tab[slot]));
    if ((e.y & kEpOcc) == 0u) return 0u;
    if (e.x == ip) { *pod = e.z; *svc = e.w; return e.y; }
    slot = (slot + 1u) & mask;
  }
}

// Pair-dictionary insert with the drop rule applied at admission: a NEW socket pair is only
// inserted if its source address is a pod right now (setFromToV2's first test, data.go:829-832).
// Unresolvable traffic is often high-cardinality (every event a new pair); letting it into the
// dictionary cost a CAS, a row and two DRAM-missing reductions per event
// (profiles/r1_v4_ingest_ncu.txt: 890k row allocations per 100M events, 190k of them real).
// Existing pairs are found without touching the endpoint table. Returns kDropRow for a rejected pair.
constexpr uint32_t kDropRow = 0xFFFFFFFDu;
__device__ __forceinline__ uint32_t find_or_insert_pair(const AccTable& t, uint64_t key, uint32_t kind,
                                                        const EpEntry* __restrict__ ep, uint32_t ep_mask) {
  // the one key that collides with the free marker has a fixed row per kind
  if (key == kEmptyKey) return t.max_rows + kind;
  DictEnt* const dict = t.dict_of(kind);
  const uint32_t mask = t.mask_of(kind);
  uint32_t slot = pair_hash(key) & mask;
  bool checked = false;
#pragma unroll 1
  for (uint32_t p = 0; p < kMaxProbe; ++p) {
    const uint4 e = __ldcg(reinterpret_cast<const uint4*>(&dict[slot]));
    uint64_t k = ((uint64_t)e.y << 32) | e.x;
    uint32_t row = e.z;
    if (k == kEmptyKey) {
      if (!checked) {
        uint32_t pod, svc;
        if ((ep_lookup(ep, ep_mask, pair_saddr(key), &pod, &svc) & kEpPod) == 0u) return kDropRow;
        checked = true;
      }
      const uint64_t old = atomicCAS((unsigned long long*)&dict[slot].key, (unsigned long long)kEmptyKey,
                                     (unsigned long long)key);
      if (old == kEmptyKey) {
        row = atomicAdd(t.n_rows, 1u);
        if (row >= t.max_rows) row = kLostRow; else { t.row_key[row] = key; t.row_kind[row] = (uint8_t)kind; }
        *reinterpret_cast<volatile uint32_t*>(&dict[slot].row) = row;
        return row;
      }
      k = old;
      row = kNoRow;
    }
    if (k == key) {
      while (row == kNoRow) row = *reinterpret_cast<volatile uint32_t*>(&dict[slot].row);
      return row;
    }
    slot = (slot + 1u) & mask;
  }
  return kLostRow;
}

// setFromToV2 on integers: false = "error finding pod with sockets saddr" (drop)
__device__ __forceinline__ bool resolve_edge(const EpEntry* __restrict__ tab, uint32_t mask, uint32_t saddr,
                                             uint32_t daddr, bool rev, uint64_t* edge_key) {
  uint32_t pod, svc;
  const uint32_t s = ep_lookup(tab, mask, saddr, &pod, &svc);
  if ((s & kEpPod) == 0u) return false;                 // data.go:829-832
  const uint32_t from_pod = pod;
  const uint32_t d = ep_lookup(tab, mask, daddr, &pod, &svc);
  uint32_t ot, ov;
  if (d & kEpSvc) { ot = ALZ_NODE_SVC; ov = svc; }       // :840-843 service first
  else if (d & kEpPod) { ot = ALZ_NODE_POD; ov = pod; }  // :845-849
  else { ot = ALZ_NODE_OUTBOUND; ov = daddr; }           // :862 raw daddr
  *edge_key = make_edge_key(from_pod, ot, ov, rev);
  return true;
}

// host-keyed outbound pair (ALZ_PROTO_F_HOSTKEY): the caller has already established that the destination is
// neither service nor pod, and HTTP rows are never reversed; only the drop rule is left (data.go:829-832, :851-854)
__device__ __forceinline__ bool resolve_edge_hostkey(const EpEntry* __restrict__ tab, uint32_t mask, uint32_t saddr,
                                                     uint32_t host_id, uint64_t* edge_key) {
  uint32_t pod, svc;
  if ((ep_lookup(tab, mask, saddr, &pod, &svc) & kEpPod) == 0u) return false;
  *edge_key = make_edge_key(pod, ALZ_NODE_OUTBOUND_HOST, host_id, false);
  return true;
}

// 32-byte record, one 256-bit load (LDG.E.256 on sm_100a), streaming: bypass L1
struct Rec { uint32_t w[8]; };
__device__ __forceinline__ Rec load_rec(const alz_l7_rec* p) {
  Rec r;
  asm volatile("ld.global.nc.L1::no_allocate.v8.u32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
               : "=r"(r.w[0]), "=r"(r.w[1]), "=r"(r.w[2]), "=r"(r.w[3]),
                 "=r"(r.w[4]), "=r"(r.w[5]), "=r"(r.w[6]), "=r"(r.w[7])
               : "l"(p));
  return r;
}
// field accessors of the packed words (layout of alz_l7_rec)
__device__ __forceinline__ uint32_t rec_saddr(const Rec& r) { return r.w[0]; }
__device__ __forceinline__ uint32_t rec_daddr(const Rec& r) { return r.w[1]; }
__device__ __forceinline__ uint32_t rec_status(const Rec& r) { return r.w[3] & 0xFFFFu; }
__device__ __forceinline__ uint32_t rec_protocol(const Rec& r) { return (r.w[3] >> 16) & 0x3Fu; }   // without the flag bits
__device__ __forceinline__ bool rec_hostkey(const Rec& r) { return (r.w[3] & ((uint32_t)ALZ_PROTO_F_HOSTKEY << 16)) != 0u; }
__device__ __forceinline__ uint32_t rec_mflags(const Rec& r) { return r.w[3] >> 24; }
__device__ __forceinline__ uint64_t rec_duration(const Rec& r) { return ((uint64_t)r.w[5] << 32) | r.w[4]; }

// ---- hot-pair feedback (alz_ingest.cu): which socket pairs took the most events last fold ----
constexpr int kHotMax = 4096;   // capacity of the list; the ingest kernel preloads as many as its table takes
struct HotState {
  uint32_t bins[128];          // quarter-octave histogram of per-pair event counts (forward pairs)
  uint32_t thr_a, thr_b;       // lowest bin of tier A (hottest, listed first) / of tier B
  uint32_t n_a, n_b;           // tier A occupies keys[0, n_a), tier B keys[kHotA, kHotA + n_b)
  uint64_t keys[kHotMax];
  uint8_t base[kHotMax];       // the pair's histogram window (first bucket / 4), see AccTable::row_base
  // tier S: the (at most) kHotS hottest pairs of all. The per-CTA table gives each of them kHotRep rows and a lane
  // uses row (lane % kHotRep) of the group: when one pair is most of a GPU's traffic — the rank that owns the
  // hottest pair of a sharded stream sees it in every second event — its reductions would otherwise pile up on
  // one shared-memory word and serialise (8 GPUs, config 2: that rank's ingest 2.2 ms against 1.13 ms elsewhere)
  uint32_t thr_s, n_s;
  uint64_t skeys[8];
  uint8_t sbase[8];
};
constexpr int kHotA = 64;
constexpr int kHotS = 8, kHotRep = 8;
// monotone bin of a count >= 1: 4 bins per octave
__device__ __forceinline__ uint32_t count_bin(uint32_t c) {
  const uint32_t o = 31u - (uint32_t)__clz((int)c);
  const uint32_t sub = o >= 2u ? (c >> (o - 2u)) & 3u : (c << (2u - o)) & 3u;
  return o * 4u + sub;
}

// device-side counters (per handle)
struct Counters {
  unsigned long long not_request;
  unsigned long long src_unresolved;
  unsigned long long capacity_events;   // events lost at ingest to an exhausted pair dictionary / row pool
  unsigned long long fold_lost_events;  // events lost at fold to an exhausted edge dictionary / row pool
  uint32_t pair_rows, edge_rows;            // row allocators of the two tables
  uint32_t defer_count, pad1;               // time-cut windows: records waiting for their window (alz_ingest.cu)
  unsigned long long late_events;           // time-cut windows: records older than the open window (reduced into it)
  unsigned long long pad2;
};

}  // namespace alz
