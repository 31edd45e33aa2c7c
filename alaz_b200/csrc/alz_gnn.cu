// alz_gnn.cu — GNN anomaly pass over the flushed service graph (docs/SPEC.md §6;
// not in the reference: north_star's extension). 2-layer GraphSAGE-mean, d = 64,
// fixed seeded weights, per-edge score.
//
//   nodes   : 2 node keys per edge -> sort -> unique (ascending (kind,value))
//   stats   : per-node in/out count, 5xx, latency sum, degree  (u64 atomics: exact,
//             order-independent, so the float features are deterministic)
//   CSR     : in-edges grouped by destination (stable sort by dst index, row
//             offsets = exclusive scan of the in-degrees)
//   layer   : mean of the in-neighbours' rows (coalesced 256-B row reads) ->
//             [h_v || m_v] (128) x W (128 x 64) + b, ReLU; the GEMM runs on tcgen05
//             (sage_layer_tc_kernel, 3xTF32), an FP32 FFMA version is kept for comparison
//   score   : sigma(a . [h2_u || h2_v || e_uv] + c), e_uv from the edge's
//             integers and float64 histogram quantiles
#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <string>
#include <mutex>
#include <vector>

#include "alz_handle.h"

using namespace alz;

namespace {

constexpr int D = 64;
constexpr uint64_t kGnnSeed = 0xA1A26E6Eull;

// ---- weights: pure integer -> double -> float, restated in tests/gnn_ref.py -----
inline double unit(uint64_t idx) {
  const uint64_t r = alz_splitmix64(kGnnSeed + idx);
  return (double)(r >> 11) * (1.0 / 9007199254740992.0) * 2.0 - 1.0;   // [-1, 1)
}

struct Weights {
  std::vector<float> W[2], b[2], a;   // W[l][k*64 + j], k in [0,128)
  float c;
};
Weights make_weights() {
  Weights w;
  const double sw = 1.0 / std::sqrt(128.0), sa = 1.0 / std::sqrt(132.0);
  uint64_t idx = 0;
  for (int l = 0; l < 2; ++l) {
    w.W[l].resize(128 * D);
    w.b[l].resize(D);
    for (int k = 0; k < 128; ++k)
      for (int j = 0; j < D; ++j) w.W[l][k * D + j] = (float)(unit(idx++) * sw);
    for (int j = 0; j < D; ++j) w.b[l][j] = (float)(unit(idx++) * 0.01);
  }
  w.a.resize(132);
  for (int k = 0; k < 132; ++k) w.a[k] = (float)(unit(idx++) * sa);
  w.c = 0.0f;
  return w;
}

// host-side cvt.rna.tf32.f32: round to nearest (ties away) on the 13 dropped mantissa bits
inline float tf32_round(float x) {
  uint32_t u;
  memcpy(&u, &x, 4);
  u = (u + 0x1000u) & 0xFFFFE000u;
  float r;
  memcpy(&r, &u, 4);
  return r;
}

__device__ __forceinline__ uint64_t node_key(uint32_t kind, uint32_t value) { return ((uint64_t)kind << 32) | value; }

__global__ void edge_node_keys_kernel(const alz_edge_out* __restrict__ e, uint32_t n_e, uint64_t* __restrict__ out) {
  const uint32_t stride = gridDim.x * blockDim.x;
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n_e; i += stride) {
    out[2 * i] = node_key(e[i].from_type, e[i].from);
    out[2 * i + 1] = node_key(e[i].to_type, e[i].to);
  }
}
__device__ __forceinline__ uint32_t lower_bound_u64(const uint64_t* __restrict__ a, uint32_t n, uint64_t k) {
  uint32_t lo = 0, hi = n;
  while (lo < hi) { const uint32_t mid = (lo + hi) >> 1; if (a[mid] < k) lo = mid + 1; else hi = mid; }
  return lo;
}

// per node: [out_count, in_count, out_err, in_err, out_lat, in_lat, out_deg, in_deg]
// the node count stays on the device: every consumer reads it from there, the host never waits for it
__global__ void edge_stats_kernel(const alz_edge_out* __restrict__ e, uint32_t n_e, const uint64_t* __restrict__ nodes,
                                  const uint32_t* __restrict__ n_v_ptr, uint32_t* __restrict__ src_idx,
                                  uint64_t* __restrict__ dst_key, unsigned long long* __restrict__ stats,
                                  uint32_t* __restrict__ in_deg) {
  const uint32_t n_v = *n_v_ptr;
  const uint32_t stride = gridDim.x * blockDim.x;
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n_e; i += stride) {
    const uint32_t u = lower_bound_u64(nodes, n_v, node_key(e[i].from_type, e[i].from));
    const uint32_t v = lower_bound_u64(nodes, n_v, node_key(e[i].to_type, e[i].to));
    src_idx[i] = u;
    dst_key[i] = v;
    atomicAdd(&stats[(size_t)u * 8 + 0], (unsigned long long)e[i].count);
    atomicAdd(&stats[(size_t)v * 8 + 1], (unsigned long long)e[i].count);
    if (e[i].err5xx) {
      atomicAdd(&stats[(size_t)u * 8 + 2], (unsigned long long)e[i].err5xx);
      atomicAdd(&stats[(size_t)v * 8 + 3], (unsigned long long)e[i].err5xx);
    }
    atomicAdd(&stats[(size_t)u * 8 + 4], (unsigned long long)e[i].lat_sum_ns);
    atomicAdd(&stats[(size_t)v * 8 + 5], (unsigned long long)e[i].lat_sum_ns);
    atomicAdd(&stats[(size_t)u * 8 + 6], 1ull);
    atomicAdd(&stats[(size_t)v * 8 + 7], 1ull);
    atomicAdd(&in_deg[v], 1u);
  }
}

__global__ void csr_cols_kernel(const uint32_t* __restrict__ sorted_edge, const uint32_t* __restrict__ src_idx,
                                uint32_t n_e, uint32_t* __restrict__ col) {
  const uint32_t stride = gridDim.x * blockDim.x;
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n_e; i += stride) col[i] = src_idx[sorted_edge[i]];
}

__device__ __forceinline__ double ratio(uint64_t a, uint64_t b) { return b ? (double)a / (double)b : 0.0; }

__global__ void node_features_kernel(const uint64_t* __restrict__ nodes, const unsigned long long* __restrict__ stats,
                                     const uint32_t* __restrict__ n_v_ptr, float* __restrict__ h0) {
  const uint32_t n_v = *n_v_ptr;
  const uint32_t stride = gridDim.x * blockDim.x;
  for (uint32_t v = blockIdx.x * blockDim.x + threadIdx.x; v < n_v; v += stride) {
    const unsigned long long* s = stats + (size_t)v * 8;
    float* o = h0 + (size_t)v * D;
    const uint32_t kind = (uint32_t)(nodes[v] >> 32);
    float f[12];
    f[0] = (float)log1p((double)s[0]);
    f[1] = (float)log1p((double)s[1]);
    f[2] = (float)ratio(s[2], s[0]);
    f[3] = (float)ratio(s[3], s[1]);
    f[4] = (float)log1p(ratio(s[4], s[0]));
    f[5] = (float)log1p(ratio(s[5], s[1]));
    f[6] = (float)log1p((double)s[6]);
    f[7] = (float)log1p((double)s[7]);
    f[8] = kind == ALZ_NODE_POD ? 1.f : 0.f;
    f[9] = kind == ALZ_NODE_SVC ? 1.f : 0.f;
    f[10] = kind >= ALZ_NODE_OUTBOUND ? 1.f : 0.f;   // outbound, keyed by address or by Host header
    f[11] = 1.f;
    for (int j = 0; j < D; ++j) o[j] = j < 12 ? f[j] : 0.f;
  }
}

// one GraphSAGE-mean layer, FP32 SIMT: warp per node, W (32 KB) in shared memory
__global__ void __launch_bounds__(256) sage_layer_kernel(const float* __restrict__ h_in, float* __restrict__ h_out,
                                                         const uint32_t* __restrict__ rowptr,
                                                         const uint32_t* __restrict__ col, const float* __restrict__ W,
                                                         const float* __restrict__ b, const uint32_t* __restrict__ n_v_ptr) {
  const uint32_t n_v = *n_v_ptr;
  __shared__ float sW[128 * D];
  __shared__ float sz[8][128];
  for (int i = threadIdx.x; i < 128 * D; i += blockDim.x) sW[i] = W[i];
  __syncthreads();
  const uint32_t lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
  const uint32_t warps_per_grid = (gridDim.x * blockDim.x) >> 5;
  for (uint32_t v = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; v < n_v; v += warps_per_grid) {
    const uint32_t beg = rowptr[v], end = rowptr[v + 1];
    float m0 = 0.f, m1 = 0.f;
    for (uint32_t p = beg; p < end; ++p) {          // CSR order: deterministic sum
      const float* hu = h_in + (size_t)col[p] * D;
      m0 += hu[lane];
      m1 += hu[32 + lane];
    }
    const float inv = end > beg ? 1.0f / (float)(end - beg) : 0.f;
    const float* hv = h_in + (size_t)v * D;
    sz[warp][lane] = hv[lane];
    sz[warp][32 + lane] = hv[32 + lane];
    sz[warp][64 + lane] = m0 * inv;
    sz[warp][96 + lane] = m1 * inv;
    __syncwarp();
    float a0 = b[lane], a1 = b[32 + lane];
#pragma unroll 8
    for (int k = 0; k < 128; ++k) {
      const float z = sz[warp][k];
      a0 = fmaf(z, sW[k * D + lane], a0);
      a1 = fmaf(z, sW[k * D + 32 + lane], a1);
    }
    h_out[(size_t)v * D + lane] = fmaxf(a0, 0.f);
    h_out[(size_t)v * D + 32 + lane] = fmaxf(a1, 0.f);
    __syncwarp();
  }
}

// ---------------------------------------------------------------------------
// The same layer on the 5th-gen tensor cores: the feature update
//   [h_v || mean_{u in N_in(v)} h_u]  (128 nodes x 128)  x  W (128 x 64)
// is the path's one dense contraction. One persistent CTA per SM, tile = 128 nodes:
//   gather   8 warps build the tile's 128 x 128 operand directly in shared memory in
//            the UMMA K-major / no-swizzle layout (8 x 16-byte core matrices)
//   MMA      one thread issues tcgen05.mma.cta_group::1.kind::tf32, M=128 N=64 K=8,
//            accumulator in TMEM (64 columns)
//   epilogue 4 warps tcgen05.ld their 32 lanes, add bias, ReLU, store rows
// Precision: kind::tf32 keeps 10 mantissa bits, which would miss the 1e-5 bound, so
// both operands are split x = hi + lo (hi = cvt.rna.tf32, lo = x - hi, exact) and
// the product is accumulated as hi*hi + hi*lo + lo*hi (3xTF32): 48 MMAs per tile.
// ---------------------------------------------------------------------------
namespace tc {
constexpr uint32_t TM = 128, TK = 128, TN = 64;
constexpr uint32_t A_BYTES = TM * TK * 4, B_BYTES = TN * TK * 4;
constexpr uint32_t A_LBO = (TM / 8) * 128, A_SBO = 128;   // K-adjacent cores TM/8 cores apart; row groups adjacent
constexpr uint32_t B_LBO = (TN / 8) * 128, B_SBO = 128;

// byte offset of element (row r, k) in a K-major no-swizzle operand with R rows:
// core matrix = 8 rows x 16 B; cores of one K-slice are contiguous over the row groups
__host__ __device__ inline uint32_t op_off(uint32_t r, uint32_t k, uint32_t rows) {
  return (k >> 2) * (rows / 8) * 128 + (r >> 3) * 128 + (r & 7) * 16 + (k & 3) * 4;
}
// UMMA shared-memory descriptor (sm_100): start >> 4, LBO >> 4 at bit 16, SBO >> 4 at bit 32,
// version 1 at bit 46, layout type 0 (no swizzle) at bit 61
__device__ __forceinline__ uint64_t smem_desc(uint32_t smem_addr, uint32_t lbo, uint32_t sbo) {
  return (uint64_t)((smem_addr & 0x3FFFFu) >> 4) | ((uint64_t)(lbo >> 4) << 16) | ((uint64_t)(sbo >> 4) << 32) |
         (1ull << 46);
}
// instruction descriptor: D = F32 (bit 4), A = B = TF32 (2 << 7, 2 << 10), both K-major, N >> 3 at bit 17, M >> 4 at bit 24
constexpr uint32_t kIdesc = (1u << 4) | (2u << 7) | (2u << 10) | ((TN >> 3) << 17) | ((TM >> 4) << 24);

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ uint32_t to_tf32(float x) {
  uint32_t u;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(u) : "f"(x));
  return u;
}
__device__ __forceinline__ void mma_tf32(uint32_t tmem_d, uint64_t da, uint64_t db, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}\n"
      :: "r"(tmem_d), "l"(da), "l"(db), "r"(kIdesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t* v) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
               : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
                 "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
               : "r"(taddr) : "memory");
}

// ---- TMA-staged neighbour gather ---------------------------------------------------------
// A warp builds 16 rows of the tile's operand. Every 256-byte feature row it needs — its nodes' own rows (16
// consecutive rows of h_in: two bulk copies) and then the rows of their in-neighbours in CSR order — is fetched
// by the TMA (cp.async.bulk global -> shared, completion on an mbarrier) into a two-slot ring of 8 rows per
// warp: while the warp sums the rows of one slot, the copies of the next 8 neighbours are in flight, 16 rows
// per warp regardless of the nodes' degrees (the edge range of the warp's rows is walked as one stream and cut
// at the row boundaries). No register holds a row in flight, unlike plain loads.
constexpr uint32_t RING_ROWS = 8, RING_BYTES = RING_ROWS * 256;
constexpr uint32_t SMEM_TC = 2 * A_BYTES + 2 * B_BYTES + 8 * 2 * RING_BYTES + 256;

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  uint32_t ok;
  do {
    asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                 : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
  } while (!ok);
}
__device__ __forceinline__ void tma_row(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(dst), "l"(src), "r"(bytes), "r"(bar) : "memory");
}
// operand row r, columns kbase + lane and kbase + 32 + lane <- (z0, z1), split hi/lo in the UMMA layout
__device__ __forceinline__ void put_pair(uint8_t* sA_hi, uint8_t* sA_lo, uint32_t r, uint32_t kbase, uint32_t lane,
                                         float z0, float z1) {
  const float z[2] = {z0, z1};
#pragma unroll
  for (int q = 0; q < 2; ++q) {
    const uint32_t k = kbase + (uint32_t)q * 32 + lane;
    const uint32_t hi = to_tf32(z[q]);
    const uint32_t lo = to_tf32(z[q] - __uint_as_float(hi));
    const uint32_t off = op_off(r, k, TM);
    *reinterpret_cast<uint32_t*>(sA_hi + off) = hi;
    *reinterpret_cast<uint32_t*>(sA_lo + off) = lo;
  }
}

__global__ void __launch_bounds__(256, 1) sage_layer_tc_kernel(const float* __restrict__ h_in, float* __restrict__ h_out,
                                                               const uint32_t* __restrict__ rowptr,
                                                               const uint32_t* __restrict__ col,
                                                               const uint8_t* __restrict__ Wcan,   // B_hi then B_lo
                                                               const float* __restrict__ bias,
                                                               const uint32_t* __restrict__ n_v_ptr) {
  extern __shared__ __align__(1024) uint8_t smem[];
  const uint32_t n_v = *n_v_ptr;
  const uint32_t zero_rt = n_v >> 31;                    // node counts are < 2^31
  uint8_t* sA_hi = smem;
  uint8_t* sA_lo = smem + A_BYTES;
  uint8_t* sB = smem + 2 * A_BYTES;                      // B_hi, then B_lo
  uint8_t* rings = smem + 2 * A_BYTES + 2 * B_BYTES;     // per warp: 2 slots of RING_ROWS rows
  uint64_t* bars = reinterpret_cast<uint64_t*>(rings + 8 * 2 * RING_BYTES);   // [0] MMA done, [1 + 2w + slot] ring slots
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 1 + 16);
  const uint32_t tid = threadIdx.x, warp = tid >> 5, lane = tid & 31u;
  uint64_t* mbar = bars;
  const float* ring = reinterpret_cast<const float*>(rings + warp * 2 * RING_BYTES);
  const uint32_t ring_a = smem_u32(ring);
  const uint32_t rbar = smem_u32(bars + 1 + 2 * warp);
  uint32_t ring_uses[2] = {0u, 0u};

  for (uint32_t i = tid; i < 2 * B_BYTES / 16; i += blockDim.x)
    reinterpret_cast<uint4*>(sB)[i] = reinterpret_cast<const uint4*>(Wcan)[i];
  if (warp == 0) {   // TMEM: 64 columns for the 128 x 64 fp32 accumulator
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 64;" :: "r"(smem_u32(tmem_slot)) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  if (tid == 0) asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" :: "r"(smem_u32(mbar)) : "memory");
  if (lane == 0) { mbar_init(rbar, 1u); mbar_init(rbar + 8u, 1u); }
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t*>(tmem_slot);
  uint32_t parity = 0;

  for (uint32_t tile = blockIdx.x; tile * TM < n_v; tile += gridDim.x) {
    // ---- gather: warp w builds rows 16w .. 16w+15 of the operand (hi and lo parts)
    const uint32_t v0 = tile * TM + warp * 16;
    const uint32_t n_rows = v0 < n_v ? min(16u, n_v - v0) : 0u;
    // (1) the nodes' own rows: two bulk copies of up to 8 consecutive rows each
    for (uint32_t half = 0; half < 2; ++half) {
      const uint32_t cnt = n_rows > half * 8 ? min(8u, n_rows - half * 8) : 0u;
      if (lane == 0 && cnt) {
        mbar_expect_tx(rbar + half * 8u, cnt * 256u);
        tma_row(ring_a + half * RING_BYTES, h_in + (size_t)(v0 + half * 8) * D, cnt * 256u, rbar + half * 8u);
      }
    }
    for (uint32_t half = 0; half < 2; ++half) {
      const uint32_t cnt = n_rows > half * 8 ? min(8u, n_rows - half * 8) : 0u;
      if (cnt) { mbar_wait(rbar + half * 8u, ring_uses[half] & 1u); ring_uses[half]++; }
      for (uint32_t j = 0; j < 8; ++j) {
        const float* row = ring + (half * RING_ROWS + j) * D;
        const bool on = j < cnt;
        put_pair(sA_hi, sA_lo, warp * 16 + half * 8 + j, 0u, lane, on ? row[lane] : 0.f, on ? row[32 + lane] : 0.f);
      }
      __syncwarp();
    }
    // (2) the in-neighbours of the warp's rows, as one stream of edges cut at the row boundaries
    const uint32_t e_beg = n_rows ? rowptr[v0] : 0u, e_end = n_rows ? rowptr[v0 + n_rows] : 0u;
    const uint32_t n_chunks = (e_end - e_beg + RING_ROWS - 1) / RING_ROWS;
    // `dep` is always 0 but derived from the last word this lane read out of the slot (zero_rt is a run-time 0 the
    // compiler cannot see through): the copies that refill a slot cannot be issued before its reads have returned
    auto issue = [&](uint32_t c, uint32_t dep) {
      const uint32_t slot = c & 1u, first = e_beg + c * RING_ROWS, cnt = min(RING_ROWS, e_end - first);
      if (lane == 0) mbar_expect_tx(rbar + slot * 8u, cnt * 256u + dep);
      __syncwarp();
      if (lane < cnt) tma_row(ring_a + (slot * RING_ROWS + lane) * 256u, h_in + (size_t)col[first + lane] * D, 256u + dep, rbar + slot * 8u);
    };
    if (n_chunks > 0) issue(0, 0u);
    if (n_chunks > 1) issue(1, 0u);
    uint32_t r = 0;                                   // current row of the warp
    uint32_t row_end = n_rows ? rowptr[v0 + 1] : 0u, row_beg = e_beg;
    float m0 = 0.f, m1 = 0.f;
    auto close_rows_until = [&](uint32_t e) {         // rows that end at or before edge e are complete
      while (r < n_rows && row_end <= e) {
        const float inv = row_end > row_beg ? 1.0f / (float)(row_end - row_beg) : 0.f;
        put_pair(sA_hi, sA_lo, warp * 16 + r, 64u, lane, m0 * inv, m1 * inv);
        m0 = m1 = 0.f;
        ++r;
        row_beg = row_end;
        if (r < n_rows) row_end = rowptr[v0 + r + 1];
      }
    };
    for (uint32_t c = 0; c < n_chunks; ++c) {
      const uint32_t slot = c & 1u, first = e_beg + c * RING_ROWS, cnt = min(RING_ROWS, e_end - first);
      mbar_wait(rbar + slot * 8u, ring_uses[slot] & 1u);
      ring_uses[slot]++;
      float last = 0.f;
      for (uint32_t j = 0; j < cnt; ++j) {          // CSR order: deterministic sum
        close_rows_until(first + j);
        const float* row = ring + (slot * RING_ROWS + j) * D;
        last = row[lane];
        m0 += last;
        m1 += row[32 + lane];
      }
      __syncwarp();
      if (c + 2 < n_chunks) issue(c + 2, __float_as_uint(last) & zero_rt);   // the slot goes back to the TMA
    }
    close_rows_until(e_end);                          // the last rows, and rows without in-edges
    for (uint32_t rr = n_rows; rr < 16; ++rr) {       // rows past the end of the graph: zeros
      put_pair(sA_hi, sA_lo, warp * 16 + rr, 0u, lane, 0.f, 0.f);
      put_pair(sA_hi, sA_lo, warp * 16 + rr, 64u, lane, 0.f, 0.f);
    }
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // generic-proxy stores -> tensor-core (async proxy) reads
    __syncthreads();
    // ---- MMA: one thread, 3 passes x 16 K-steps of M128 N64 K8
    if (tid == 0) {
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
      const uint32_t a_hi = smem_u32(sA_hi), a_lo = smem_u32(sA_lo), b_hi = smem_u32(sB), b_lo = smem_u32(sB + B_BYTES);
      const uint32_t pa[3] = {a_hi, a_hi, a_lo}, pb[3] = {b_hi, b_lo, b_hi};
      uint32_t acc = 0;
#pragma unroll
      for (int ps = 0; ps < 3; ++ps) {
        for (uint32_t ks = 0; ks < TK / 8; ++ks) {
          const uint64_t da = smem_desc(pa[ps] + ks * 2 * A_LBO, A_LBO, A_SBO);
          const uint64_t db = smem_desc(pb[ps] + ks * 2 * B_LBO, B_LBO, B_SBO);
          mma_tf32(tmem_base, da, db, acc);
          acc = 1;
        }
      }
      asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];"
                   :: "r"(smem_u32(mbar)) : "memory");
    }
    // ---- epilogue: warps 0..3 own TMEM lanes 32w .. 32w+31
    if (warp < 4) {
      uint32_t done = 0;
      while (!done) {
        asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}\n"
                     : "=r"(done) : "r"(smem_u32(mbar)), "r"(parity) : "memory");
      }
      __syncwarp();   // lane 0 of warp 0 comes from the MMA issue: .sync.aligned loads need the whole warp together
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
      const uint32_t v = tile * TM + warp * 32 + lane;
      float* orow = h_out + (size_t)v * D;
#pragma unroll
      for (uint32_t c = 0; c < TN; c += 16) {
        uint32_t acc[16];
        tmem_ld16(tmem_base + ((warp * 32u) << 16) + c, acc);
        asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
        if (v < n_v) {
#pragma unroll
          for (int j = 0; j < 16; j += 4) {
            float4 o;
            o.x = fmaxf(__uint_as_float(acc[j + 0]) + bias[c + j + 0], 0.f);
            o.y = fmaxf(__uint_as_float(acc[j + 1]) + bias[c + j + 1], 0.f);
            o.z = fmaxf(__uint_as_float(acc[j + 2]) + bias[c + j + 2], 0.f);
            o.w = fmaxf(__uint_as_float(acc[j + 3]) + bias[c + j + 3], 0.f);
            *reinterpret_cast<float4*>(orow + c + j) = o;
          }
        }
      }
      asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    }
    parity ^= 1u;
    __syncthreads();   // operand tile and accumulator are free again
  }
  __syncthreads();
  if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 64;" :: "r"(tmem_base) : "memory");
}
}  // namespace tc

// docs/SPEC.md §4/§5 on the device, float64
__device__ __forceinline__ double bucket_lo(uint32_t b) {
  if (b == 0) return 0.0;
  const double base = (double)(1ull << (8 + b / 2));
  return (b & 1u) ? base * 1.5 : base;
}
__device__ __forceinline__ double bucket_hi(uint32_t b) { return b == ALZ_NB - 1 ? (double)(1ull << 40) : bucket_lo(b + 1); }
__global__ void __launch_bounds__(256) edge_score_kernel(const alz_edge_out* __restrict__ e, uint32_t n_e,
                                                         const uint32_t* __restrict__ src_idx,
                                                         const uint64_t* __restrict__ dst_key,
                                                         const float* __restrict__ h2, const float* __restrict__ a,
                                                         float c, float* __restrict__ scores) {
  const uint32_t lane = threadIdx.x & 31u;
  const uint32_t warps_per_grid = (gridDim.x * blockDim.x) >> 5;
  for (uint32_t i = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; i < n_e; i += warps_per_grid) {
    const float* hu = h2 + (size_t)src_idx[i] * D;
    const float* hv = h2 + (size_t)dst_key[i] * D;
    float acc = hu[lane] * a[lane] + hu[32 + lane] * a[32 + lane] + hv[lane] * a[64 + lane] +
                hv[32 + lane] * a[96 + lane];
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xFFFFFFFFu, acc, o);
    // quantiles with the whole warp: lane l owns buckets 2l and 2l+1; an inclusive scan of the
    // (exactly representable) counts finds the bucket each quantile falls into, then the one
    // lane that owns it interpolates exactly like hist_quantile() / SPEC §5
    const double c0 = (double)e[i].hist[2 * lane], c1 = (double)e[i].hist[2 * lane + 1];
    double incl = c0 + c1;
    for (int o = 1; o < 32; o <<= 1) {
      const double t = __shfl_up_sync(0xFFFFFFFFu, incl, o);
      if ((int)lane >= o) incl += t;
    }
    const double total = __shfl_sync(0xFFFFFFFFu, incl, 31);
    const double before = incl - (c0 + c1);
    double qv[2];
#pragma unroll
    for (int qi = 0; qi < 2; ++qi) {
      const double target = (qi == 0 ? 0.5 : 0.99) * total;
      // first bucket with c > 0 and cum + c >= target
      const bool h0 = c0 > 0.0 && before + c0 >= target;
      const bool h1 = c1 > 0.0 && before + c0 + c1 >= target;
      const uint32_t m = __ballot_sync(0xFFFFFFFFu, h0 || h1);
      double val = total > 0.0 ? bucket_hi(ALZ_NB - 1) : 0.0;
      const int owner = m ? __ffs(m) - 1 : 0;
      if (m && (int)lane == owner) {
        const uint32_t b = h0 ? 2u * lane : 2u * lane + 1u;
        const double cum = h0 ? before : before + c0;
        const double cb = h0 ? c0 : c1;
        double f = (target - cum) / cb;
        if (f < 0.0) f = 0.0;
        val = bucket_lo(b) + f * (bucket_hi(b) - bucket_lo(b));
      }
      qv[qi] = __shfl_sync(0xFFFFFFFFu, val, owner);
    }
    if (lane == 0) {
      const float f0 = (float)log1p((double)e[i].count);
      const float f1 = (float)ratio(e[i].err5xx, e[i].count);
      const float f2 = (float)log1p(qv[0]);
      const float f3 = (float)log1p(qv[1]);
      const float z = acc + f0 * a[128] + f1 * a[129] + f2 * a[130] + f3 * a[131] + c;
      scores[i] = 1.0f / (1.0f + expf(-z));
    }
  }
}

}  // namespace

struct alz_gnn_state {
  Owned mem;
  uint32_t cap_e = 0, cap_v = 0;
  uint64_t *d_nk = nullptr, *d_nk_sorted = nullptr, *d_nodes = nullptr, *d_dst_key = nullptr, *d_dst_sorted = nullptr;
  uint32_t *d_flags = nullptr, *d_pos = nullptr, *d_iota = nullptr, *d_vals = nullptr, *d_src_idx = nullptr;
  uint32_t *d_in_deg = nullptr, *d_rowptr = nullptr, *d_col = nullptr, *d_sorted_edge = nullptr;
  unsigned long long* d_stats = nullptr;
  float *d_h[3] = {nullptr, nullptr, nullptr}, *d_W[2] = {nullptr, nullptr}, *d_b[2] = {nullptr, nullptr};
  float *d_a = nullptr, *d_scores = nullptr;
  uint8_t* d_Wcan[2] = {nullptr, nullptr};   // per layer: W^T split hi/lo in the UMMA operand layout (64 KB)
  bool use_tc = true;
  float c = 0.f;
  void* d_tmp = nullptr;
  size_t tmp_bytes = 0;
  uint32_t n_v = 0, n_e = 0;
  bool n_v_known = true;
  uint32_t* d_nv = nullptr;      // node count of the last pass, on the device
};
void StateDelete::operator()(alz_gnn_state* g) const { delete g; }

// built on first use and published only when complete: after a failed allocation the next call starts again
static int gnn_init(alz_handle* h) {
  if (h->gnn) return ALZ_OK;
  StatePtr<alz_gnn_state> g(new alz_gnn_state());
  Owned& m = g->mem;
  g->cap_e = h->cfg.max_edges;
  g->cap_v = 2 * h->cfg.max_edges;
  const size_t E = g->cap_e, V = g->cap_v;
  CK(m.dev(&g->d_nk, V * 8));
  CK(m.dev(&g->d_nk_sorted, V * 8));
  CK(m.dev(&g->d_nodes, V * 8));
  CK(m.dev(&g->d_dst_key, E * 8));
  CK(m.dev(&g->d_dst_sorted, E * 8));
  CK(m.dev(&g->d_flags, V * 4));
  CK(m.dev(&g->d_pos, V * 4));
  CK(m.dev(&g->d_iota, V * 4));
  CK(m.dev(&g->d_vals, V * 4));
  CK(m.dev(&g->d_src_idx, E * 4));
  CK(m.dev(&g->d_in_deg, (V + 1) * 4));
  CK(m.dev(&g->d_rowptr, (V + 1) * 4));
  CK(m.dev(&g->d_col, E * 4));
  CK(m.dev(&g->d_sorted_edge, E * 4));
  CK(m.dev(&g->d_stats, V * 8 * 8));
  for (int i = 0; i < 3; ++i) CK(m.dev(&g->d_h[i], V * D * 4));
  CK(m.dev(&g->d_scores, E * 4));
  CK(m.dev(&g->d_nv, 4));
  g->tmp_bytes = std::max(sort_pairs_temp_bytes((uint32_t)V), scan_temp_bytes((uint32_t)V + 1));
  CK(m.dev(&g->d_tmp, g->tmp_bytes));
  const Weights w = make_weights();
  for (int l = 0; l < 2; ++l) {
    CK(m.dev(&g->d_W[l], 128 * D * 4));
    CK(m.dev(&g->d_b[l], D * 4));
    CK(cudaMemcpyAsync(g->d_W[l], w.W[l].data(), 128 * D * 4, cudaMemcpyHostToDevice, h->stream));
    CK(cudaMemcpyAsync(g->d_b[l], w.b[l].data(), D * 4, cudaMemcpyHostToDevice, h->stream));
  }
  {
    const char* simt = getenv("ALZ_GNN_SIMT");   // comparison knob: FP32 FFMA layer instead of tcgen05
    g->use_tc = !(simt && simt[0] == '1');
    std::vector<float> can(2 * tc::TN * tc::TK);
    for (int l = 0; l < 2; ++l) {
      for (uint32_t n = 0; n < tc::TN; ++n)
        for (uint32_t k = 0; k < tc::TK; ++k) {
          const float x = w.W[l][k * D + n];               // B[n][k] = W[k][n]
          const float hi = tf32_round(x), lo = tf32_round(x - hi);
          const uint32_t off = tc::op_off(n, k, tc::TN) / 4;
          can[off] = hi;
          can[tc::TN * tc::TK + off] = lo;
        }
      CK(m.dev(&g->d_Wcan[l], 2 * tc::B_BYTES));
      CK(cudaMemcpyAsync(g->d_Wcan[l], can.data(), 2 * tc::B_BYTES, cudaMemcpyHostToDevice, h->stream));
      CK(cudaStreamSynchronize(h->stream));   // `can` is rewritten for the next layer
    }
    CK(cudaFuncSetAttribute(tc::sage_layer_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tc::SMEM_TC));
  }
  CK(m.dev(&g->d_a, 132 * 4));
  CK(cudaMemcpyAsync(g->d_a, w.a.data(), 132 * 4, cudaMemcpyHostToDevice, h->stream));
  CK(cudaStreamSynchronize(h->stream));     // the host-side weight vectors die with this frame
  g->c = w.c;
  h->gnn = std::move(g);
  return ALZ_OK;
}

// CSR build + 2 layers + scoring over the last flushed window (h->d_out). Nothing here waits for the device:
// the node count lives in device memory and every kernel reads it there; buffers and grids are sized by the
// bound 2 * n_e the host knows. Sorts only cover the key bits that can differ.
static int bits_for(uint64_t x) { int b = 1; while (b < 64 && (x >> b) != 0) ++b; return b; }

static int gnn_run(alz_handle* h) {
  int rc = gnn_init(h);
  if (rc != ALZ_OK) return rc;
  alz_gnn_state* g = h->gnn.get();
  cudaStream_t s = h->stream;
  const uint32_t n_e = h->last_n_edges;
  g->n_e = n_e;
  g->n_v = 0;
  g->n_v_known = n_e == 0;
  if (n_e == 0) { CK(cudaMemsetAsync(g->d_nv, 0, 4, s)); return ALZ_OK; }
  if (n_e > g->cap_e) return ALZ_E_CAPACITY;
  const unsigned grid = (unsigned)h->sms * 4;
  const uint32_t n2 = 2 * n_e;   // bound on the node count
  // nodes: (kind 2 bits << 32 | value 32 bits): 34 key bits
  edge_node_keys_kernel<<<grid, 256, 0, s>>>(h->d_out, n_e, g->d_nk);
  launch_iota(g->d_iota, n2, h->sms, s);
  sort_pairs(g->d_tmp, g->tmp_bytes, g->d_nk, g->d_nk_sorted, g->d_iota, g->d_vals, n2, s, 34);
  unique_sorted_u64(g->d_tmp, g->tmp_bytes, g->d_nk_sorted, n2, g->d_flags, g->d_pos, g->d_nodes, g->d_nv, h->sms, s);
  // stats + CSR by destination (destination index < n2)
  CK(cudaMemsetAsync(g->d_stats, 0, (size_t)n2 * 64, s));
  CK(cudaMemsetAsync(g->d_in_deg, 0, ((size_t)n2 + 1) * 4, s));
  edge_stats_kernel<<<grid, 256, 0, s>>>(h->d_out, n_e, g->d_nodes, g->d_nv, g->d_src_idx, g->d_dst_key, g->d_stats,
                                         g->d_in_deg);
  launch_iota(g->d_iota, n_e, h->sms, s);
  sort_pairs(g->d_tmp, g->tmp_bytes, g->d_dst_key, g->d_dst_sorted, g->d_iota, g->d_sorted_edge, n_e, s, bits_for(n2));
  csr_cols_kernel<<<grid, 256, 0, s>>>(g->d_sorted_edge, g->d_src_idx, n_e, g->d_col);
  exclusive_scan_u32(g->d_tmp, g->tmp_bytes, g->d_in_deg, g->d_rowptr, n2 + 1, s);
  // features, layers, scores
  node_features_kernel<<<grid, 256, 0, s>>>(g->d_nodes, g->d_stats, g->d_nv, g->d_h[0]);
  for (int l = 0; l < 2; ++l) {
    if (g->use_tc) {
      const unsigned tiles = (n2 + tc::TM - 1) / tc::TM;
      tc::sage_layer_tc_kernel<<<std::min<unsigned>(tiles, (unsigned)h->sms), 256, tc::SMEM_TC, s>>>(
          g->d_h[l], g->d_h[l + 1], g->d_rowptr, g->d_col, g->d_Wcan[l], g->d_b[l], g->d_nv);
    } else {
      sage_layer_kernel<<<grid, 256, 0, s>>>(g->d_h[l], g->d_h[l + 1], g->d_rowptr, g->d_col, g->d_W[l], g->d_b[l], g->d_nv);
    }
  }
  edge_score_kernel<<<grid, 256, 0, s>>>(h->d_out, n_e, g->d_src_idx, g->d_dst_key, g->d_h[2], g->d_a, g->c,
                                         g->d_scores);
  h->launches += 12;
  CK(cudaGetLastError());
  return ALZ_OK;
}

static int gnn_score_device_locked(alz_handle* h, const float** dev_scores, size_t* n_out) {
  CK(cudaSetDevice(h->device));
  int rc = gnn_run(h);
  *n_out = h->gnn ? h->gnn->n_e : 0;
  if (rc != ALZ_OK) return rc;
  if (dev_scores) *dev_scores = h->gnn->d_scores;
  return ALZ_OK;
}

extern "C" int alz_gnn_score_device(alz_handle* h, const float** dev_scores, size_t* n_out) {
  if (!h || !n_out) return ALZ_E_INVAL;
  std::lock_guard<std::mutex> g(h->mu);
  return gnn_score_device_locked(h, dev_scores, n_out);
}

extern "C" int alz_gnn_score(alz_handle* h, float* edge_scores, size_t cap, size_t* n_out) {
  if (!h || !n_out || (!edge_scores && cap)) return ALZ_E_INVAL;
  std::lock_guard<std::mutex> g(h->mu);
  const float* d = nullptr;
  int rc = gnn_score_device_locked(h, &d, n_out);
  if (rc != ALZ_OK) return rc;
  if (*n_out > cap) return ALZ_E_CAPACITY;
  if (*n_out) CK(cudaMemcpyAsync(edge_scores, d, *n_out * 4, cudaMemcpyDeviceToHost, h->stream));
  CK(cudaStreamSynchronize(h->stream));
  return ALZ_OK;
}

// debug/test: node keys ((kind << 32) | value, ascending) and the layer-2 embeddings of the last alz_gnn_score
extern "C" int alz_gnn_nodes(alz_handle* h, uint64_t* node_keys, float* h2, size_t cap, size_t* n_out) {
  if (!h || !n_out) return ALZ_E_INVAL;
  std::lock_guard<std::mutex> g(h->mu);
  if (!h->gnn) return ALZ_E_STATE;
  CK(cudaSetDevice(h->device));
  if (!h->gnn->n_v_known) {   // the pass itself never needed the count on the host
    CK(cudaMemcpyAsync(&h->gnn->n_v, h->gnn->d_nv, 4, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    h->gnn->n_v_known = true;
  }
  *n_out = h->gnn->n_v;
  if (h->gnn->n_v > cap) return ALZ_E_CAPACITY;
  if (h->gnn->n_v) {
    if (node_keys) CK(cudaMemcpyAsync(node_keys, h->gnn->d_nodes, (size_t)h->gnn->n_v * 8, cudaMemcpyDeviceToHost, h->stream));
    if (h2) CK(cudaMemcpyAsync(h2, h->gnn->d_h[2], (size_t)h->gnn->n_v * D * 4, cudaMemcpyDeviceToHost, h->stream));
  }
  CK(cudaStreamSynchronize(h->stream));
  return ALZ_OK;
}

// SPEC §5 on the host: the same interpolation, float64
extern "C" int alz_edge_quantiles(const alz_edge_out* e, const double* qs, size_t nq, double* out_ns) {
  if (!e || (!qs && nq) || (!out_ns && nq)) return ALZ_E_INVAL;
  uint64_t total = 0;
  for (int b = 0; b < ALZ_NB; ++b) total += e->hist[b];
  auto lo = [](uint32_t b) -> double {
    if (b == 0) return 0.0;
    const double base = (double)(1ull << (8 + b / 2));
    return (b & 1u) ? base * 1.5 : base;
  };
  auto hi = [&](uint32_t b) -> double { return b == ALZ_NB - 1 ? (double)(1ull << 40) : lo(b + 1); };
  for (size_t i = 0; i < nq; ++i) {
    double r = total ? hi(ALZ_NB - 1) : 0.0;
    if (total) {
      const double target = qs[i] * (double)total;
      double cum = 0.0;
      for (uint32_t b = 0; b < ALZ_NB; ++b) {
        const double c = (double)e->hist[b];
        if (c > 0.0 && cum + c >= target) {
          double f = (target - cum) / c;
          if (f < 0.0) f = 0.0;
          r = lo(b) + f * (hi(b) - lo(b));
          break;
        }
        cum += c;
      }
    }
    out_ns[i] = r;
  }
  return ALZ_OK;
}
