// alz_kernels.cuh — launcher declarations shared by the kernels and the C-ABI layer.
#pragma once
#include "alz_device.cuh"
#include "../synth/alz_synth.h"

namespace alz {
void launch_ingest_pairs_v1(const alz_l7_rec* recs, uint64_t n, const AccTable& pairs, Counters* ctr,
                            const EpEntry* ep, uint32_t ep_mask, int sms, cudaStream_t s);
void launch_ingest_pairs(const alz_l7_rec* recs, uint64_t n, const AccTable& pairs, Counters* ctr,
                         const HotState* hot, const EpEntry* ep, uint32_t ep_mask, const uint32_t* bloom, int sms,
                         cudaStream_t s);
void launch_ingest_pairs_rec16(const alz_l7_rec16* recs, uint64_t n, const uint64_t* dur_ovf, const AccTable& pairs,
                               Counters* ctr, const HotState* hot, const EpEntry* ep, uint32_t ep_mask,
                               const uint32_t* bloom, int sms, cudaStream_t s);
void launch_ingest_pairs_windowed(const alz_l7_rec* recs, uint64_t n, const AccTable& pairs, Counters* ctr,
                                  const HotState* hot, const EpEntry* ep, uint32_t ep_mask, const uint32_t* bloom,
                                  uint64_t* win, uint64_t off, alz_l7_rec* defer_buf, uint32_t defer_cap, int sms,
                                  cudaStream_t s);
void launch_window_advance(uint64_t* win, cudaStream_t s);
uint32_t ingest_table_rows();
void launch_hot_select(const AccTable& pairs, HotState* hot, int sms, cudaStream_t s);
void launch_ingest_eager(const alz_l7_rec* recs, uint64_t n, const EpEntry* ep, uint32_t ep_mask,
                         const AccTable& edges, Counters* ctr, int sms, cudaStream_t s);
void launch_fold_resolve(const AccTable& pairs, const EpEntry* ep, uint32_t ep_mask, const AccTable& edges,
                         Counters* ctr, HotState* hot, int sms, cudaStream_t s);
void launch_fold_add(const AccTable& pairs, const AccTable& edges, Counters* ctr, HotState* hot, int sms,
                     cudaStream_t s);
void launch_ep_patch(EpEntry* tab, const void* patch, uint32_t n, int sms, cudaStream_t s);
void launch_iota(uint32_t* out, uint32_t n, int sms, cudaStream_t s);
void launch_gather_edges(const AccTable& edges, const uint64_t* keys, const uint32_t* rows, uint32_t n_live,
                         alz_edge_out* out, bool reset, int sms, cudaStream_t s);
void launch_compact_raw(const uint8_t* raw, uint64_t n, alz_l7_rec* out, int sms, cudaStream_t s);
void launch_synth(const alz_synth_view& v, uint64_t first, uint64_t n, alz_l7_rec* out, int sms, cudaStream_t s);
void launch_synth_owned(const alz_synth_view& v, uint64_t first, uint64_t n, uint32_t nranks, uint32_t rank,
                        alz_l7_rec* out, uint64_t cap, unsigned long long* n_written, int sms, cudaStream_t s);
// radix sort of (edge key, row) pairs by key (alz_sort.cu)
size_t sort_pairs_temp_bytes(uint32_t n);
void sort_pairs(void* temp, size_t temp_bytes, const uint64_t* keys_in, uint64_t* keys_out,
                const uint32_t* vals_in, uint32_t* vals_out, uint32_t n, cudaStream_t s, int end_bit = 64);
size_t scan_temp_bytes(uint32_t n);
void exclusive_scan_u32(void* temp, size_t temp_bytes, const uint32_t* in, uint32_t* out, uint32_t n, cudaStream_t s);
// out[0 .. *n_unique) = the distinct values of sorted[0 .. n), ascending. The count stays on the device, so no
// caller has to wait for it. flags and pos: n words of scratch each; temp: exclusive_scan_u32's. Three own launches.
void unique_sorted_u64(void* temp, size_t temp_bytes, const uint64_t* sorted, uint32_t n, uint32_t* flags,
                       uint32_t* pos, uint64_t* out, uint32_t* n_unique, int sms, cudaStream_t s);

// ---- blocks of sorted edge rows: the gathered blocks of a multi-rank flush (alz_comm.cu) and the slots of the
// window history (alz_history.cu). A block is a header row, then header.count live rows in ascending key order.
constexpr uint32_t kRowWords64 = sizeof(alz_edge_out) / 8;   // 37
constexpr uint32_t kHdrMagic = 0xA1A2C0DEu;
struct BlockHeader {      // first row of a block
  uint32_t magic, count;
  int32_t status;
  uint32_t pad;
};
// n blocks of base: block q's header is row ((first + q) % ring) * stride. Row indices are u32.
struct RowBlocks {
  const alz_edge_out* base;
  uint32_t stride, first, n, ring;
};
// out[0 .. *n_unique) = one row per distinct packed key among the blocks' n_rows live rows, in ascending key order:
// the type and id words of the key's first row, count, err5xx and lat_sum_ns summed modulo 2^64 and each histogram
// cell modulo 2^32. n_rows = the sum of the header counts, > 0. keys: 2 n_rows words of scratch, idx: 4 n_rows,
// temp: sum_blocks_temp_bytes(n_rows). The count stays on the device. Five own launches.
size_t sum_blocks_temp_bytes(uint32_t n_rows);
void sum_blocks_by_key(const RowBlocks& b, uint32_t n_rows, uint64_t* keys, uint32_t* idx, void* temp,
                       size_t temp_bytes, alz_edge_out* out, uint32_t* n_unique, int sms, cudaStream_t s);
}  // namespace alz
