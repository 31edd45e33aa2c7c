/*
 * alazgpu_synth.h — bench/test support exported by libalazgpu next to the
 * product ABI: device-memory helpers and the device-side synthetic l7_req
 * stream (alaz_b200/synth/alz_synth.h). Not part of the drop-in boundary.
 */
#ifndef ALAZGPU_SYNTH_H
#define ALAZGPU_SYNTH_H
#include "alazgpu.h"
#include "../alaz_b200/synth/alz_synth.h"
#ifdef __cplusplus
extern "C" {
#endif

/* pinned host buffers: alz_submit_l7 / alz_submit_l7_raw from such a buffer skip
 * the staging memcpy (the Go side can fill them directly: C memory, cgo-legal) */
int alz_pinned_alloc(size_t bytes, void** out);
/* same, on the NUMA node next to the handle's GPU (8 ranks feeding 8 GPUs: staging on the remote socket
 * halves the reachable H2D rate) */
int alz_pinned_alloc_local(alz_handle* h, size_t bytes, void** out);
int alz_pinned_free(void* p);

int alz_dev_alloc(alz_handle* h, size_t bytes, void** out);
int alz_dev_free(alz_handle* h, void* p);
int alz_memcpy_h2d(alz_handle* h, void* dst, const void* src, size_t bytes);
int alz_memcpy_d2h(alz_handle* h, void* dst, const void* src, size_t bytes);
/* fold pending socket pairs into the edge accumulators now (flush does it anyway) */
int alz_fold(alz_handle* h);

/* test/debug: node keys ((kind << 32) | value, ascending) and layer-2 embeddings [n x 64] of the last GNN pass */
int alz_gnn_nodes(alz_handle* h, uint64_t* node_keys, float* h2, size_t cap, size_t* n_out);
/* test: the multi-rank flush's merge after its all-gather, without the collective and the window reset.
 * dev_blocks: nranks blocks as the ranks send them, each a header row {magic, count, status} followed by
 * block_rows rows of which `count` are live, in ascending packed-key order. The merged rows go to the handle's
 * flush output (*dev_out, *n_out: as alz_window_flush_device). Returns a block's nonzero status, or
 * ALZ_E_CAPACITY when a count exceeds block_rows or the rows exceed max_edges. */
int alz_merge_blocks_device(alz_handle* h, const alz_edge_out* dev_blocks, uint32_t nranks, uint32_t block_rows,
                            const alz_edge_out** dev_out, size_t* n_out);

typedef struct alz_synth_dev alz_synth_dev;
int alz_synth_dev_create(alz_handle* h, const alz_synth_topo* topo, alz_synth_dev** out);
int alz_synth_dev_fill(alz_handle* h, alz_synth_dev* d, uint64_t first, uint64_t n, alz_l7_rec* dev_out);
int alz_synth_dev_fill_owned(alz_handle* h, alz_synth_dev* d, uint64_t first, uint32_t nranks, uint32_t rank,
                             alz_l7_rec* dev_out, uint64_t want, uint64_t* n_written, uint64_t* n_scanned);
int alz_synth_dev_destroy(alz_handle* h, alz_synth_dev* d);

#ifdef __cplusplus
}
#endif
#endif
