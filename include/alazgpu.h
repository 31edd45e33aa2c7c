/*
 * alazgpu.h — C ABI of libalazgpu: the B200-native replacement for the
 * service-map aggregation hot path of getanteon/alaz (reference @ 828b997f).
 *
 * The reference has no FFI boundary for this path; the seam this library sits
 * behind is the aggregator's channel-in / DataStore-out pair:
 *   in : *l7_req.L7Event              ebpf/l7_req/l7.go:396-421 (from bpfL7Event, l7.go:345-369)
 *        *tcp_state.TcpConnectEvent   ebpf/tcp_state/tcp.go:75-84 (from BpfTcpEvent, tcp.go:63-72)
 *        k8s.K8sResourceMessage       k8s/informer.go:236-240 -> processPod/processSvc
 *                                     aggregator/persist.go:55-71, 114-130
 *   out: datastore.DataStore.PersistRequest  datastore/datastore.go:13
 *                                     (one row per request; this library instead
 *                                     returns the rows grouped by (From,To))
 *
 * Rules: plain C, flat PODs, no pointer is retained past the call that
 * received it (cgo rule), every entry point returns 0 on success or a negative
 * alz_status. No exceptions cross the boundary. One handle drives one GPU.
 * INTEGRATION.md shows the cgo binding a maintainer would add.
 */
#ifndef ALAZGPU_H
#define ALAZGPU_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ALZ_ABI_VERSION 2

/* ---- status codes -------------------------------------------------------- */
typedef enum alz_status {
  ALZ_OK = 0,
  ALZ_E_INVAL = -1,      /* bad argument */
  ALZ_E_NOMEM = -2,      /* host or device allocation failed */
  ALZ_E_CUDA = -3,       /* CUDA runtime error (alz_last_cuda_error) */
  ALZ_E_NODEVICE = -4,   /* no CUDA device: there is NO CPU fallback */
  ALZ_E_CAPACITY = -5,   /* pair/edge dictionary or output buffer too small */
  ALZ_E_STATE = -6,      /* call not valid in this state (e.g. no comm) */
  ALZ_E_NCCL = -7,       /* NCCL error or libnccl.so.2 not loadable */
  ALZ_E_UNSUPPORTED = -8
} alz_status;

/* ---- wire enums: values equal the eBPF side (ebpf/l7_req/l7.go:19-29) ----- */
enum {
  ALZ_PROTO_UNKNOWN = 0, ALZ_PROTO_HTTP = 1, ALZ_PROTO_AMQP = 2,
  ALZ_PROTO_POSTGRES = 3, ALZ_PROTO_HTTP2 = 4, ALZ_PROTO_REDIS = 5,
  ALZ_PROTO_KAFKA = 6, ALZ_PROTO_MYSQL = 7, ALZ_PROTO_MONGO = 8
};
/* method enums that change routing (l7.go:91-95, 120-125) */
enum { ALZ_AMQP_PUBLISH = 1, ALZ_AMQP_DELIVER = 2 };
enum { ALZ_REDIS_COMMAND = 1, ALZ_REDIS_PUSHED_EVENT = 2, ALZ_REDIS_PING = 3 };

/* method_flags byte of alz_l7_rec */
#define ALZ_MF_METHOD_MASK 0x3Fu
#define ALZ_MF_PAYLOAD_REJECT 0x40u /* host-side payload parser says the reference
                                       would drop the row: Postgres/MySQL text query
                                       without SQL keyword (aggregator/data.go:1440-1443,
                                       1495-1497), Mongo parse failure (:1252-1255) */
#define ALZ_MF_TLS 0x80u

/* protocol byte of alz_l7_rec: bit 6 says "daddr holds a host id, not an address". The caller sets it for an
 * HTTP event whose payload carried a Host header AND whose daddr is neither a service nor a pod in the
 * tables as committed so far — the case in which setFromToV2 keys the destination by the header
 * (aggregator/data.go:851-854). The caller owns both the payload parser and the interner of header strings
 * (strings never cross this ABI), and it owns the tables it upserts here, so it can decide this exactly
 * as the reference does; the device keeps such events in their own key space. */
#define ALZ_PROTO_F_HOSTKEY 0x40u

/* node kinds of an edge end (aggregator/data.go POD/SVC/OUTBOUND) */
enum { ALZ_NODE_POD = 0, ALZ_NODE_SVC = 1, ALZ_NODE_OUTBOUND = 2,
       ALZ_NODE_OUTBOUND_HOST = 3 /* outbound destination keyed by the HTTP Host header (aggregator/data.go:851-854);
                                     value = the caller's dense id of the header string */ };
/* tables of the join's build side (aggregator/cluster.go:15-16) */
enum { ALZ_TABLE_POD = 0, ALZ_TABLE_SVC = 1 };

#define ALZ_NB 64 /* latency histogram buckets, see docs/SPEC.md §4 */

/* ---- records -------------------------------------------------------------- */

/* Compact L7 record, 32 B. Lossless w.r.t. struct l7_event (ebpf/c/l7.c:19-47)
 * for everything resolve/emit/reduce reads; pid/fd/payload stay host-side.
 * saddr/daddr are host-order u32 with the first octet in the MSB, exactly the
 * integer the reference feeds to IntToIPv4 (aggregator/data.go:1751-1767). */
typedef struct alz_l7_rec {
  uint32_t saddr;
  uint32_t daddr;
  uint16_t sport;
  uint16_t dport;
  uint16_t status;       /* l7_event.status saturated to 65535 */
  uint8_t protocol;      /* ALZ_PROTO_* */
  uint8_t method_flags;  /* method | ALZ_MF_* */
  uint64_t duration_ns;  /* l7_event.duration (l7.c:788) */
  uint64_t write_time_ns;
} alz_l7_rec;

/* Packed L7 record, 16 B: the fields of alz_l7_rec that resolve/emit/reduce read, for callers whose
 * events cross PCIe (half the bytes per event on the wire). Lossless: a duration >= 2^32 ns is stored
 * in the overflow array handed to the same submit call, the record carries its index there and bit 7
 * of `protocol` is set. No ports and no write time: windows of packed records are cut by the caller. */
typedef struct alz_l7_rec16 {
  uint32_t saddr;
  uint32_t daddr;
  uint16_t status;
  uint8_t protocol;      /* ALZ_PROTO_* | ALZ_REC16_DUR_OVERFLOW */
  uint8_t method_flags;  /* method | ALZ_MF_* */
  uint32_t duration_ns;  /* or index into the overflow array */
} alz_l7_rec16;
#define ALZ_REC16_DUR_OVERFLOW 0x80u

/* tcp_state record, 40 B, from struct tcp_event (ebpf/c/struct.h:2-12).
 * type: 1=ESTABLISHED 5=CLOSED (ebpf/tcp_state/tcp.go:19-25); addresses as in
 * alz_l7_rec (first octet in MSB). */
typedef struct alz_tcp_rec {
  uint64_t fd;
  uint64_t timestamp_ns;
  uint32_t pid;
  uint32_t saddr;
  uint32_t daddr;
  uint16_t sport;
  uint16_t dport;
  uint32_t type;
  uint32_t _pad;
} alz_tcp_rec;

/* query / result of the temporal socket join (SocketLine.GetValue,
 * aggregator/sock_num_line.go:82-158) */
typedef struct alz_sock_query {
  uint64_t fd;
  uint64_t timestamp_ns;
  uint32_t pid;
  uint32_t _pad;
} alz_sock_query;

typedef struct alz_sock_result {
  uint32_t found; /* 1 = SockInfo returned, 0 = the reference returns an error */
  uint32_t saddr;
  uint32_t daddr;
  uint16_t sport;
  uint16_t dport;
} alz_sock_result;

/* One edge of the service graph for one window. Rows the reference would have
 * handed to PersistRequest (datastore/backend.go:819-847), grouped by
 * (FromType,FromUID,ToType,ToUID). from/to are the caller's dense ids for pod
 * and service ends and the raw IPv4 for outbound ends (aggregator/data.go:862). */
typedef struct alz_edge_out {
  uint8_t from_type; /* ALZ_NODE_* */
  uint8_t to_type;
  uint8_t _pad[6];
  uint32_t from;
  uint32_t to;
  uint64_t count;
  uint64_t err5xx;
  uint64_t lat_sum_ns;
  uint32_t hist[ALZ_NB];
} alz_edge_out;

typedef struct alz_config {
  uint32_t abi_version;     /* ALZ_ABI_VERSION */
  int32_t device;           /* CUDA device ordinal */
  uint32_t max_endpoints;   /* pods + services the tables must hold */
  uint32_t max_pairs;       /* distinct (saddr,daddr) pairs per window */
  uint32_t max_edges;       /* distinct edges per window */
  uint32_t max_batch;       /* largest n of one alz_submit_l7 (host staging) */
  uint32_t flags;           /* ALZ_CFG_* */
  uint32_t _reserved[9];
} alz_config;

#define ALZ_CFG_EAGER_JOIN 0x1u /* resolve every event through the tables before
                                   reducing (the textbook plan) instead of
                                   reducing per socket pair and joining the
                                   distinct pairs (default); same results */

#define ALZ_CFG_NO_SMEM_CACHE 0x2u /* ingest without the per-CTA shared-memory cache of
                                      hot socket pairs (profiling comparison only) */

typedef struct alz_stats {
  uint64_t events_in;        /* records submitted */
  uint64_t rows_emitted;     /* rows the reference would have persisted */
  uint64_t not_request;      /* protocol switch emits no request row
                                (HTTP2/KAFKA/UNKNOWN, payload reject) */
  uint64_t src_unresolved;   /* setFromToV2 error: saddr is not a pod
                                (aggregator/data.go:829-832) */
  uint64_t pairs_live;
  uint64_t edges_live;
  uint64_t tcp_events_in;
  uint64_t tcp_localhost_dropped; /* aggregator/data.go:409, 455 */
  uint64_t capacity_events;  /* events lost to an exhausted pair/edge table (cumulative) */
  uint64_t windows;          /* windows flushed */
  uint64_t kernel_launches;  /* kernels of this library launched so far (CUB passes, memsets, copies not counted) */
  uint64_t collective_bytes_last; /* bytes this rank contributed to / received from the last window's collective */
  uint64_t flush_local_us_last;   /* device time of the last flush up to the cross-rank merge */
  uint64_t merge_us_last;         /* device time of the last cross-rank merge (0 on one rank) */
  uint64_t late_events;           /* time-cut windows: records older than the open window (cumulative) */
  uint64_t deferred_events;       /* time-cut windows: records waiting on the device for their window */
} alz_stats;

typedef struct alz_handle alz_handle;

/* ---- lifecycle -------------------------------------------------------------- */
int alz_create(const alz_config* cfg, alz_handle** out);
int alz_destroy(alz_handle* h);
const char* alz_strerror(int status);
const char* alz_last_cuda_error(alz_handle* h);
/* Run all device work of this handle on `cuda_stream` (a cudaStream_t; 0 =
 * the library's own stream). Lets a host time the work with its own events. */
int alz_set_stream(alz_handle* h, void* cuda_stream);
int alz_sync(alz_handle* h);

/* ---- join build side: replaces ClusterInfo map writes ------------------------
 * (aggregator/persist.go:55-71 PodIPToPodUid, :114-130 ServiceIPToServiceUid).
 * UID strings stay with the caller, who interns them to dense ids < 2^29.
 * Single writer. Changes become visible to submits after alz_table_commit,
 * which first folds everything already submitted through the old tables, so
 * each event is resolved by the tables in force when it was submitted. */
int alz_table_upsert(alz_handle* h, int table, uint32_t ipv4, uint32_t id);
int alz_table_erase(alz_handle* h, int table, uint32_t ipv4);
/* n upserts in one call (informer resync / initial list: k8s/informer.go hands the whole cluster at start) */
int alz_table_upsert_batch(alz_handle* h, int table, const uint32_t* ipv4, const uint32_t* ids, size_t n);
int alz_table_commit(alz_handle* h);

/* ---- event ingest: replaces processL7 .. PersistRequest --------------------
 * (aggregator/data.go:1364-1383 dispatch, :1081-1362 row build,
 *  :827-870 setFromToV2). The alz_submit_* calls may be made from many OS threads at once, like the
 * reference's 4*NumCPU processL7 workers (aggregator/data.go:230-232): callers copy into separate
 * pinned staging slots in parallel and only the enqueue is serialised. A flush or table commit is
 * ordered after every submit that returned before it was called. */
int alz_submit_l7(alz_handle* h, const alz_l7_rec* host_recs, size_t n);
/* same, records already resident in this GPU's HBM */
int alz_submit_l7_device(alz_handle* h, const alz_l7_rec* dev_recs, size_t n);
/* same, 16-B packed records (host memory); dur_overflow[n_overflow] holds the durations the records
 * index (may be NULL when n_overflow == 0) */
int alz_submit_l7_packed(alz_handle* h, const alz_l7_rec16* host_recs, size_t n,
                         const uint64_t* dur_overflow, size_t n_overflow);
int alz_submit_l7_packed_device(alz_handle* h, const alz_l7_rec16* dev_recs, size_t n,
                                const uint64_t* dev_dur_overflow);
/* host-side packer: alz_l7_rec[n] -> alz_l7_rec16[n]; overflow durations appended to dur_overflow
 * (capacity cap_overflow). Returns the number of overflow entries written, or -1 if cap is too small. */
long alz_pack_l7(const alz_l7_rec* recs, size_t n, alz_l7_rec16* out, uint64_t* dur_overflow, size_t cap_overflow);
/* n raw perf samples exactly as perf.Reader yields them: 1096-B
 * struct l7_event (ebpf/l7_req/l7.go:345-369, :704); payload ignored. */
int alz_submit_l7_raw(alz_handle* h, const void* host_bpf_l7_events, size_t n);
#define ALZ_BPF_L7_EVENT_SIZE 1096

/* ---- window result: the grouped rows ----------------------------------------
 * Folds pending pairs, (multi-GPU: merges all ranks, one all-gather of their
 * sorted rows), writes the live edges in ascending packed-key order
 * (docs/SPEC.md §3; the same order on every rank) and resets the window. n_out is always set to the number of live edges; if
 * cap is too small returns ALZ_E_CAPACITY and keeps the window. */
int alz_window_flush(alz_handle* h, alz_edge_out* out, size_t cap, size_t* n_out);
/* as above but leaves the result on the device for alz_gnn_score / peers;
 * *dev_edges stays valid until the next flush on this handle */
int alz_window_flush_device(alz_handle* h, const alz_edge_out** dev_edges, size_t* n_out);
/* the rows of the last flushed window once more. On a multi-rank handle the merge consumes the window on
 * every rank, so a flush whose `cap` was too small cannot keep it: it returns ALZ_E_CAPACITY with *n_out set
 * and the merged rows stay fetchable here until the next flush. */
int alz_window_fetch(alz_handle* h, alz_edge_out* out, size_t cap, size_t* n_out);
int alz_get_stats(alz_handle* h, alz_stats* out);

/* ---- time-cut windows (SURVEY §8 row R13, docs/SPEC.md §8) ---------------------
 * By default a window is whatever was submitted between two flushes. After alz_window_clock the records' own
 * write_time decides: epoch(t) = convertKernelTimeToUserspaceTime(t) / window_ns with
 * convertKernelTimeToUserspaceTime(t) = first_user_ns - (first_kernel_ns - t) (aggregator/data.go:1740-1743;
 * l7_req.FirstKernelTime / FirstUserspaceTime). The open window is the epoch of the first record submitted
 * afterwards. A record of a later epoch is kept on the device and submitted again by the flush that opens its
 * window; a record of an earlier epoch is late: it is reduced into the open window and counted
 * (alz_stats.late_events). Each alz_window_flush* closes the open epoch and opens the next one. Only 32-byte
 * records carry a write time: packed submits return ALZ_E_STATE while the clock is set. window_ns = 0 turns
 * the clock off again. */
int alz_window_clock(alz_handle* h, uint64_t first_kernel_ns, uint64_t first_user_ns, uint64_t window_ns);
/* epoch of the open window; ALZ_E_STATE until the first record has been submitted */
int alz_window_epoch(alz_handle* h, uint64_t* epoch);

/* ---- GNN anomaly pass over the last flushed window (docs/SPEC.md §6) -------- */
int alz_gnn_score(alz_handle* h, float* edge_scores, size_t cap, size_t* n_out);
/* same, scores left on the device (valid until the next call on this handle) */
int alz_gnn_score_device(alz_handle* h, const float** dev_scores, size_t* n_out);
/* quantiles from the histogram, the same float64 interpolation the scores use */
int alz_edge_quantiles(const alz_edge_out* e, const double* qs, size_t nq, double* out_ns);

/* ---- rollups over recent windows (docs/SPEC.md §12) -------------------------
 * alz_history_init keeps the edge rows of the last `depth` flushed windows on the device, starting with the
 * next flush. A window enters exactly when alz_stats.windows counts it: empty windows too (k windows are k
 * clock periods), and a window that lost rows to capacity, as it was returned. A single-rank alz_window_flush
 * that returns ALZ_E_CAPACITY before consuming the window, and a multi-rank merge larger than max_edges, do
 * not enter. The ring, depth * (max_edges + 1) rows of 296 B, is allocated here, all or nothing; no flush
 * allocates. ALZ_E_INVAL: depth == 0 or depth * (max_edges + 1) >= 2^32. ALZ_E_STATE: history is already on.
 * ALZ_E_NOMEM leaves the handle without history; the call may be repeated. */
int alz_history_init(alz_handle* h, uint32_t depth);
/* *held: windows held (at most depth); *newest: the alz_stats.windows ordinal of the newest one (0 while none
 * is held). With alz_window_clock, a window's epoch is its ordinal plus a fixed offset. ALZ_E_STATE without
 * history. */
int alz_history_info(alz_handle* h, uint32_t* held, uint64_t* newest);
/* The sum of the newest min(k, held) windows: one row per distinct packed edge key, in ascending key order
 * (docs/SPEC.md §3). Type and id words come from the key; count, err5xx and lat_sum_ns add modulo 2^64, each
 * hist cell modulo 2^32. ALZ_E_INVAL: k == 0. ALZ_E_STATE: no history. held == 0 gives 0 rows. No side effects:
 * the open window, the last flush (alz_window_fetch, alz_gnn_score), the history and the next flush are as
 * they were. *n_out is always set; if cap is too small returns ALZ_E_CAPACITY and nothing is lost. One stream
 * synchronisation per call. Local: no collective on a multi-rank handle, and the same bytes on every rank. */
int alz_rollup(alz_handle* h, uint32_t k, alz_edge_out* out, size_t cap, size_t* n_out);
/* as above but leaves the rows on the device; *dev_edges stays valid until the next alz_rollup* call on this
 * handle */
int alz_rollup_device(alz_handle* h, uint32_t k, const alz_edge_out** dev_edges, size_t* n_out);

/* ---- tcp_state sink + temporal socket join (SURVEY §8f.2) -------------------
 * alz_submit_tcp replaces processTcpConnect (aggregator/data.go:404-506) +
 * SocketLine.AddValue (sock_num_line.go:62-80); alz_sock_lookup replaces
 * SocketLine.GetValue (sock_num_line.go:82-158). */
int alz_submit_tcp(alz_handle* h, const alz_tcp_rec* host_recs, size_t n);
/* n raw perf samples of the tcp_connect_events ring exactly as perf.Reader yields
 * them: struct tcp_event (ebpf/c/struct.h:2-12; BpfTcpEvent, ebpf/tcp_state/
 * tcp.go:63-72), 64 bytes with its tail padding. The IPv4 sits in the first four
 * address bytes, first octet first (tcp.go:241-242). */
#define ALZ_BPF_TCP_EVENT_SIZE 64
int alz_submit_tcp_raw(alz_handle* h, const void* host_bpf_tcp_events, size_t n);
int alz_sock_lookup(alz_handle* h, const alz_sock_query* host_q, size_t n,
                    alz_sock_result* host_out);
/* the same with the caller's clock for the LastMatch stamps (the reference uses
 * time.Now(), sock_num_line.go:96, :156); alz_sock_lookup passes CLOCK_REALTIME */
int alz_sock_lookup_at(alz_handle* h, const alz_sock_query* host_q, size_t n,
                       alz_sock_result* host_out, uint64_t now_ns);
/* L7 events that may carry an empty 5-tuple (get_sock miss, ebpf/c/l7.c:313-314):
 * host_keys[i] = (Pid, Fd, WriteTimeNs) of host_recs[i]. Records with saddr == 0
 * and daddr == 0 take their addresses from the (pid, fd) timeline on the device
 * (findRelatedSocket, aggregator/data.go:1407-1429), then the whole batch is
 * ingested like alz_submit_l7. A miss leaves the zeros and the event is dropped
 * and counted as src_unresolved (0.0.0.0 is no pod, data.go:829-832).
 * now_ns: LastMatch stamp, 0 = CLOCK_REALTIME. */
int alz_submit_l7_join(alz_handle* h, const alz_l7_rec* host_recs,
                       const alz_sock_query* host_keys, size_t n, uint64_t now_ns);
/* One tick of clearSocketLines (aggregator/data.go:1681-1716): SocketLine.
 * DeleteUnused (sock_num_line.go:160-209) on every line. */
int alz_sock_gc(alz_handle* h);
/* sendOpenConnection (aggregator/data.go:1628-1679) for every line: one row per
 * line whose last value is an open socket with a pod at its source address.
 * Rows come in no particular order. *n_out = rows there are; ALZ_E_CAPACITY
 * (first `cap` rows written) when cap was too small. Resolves against the
 * tables as of the last alz_table_commit. */
typedef struct alz_alive_conn {
  uint32_t from_ip;
  uint32_t from_id;   /* pod id */
  uint32_t to_ip;
  uint32_t to_id;     /* pod / service id; the raw address for ALZ_NODE_OUTBOUND */
  uint16_t from_port;
  uint16_t to_port;
  uint8_t to_type;    /* ALZ_NODE_* */
  uint8_t _pad[3];
} alz_alive_conn;
int alz_sock_alive(alz_handle* h, alz_alive_conn* host_out, size_t cap, size_t* n_out);
typedef struct alz_sock_stats_t {
  uint64_t lines;          /* (pid, fd) timelines */
  uint64_t pool_records;   /* device pool: records allocated to segments */
  uint64_t pool_garbage;   /* ... of which in segments left behind by grown lines */
  uint64_t syncs;          /* host -> device syncs so far */
  uint64_t sync_ops;       /* inserts they carried */
  uint64_t sync_bytes;     /* bytes they copied */
  uint64_t repools;        /* times the pool was re-laid (full or half garbage) */
  uint64_t joined_events;  /* alz_submit_l7_join: empty 5-tuples filled */
} alz_sock_stats_t;
int alz_sock_stats(alz_handle* h, alz_sock_stats_t* st);

/* ---- multi-GPU: one rank per GPU, events pre-partitioned by alz_owner_rank ---- */
#define ALZ_COMM_ID_BYTES 128
int alz_comm_unique_id(void* out_id /* ALZ_COMM_ID_BYTES */);
/* up to 64 ranks: ALZ_E_UNSUPPORTED for more */
int alz_comm_init(alz_handle* h, int nranks, int rank, const void* id);
/* rank that owns an event: hash of the source address only, so every event of
 * an edge lands on one rank before any resolve (From is the pod at saddr,
 * aggregator/data.go:834-835) */
uint32_t alz_owner_rank(uint32_t saddr, uint32_t nranks);

#ifdef __cplusplus
}
#endif
#endif /* ALAZGPU_H */
