"""ctypes binding of libalazgpu.so (include/alazgpu.h). Thin: every method is
one C call. Fails loudly when the library or a CUDA device is missing — there
is no Python or CPU fallback for any of it."""
import ctypes as C
import os

import numpy as np

from . import abi, build as _build


class AlzError(RuntimeError):
    def __init__(self, status, what, detail=""):
        self.status = status
        super().__init__(f"{what}: status {status} {detail}".strip())


_lib = None

# every symbol include/alazgpu.h declares (tests/test_abi.py checks the header against this)
EXPORTS = [
    "alz_create", "alz_destroy", "alz_strerror", "alz_last_cuda_error", "alz_set_stream", "alz_sync",
    "alz_table_upsert", "alz_table_upsert_batch", "alz_table_erase", "alz_table_commit", "alz_submit_l7", "alz_submit_l7_device",
    "alz_submit_l7_packed", "alz_submit_l7_packed_device", "alz_pack_l7",
    "alz_submit_l7_raw", "alz_window_flush", "alz_window_flush_device", "alz_window_fetch", "alz_get_stats",
    "alz_window_clock", "alz_window_epoch", "alz_gnn_score",
    "alz_gnn_score_device", "alz_edge_quantiles", "alz_submit_tcp", "alz_submit_tcp_raw", "alz_sock_lookup", "alz_sock_lookup_at",
    "alz_submit_l7_join", "alz_sock_gc", "alz_sock_alive", "alz_sock_stats", "alz_comm_unique_id", "alz_comm_init",
    "alz_owner_rank",
]


def load(rebuild=False):
    """dlopen alaz_b200/lib/libalazgpu.so (building it first when it is missing and nvcc exists)."""
    global _lib
    if _lib is not None and not rebuild:
        return _lib
    path = os.environ.get("ALZ_LIB_PATH") or _build.LIB   # ALZ_LIB_PATH: A/B runs of two builds on one box
    if rebuild or not os.path.exists(path):
        path = _build.build(force=rebuild)
    L = C.CDLL(path, mode=C.RTLD_GLOBAL)
    vp, u32, u64, sz, i = C.c_void_p, C.c_uint32, C.c_uint64, C.c_size_t, C.c_int
    pp = C.POINTER(vp)
    sig = {
        "alz_create": ([C.POINTER(abi.Config), pp], i),
        "alz_destroy": ([vp], i),
        "alz_strerror": ([i], C.c_char_p),
        "alz_last_cuda_error": ([vp], C.c_char_p),
        "alz_set_stream": ([vp, vp], i),
        "alz_sync": ([vp], i),
        "alz_table_upsert": ([vp, i, u32, u32], i),
        "alz_table_erase": ([vp, i, u32], i),
        "alz_table_upsert_batch": ([vp, i, vp, vp, sz], i),
        "alz_table_commit": ([vp], i),
        "alz_submit_l7": ([vp, vp, sz], i),
        "alz_submit_l7_device": ([vp, vp, sz], i),
        "alz_submit_l7_raw": ([vp, vp, sz], i),
        "alz_submit_l7_packed": ([vp, vp, sz, vp, sz], i),
        "alz_submit_l7_packed_device": ([vp, vp, sz, vp], i),
        "alz_pack_l7": ([vp, sz, vp, vp, sz], C.c_long),
        "alz_window_fetch": ([vp, vp, sz, C.POINTER(sz)], i),
        "alz_window_clock": ([vp, u64, u64, u64], i),
        "alz_window_epoch": ([vp, C.POINTER(u64)], i),
        "alz_pinned_alloc_local": ([vp, sz, pp], i),
        "alz_window_flush": ([vp, vp, sz, C.POINTER(sz)], i),
        "alz_window_flush_device": ([vp, pp, C.POINTER(sz)], i),
        "alz_get_stats": ([vp, C.POINTER(abi.Stats)], i),
        "alz_gnn_score": ([vp, vp, sz, C.POINTER(sz)], i),
        "alz_gnn_score_device": ([vp, pp, C.POINTER(sz)], i),
        "alz_gnn_nodes": ([vp, vp, vp, sz, C.POINTER(sz)], i),
        "alz_merge_blocks_device": ([vp, vp, u32, u32, pp, C.POINTER(sz)], i),
        "alz_edge_quantiles": ([vp, vp, sz, vp], i),
        "alz_submit_tcp": ([vp, vp, sz], i),
        "alz_sock_lookup": ([vp, vp, sz, vp], i),
        "alz_sock_lookup_at": ([vp, vp, sz, vp, u64], i),
        "alz_submit_tcp_raw": ([vp, vp, sz], i),
        "alz_submit_l7_join": ([vp, vp, vp, sz, u64], i),
        "alz_sock_gc": ([vp], i),
        "alz_sock_alive": ([vp, vp, sz, C.POINTER(sz)], i),
        "alz_sock_stats": ([vp, C.POINTER(abi.SockStats)], i),
        "alz_comm_unique_id": ([vp], i),
        "alz_comm_init": ([vp, i, i, vp], i),
        "alz_owner_rank": ([u32, u32], u32),
        "alz_pinned_alloc": ([sz, pp], i),
        "alz_pinned_free": ([vp], i),
        "alz_dev_alloc": ([vp, sz, pp], i),
        "alz_dev_free": ([vp, vp], i),
        "alz_memcpy_h2d": ([vp, vp, vp, sz], i),
        "alz_memcpy_d2h": ([vp, vp, vp, sz], i),
        "alz_fold": ([vp], i),
        "alz_synth_topo_create": ([u32, u64, u32], C.POINTER(abi.SynthTopo)),
        "alz_synth_topo_destroy": ([C.POINTER(abi.SynthTopo)], None),
        "alz_synth_fill": ([C.POINTER(abi.SynthTopo), u64, u64, vp], None),
        "alz_synth_dev_create": ([vp, C.POINTER(abi.SynthTopo), pp], i),
        "alz_synth_dev_fill": ([vp, vp, u64, u64, vp], i),
        "alz_synth_dev_fill_owned": ([vp, vp, u64, u32, u32, vp, u64, C.POINTER(u64), C.POINTER(u64)], i),
        "alz_synth_dev_destroy": ([vp, vp], i),
    }
    if abi.ABI_VERSION < 2:    # A/B timing against a round-1 build (ALZ_LIB_PATH + ALZ_ABI_VERSION=1)
        for k in ("alz_submit_l7_packed", "alz_submit_l7_packed_device", "alz_pack_l7", "alz_window_fetch",
                  "alz_pinned_alloc_local", "alz_table_upsert_batch", "alz_window_clock", "alz_window_epoch",
                  "alz_sock_lookup_at", "alz_submit_l7_join", "alz_sock_gc", "alz_sock_alive", "alz_sock_stats",
                  "alz_submit_tcp_raw"):
            sig.pop(k)
    for name, (args, res) in sig.items():
        f = getattr(L, name)   # AttributeError = header/library mismatch: loud
        f.argtypes, f.restype = args, res
    _lib = L
    return L


def _ptr(a):
    return a.ctypes.data_as(C.c_void_p)


class PinnedBuffer:
    """Library-owned pinned host memory exposed as a numpy array."""

    def __init__(self, n, dtype, handle=None):
        """handle: allocate on the NUMA node next to that handle's GPU (alz_pinned_alloc_local)."""
        self.L = load()
        self.dtype = np.dtype(dtype)
        self.nbytes = int(n) * self.dtype.itemsize
        p = C.c_void_p()
        if handle is not None and abi.ABI_VERSION >= 2:
            rc = self.L.alz_pinned_alloc_local(handle.h, max(self.nbytes, 1), C.byref(p))
        else:
            rc = self.L.alz_pinned_alloc(max(self.nbytes, 1), C.byref(p))
        if rc != 0:
            raise AlzError(rc, "alz_pinned_alloc")
        self.ptr = p.value
        buf = (C.c_char * max(self.nbytes, 1)).from_address(self.ptr)
        self.array = np.frombuffer(buf, dtype=self.dtype, count=int(n))

    def free(self):
        if self.ptr:
            self.array = None
            self.L.alz_pinned_free(self.ptr)
            self.ptr = None


class Handle:
    """One GPU's aggregator instance (alz_handle)."""

    def __init__(self, device=0, max_endpoints=1 << 16, max_pairs=1 << 20, max_edges=0,
                 max_batch=1 << 22, flags=0):
        self.L = load()
        cfg = abi.Config(abi_version=abi.ABI_VERSION, device=device, max_endpoints=max_endpoints,
                         max_pairs=max_pairs, max_edges=max_edges, max_batch=max_batch, flags=flags)
        h = C.c_void_p()
        rc = self.L.alz_create(C.byref(cfg), C.byref(h))
        if rc != 0:
            raise AlzError(rc, "alz_create", self.L.alz_strerror(rc).decode())
        self.h = h
        self.max_edges = max_edges or max_pairs

    def _ck(self, rc, what, allow=()):
        if rc != 0 and rc not in allow:
            raise AlzError(rc, what, self.L.alz_strerror(rc).decode() + " | " +
                           self.L.alz_last_cuda_error(self.h).decode())
        return rc

    def close(self):
        if getattr(self, "h", None):
            self.L.alz_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- tables
    def upsert(self, table, ip, id_):
        self._ck(self.L.alz_table_upsert(self.h, table, int(ip), int(id_)), "alz_table_upsert")

    def erase(self, table, ip):
        self._ck(self.L.alz_table_erase(self.h, table, int(ip)), "alz_table_erase")

    def commit(self):
        self._ck(self.L.alz_table_commit(self.h), "alz_table_commit")

    def upsert_batch(self, table, ips, ids):
        ips = np.ascontiguousarray(ips, dtype=np.uint32)
        ids = np.ascontiguousarray(ids, dtype=np.uint32)
        assert len(ips) == len(ids)
        self._ck(self.L.alz_table_upsert_batch(self.h, table, _ptr(ips), _ptr(ids), len(ips)), "alz_table_upsert_batch")

    def load_tables(self, pod_ip, svc_ip):
        if abi.ABI_VERSION < 2:
            for k, v in enumerate(pod_ip):
                self.upsert(abi.TABLE_POD, int(v), k)
            for k, v in enumerate(svc_ip):
                self.upsert(abi.TABLE_SVC, int(v), k)
        else:
            self.upsert_batch(abi.TABLE_POD, pod_ip, np.arange(len(pod_ip)))
            self.upsert_batch(abi.TABLE_SVC, svc_ip, np.arange(len(svc_ip)))
        self.commit()

    # ---- ingest
    def submit(self, recs):
        recs = np.ascontiguousarray(recs, dtype=abi.L7_REC)
        self._ck(self.L.alz_submit_l7(self.h, _ptr(recs), len(recs)), "alz_submit_l7")

    def submit_ptr(self, host_ptr, n):
        self._ck(self.L.alz_submit_l7(self.h, C.c_void_p(host_ptr), n), "alz_submit_l7")

    def submit_device(self, dev_ptr, n):
        self._ck(self.L.alz_submit_l7_device(self.h, C.c_void_p(dev_ptr), n), "alz_submit_l7_device")

    def submit_packed(self, recs16, overflow=None):
        recs16 = np.ascontiguousarray(recs16, dtype=abi.L7_REC16)
        ovf = np.ascontiguousarray(overflow if overflow is not None else np.zeros(0, np.uint64), dtype=np.uint64)
        self._ck(self.L.alz_submit_l7_packed(self.h, _ptr(recs16), len(recs16), _ptr(ovf) if len(ovf) else None,
                                             len(ovf)), "alz_submit_l7_packed")

    def submit_packed_ptr(self, host_ptr, n, ovf_ptr=None, n_ovf=0):
        self._ck(self.L.alz_submit_l7_packed(self.h, C.c_void_p(host_ptr), n, C.c_void_p(ovf_ptr) if ovf_ptr else None,
                                             n_ovf), "alz_submit_l7_packed")

    def submit_raw(self, raw):
        raw = np.ascontiguousarray(raw, dtype=np.uint8)
        n = raw.size // abi.BPF_L7_EVENT_SIZE
        self._ck(self.L.alz_submit_l7_raw(self.h, _ptr(raw), n), "alz_submit_l7_raw")

    def submit_raw_ptr(self, host_ptr, n):
        self._ck(self.L.alz_submit_l7_raw(self.h, C.c_void_p(host_ptr), n), "alz_submit_l7_raw")

    # ---- results
    def flush(self, cap=None):
        cap = self.max_edges if cap is None else cap
        out = np.zeros(cap, dtype=abi.EDGE_OUT)
        n = C.c_size_t(0)
        self._ck(self.L.alz_window_flush(self.h, _ptr(out), cap, C.byref(n)), "alz_window_flush")
        return out[: n.value].copy()

    def flush_device(self):
        p = C.c_void_p()
        n = C.c_size_t(0)
        self._ck(self.L.alz_window_flush_device(self.h, C.byref(p), C.byref(n)), "alz_window_flush_device")
        return p.value, n.value

    def stats(self):
        st = abi.Stats()
        self._ck(self.L.alz_get_stats(self.h, C.byref(st)), "alz_get_stats")
        return st.as_dict()

    # ---- tcp_state sink + socket timelines (alz_sock.cu) ----
    def submit_tcp(self, recs):
        recs = np.ascontiguousarray(recs, dtype=abi.TCP_REC)
        self._ck(self.L.alz_submit_tcp(self.h, _ptr(recs), len(recs)), "alz_submit_tcp")

    def sock_lookup(self, q, now_ns=None):
        q = np.ascontiguousarray(q, dtype=abi.SOCK_QUERY)
        out = np.zeros(len(q), dtype=abi.SOCK_RESULT)
        if now_ns is None:
            self._ck(self.L.alz_sock_lookup(self.h, _ptr(q), len(q), _ptr(out)), "alz_sock_lookup")
        else:
            self._ck(self.L.alz_sock_lookup_at(self.h, _ptr(q), len(q), _ptr(out), int(now_ns)), "alz_sock_lookup_at")
        return out

    def submit_join(self, recs, keys, now_ns=0):
        recs = np.ascontiguousarray(recs, dtype=abi.L7_REC)
        keys = np.ascontiguousarray(keys, dtype=abi.SOCK_QUERY)
        assert len(recs) == len(keys)
        self._ck(self.L.alz_submit_l7_join(self.h, _ptr(recs), _ptr(keys), len(recs), int(now_ns)), "alz_submit_l7_join")

    def sock_gc(self):
        self._ck(self.L.alz_sock_gc(self.h), "alz_sock_gc")

    def sock_alive(self, cap=1 << 20):
        out = np.zeros(cap, dtype=abi.ALIVE_CONN)
        n = C.c_size_t(0)
        self._ck(self.L.alz_sock_alive(self.h, _ptr(out), cap, C.byref(n)), "alz_sock_alive")
        return out[: n.value]

    def sock_stats(self):
        st = abi.SockStats()
        self._ck(self.L.alz_sock_stats(self.h, C.byref(st)), "alz_sock_stats")
        return st.as_dict()

    def window_clock(self, first_kernel_ns, first_user_ns, window_ns):
        self._ck(self.L.alz_window_clock(self.h, int(first_kernel_ns), int(first_user_ns), int(window_ns)),
                 "alz_window_clock")

    def window_epoch(self):
        e = C.c_uint64(0)
        self._ck(self.L.alz_window_epoch(self.h, C.byref(e)), "alz_window_epoch")
        return e.value

    def fold(self):
        self._ck(self.L.alz_fold(self.h), "alz_fold")

    def sync(self):
        self._ck(self.L.alz_sync(self.h), "alz_sync")

    def set_stream(self, cuda_stream):
        self._ck(self.L.alz_set_stream(self.h, C.c_void_p(cuda_stream)), "alz_set_stream")

    # ---- device helpers (bench/test support)
    def dev_alloc(self, nbytes):
        p = C.c_void_p()
        self._ck(self.L.alz_dev_alloc(self.h, nbytes, C.byref(p)), "alz_dev_alloc")
        return p.value

    def dev_free(self, p):
        self._ck(self.L.alz_dev_free(self.h, C.c_void_p(p)), "alz_dev_free")

    def h2d(self, dev_ptr, arr):
        arr = np.ascontiguousarray(arr)
        self._ck(self.L.alz_memcpy_h2d(self.h, C.c_void_p(dev_ptr), _ptr(arr), arr.nbytes), "alz_memcpy_h2d")

    def d2h(self, dev_ptr, n, dtype):
        out = np.zeros(n, dtype=dtype)
        self._ck(self.L.alz_memcpy_d2h(self.h, _ptr(out), C.c_void_p(dev_ptr), out.nbytes), "alz_memcpy_d2h")
        return out


def pack_l7(recs):
    """alz_pack_l7: 32-B records -> (16-B records, overflow durations)."""
    L = load()
    recs = np.ascontiguousarray(recs, dtype=abi.L7_REC)
    out = np.zeros(len(recs), dtype=abi.L7_REC16)
    cap = max(16, len(recs) // 64)
    while True:
        ovf = np.zeros(cap, dtype=np.uint64)
        k = L.alz_pack_l7(_ptr(recs), len(recs), _ptr(out), _ptr(ovf), cap)
        if k >= 0:
            return out, ovf[:k].copy()
        if cap >= len(recs):
            raise AlzError(abi.E_INVAL, "alz_pack_l7")
        cap = len(recs)


class Topo:
    """Synthetic cluster + stream tables via libalazgpu's own copy of the generator."""

    def __init__(self, n_services, seed=0xA1A20000, mix=abi.MIX_SURVEY):
        self.L = load()
        self.p = self.L.alz_synth_topo_create(n_services, seed, mix)
        if not self.p:
            raise MemoryError("alz_synth_topo_create")
        t = self.p.contents
        self.n_services, self.n_pods, self.n_edges = t.n_services, t.n_pods, t.n_edges
        self.pod_ip = np.ctypeslib.as_array(t.pod_ip, (t.n_pods,)).copy()
        self.svc_ip = np.ctypeslib.as_array(t.svc_ip, (t.n_services,)).copy()
        self.dev = None
        self._handle = None

    def events(self, first, n):
        out = np.zeros(n, dtype=abi.L7_REC)
        self.L.alz_synth_fill(self.p, int(first), int(n), _ptr(out))
        return out

    def to_device(self, handle):
        d = C.c_void_p()
        handle._ck(self.L.alz_synth_dev_create(handle.h, self.p, C.byref(d)), "alz_synth_dev_create")
        self.dev, self._handle = d, handle
        return d

    def fill_device(self, handle, first, n, dev_ptr):
        if self.dev is None:
            self.to_device(handle)
        handle._ck(self.L.alz_synth_dev_fill(handle.h, self.dev, int(first), int(n), C.c_void_p(dev_ptr)),
                   "alz_synth_dev_fill")

    def close(self):
        if self.dev is not None and self._handle is not None and getattr(self._handle, "h", None):
            self.L.alz_synth_dev_destroy(self._handle.h, self.dev)
        self.dev = None
        if self.p:
            self.L.alz_synth_topo_destroy(self.p)
            self.p = None
