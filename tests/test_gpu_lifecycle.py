"""GPU: a handle gives back all the device memory it took. Each handle below is sized so that keeping one
handle's tables would cost gigabytes, and it touches every subsystem that allocates: host, packed and raw
staging, a table commit, the GNN state, the socket timelines, a synthetic device stream and the window clock."""
import ctypes as C

import numpy as np
import pytest

from alaz_b200 import abi, capi
from test_gpu_parity import _to_raw

pytestmark = pytest.mark.gpu


def _one_handle_lifetime(seed):
    S, N, NJ = 300, 200_000, 20_000
    t = capi.Topo(S, seed=seed, mix=abi.MIX_ALL)
    ev = t.events(0, N)
    h = capi.Handle(max_endpoints=4 * S, max_pairs=1 << 22, max_batch=1 << 16)   # several staging chunks
    try:
        h.load_tables(t.pod_ip, t.svc_ip)                 # table commit: patch buffers, bloom upload
        h.submit(ev)
        r16, ovf = capi.pack_l7(ev)
        h.submit_packed(r16, ovf)
        h.submit_raw(_to_raw(ev[:NJ]))
        d = h.dev_alloc(N * 32)
        t.fill_device(h, N, N, d)                         # synthetic stream generated on the device
        h.submit_device(d, N)
        h.sync()
        h.dev_free(d)
        assert len(h.flush()) > 0
        scores = np.zeros(h.max_edges, dtype=np.float32)
        n = C.c_size_t(0)
        h._ck(h.L.alz_gnn_score(h.h, scores.ctypes.data_as(C.c_void_p), len(scores), C.byref(n)), "alz_gnn_score")
        assert n.value > 0
        # socket timelines: one open connection per (pid, fd), then lookup, join and the alive export
        tcp = np.zeros(1000, dtype=abi.TCP_REC)
        tcp["pid"] = 1000 + np.arange(1000) // 64
        tcp["fd"] = 3 + np.arange(1000) % 64
        tcp["timestamp_ns"] = 1
        tcp["type"] = 1
        tcp["saddr"] = 0x0A000000 + np.arange(1000)
        tcp["daddr"] = t.pod_ip[np.arange(1000) % len(t.pod_ip)]
        tcp["sport"], tcp["dport"] = 40000, 80
        h.submit_tcp(tcp)
        keys = np.zeros(NJ, dtype=abi.SOCK_QUERY)
        keys["pid"] = tcp["pid"][np.arange(NJ) % 1000]
        keys["fd"] = tcp["fd"][np.arange(NJ) % 1000]
        keys["timestamp_ns"] = 2
        assert h.sock_lookup(keys, now_ns=3)["found"].all()
        h.submit_join(ev[:NJ], keys, now_ns=3)
        h.sock_alive()
        h.flush()
        # time-cut windows: everything below falls into one epoch
        wt0 = int(ev["write_time_ns"][0])
        h.window_clock(wt0, wt0, 1 << 62)
        h.submit(ev[:NJ])
        assert len(h.flush()) > 0
    finally:
        t.close()
        h.close()


def test_destroyed_handles_return_their_device_memory():
    torch = pytest.importorskip("torch")
    _one_handle_lifetime(1)   # first use: modules load, library workspaces appear
    torch.cuda.synchronize()
    free0, _ = torch.cuda.mem_get_info(0)
    for k in range(10):
        _one_handle_lifetime(2 + k)
    torch.cuda.synchronize()
    free1, _ = torch.cuda.mem_get_info(0)
    assert free1 >= free0 - (1 << 30), f"{(free0 - free1) / 2**30:.2f} GiB not returned after 10 handles"
