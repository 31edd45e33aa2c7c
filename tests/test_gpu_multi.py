"""GPU, >= 2 devices: the ranks (threads, one handle per GPU) each ingest their shard, the window
flush merges them with one NCCL all-gather of their sorted rows; every rank must return the
single-rank oracle's edges bit for bit. With overlapping shards every rank sums the rows of a key
found on several ranks from the gathered blocks. Skips on a machine with fewer GPUs; the merge
after the all-gather also runs on one GPU in tests/test_gpu_merge.py."""
import ctypes as C
import threading

import numpy as np
import pytest

import oracle_lib as ol
from alaz_b200 import abi, capi
from helpers import edges_equal, explain_diff

pytestmark = pytest.mark.gpu


def _ngpu():
    import torch
    return torch.cuda.device_count() if torch.cuda.is_available() else 0


@pytest.mark.parametrize("overlap", [False, True])
@pytest.mark.parametrize("world", [2, 4, 8])
def test_ranks_merge_to_the_single_rank_oracle(world, overlap):
    if _ngpu() < world:
        pytest.skip(f"needs {world} GPUs")
    L = capi.load()
    S, N = 2000, 2_000_000
    t = ol.Topo(S, seed=31, mix=abi.MIX_ALL)
    ev = t.events(0, N)
    o = ol.Oracle()
    o.load_tables(t.pod_ip, t.svc_ip)
    o.process(ev, 4)
    if overlap:
        # a caller that does NOT partition cleanly: the first 20k events reach every rank. The merge must
        # notice keys present on several ranks and still return exact sums (sort + sum of the gathered rows).
        for _ in range(world - 1):
            o.process(ev[:20_000])
    exp = o.edges()
    us = np.unique(ev["saddr"])
    own_of = dict(zip(us.tolist(), [L.alz_owner_rank(int(s), world) for s in us]))
    owner = np.array([own_of[int(s)] for s in ev["saddr"]])
    idbuf = (C.c_uint8 * abi.COMM_ID_BYTES)()
    assert L.alz_comm_unique_id(idbuf) == 0
    out, errs = [None] * world, []
    # One process drives all GPUs here, so allocation phases and collective phases are fenced apart:
    # a cudaMalloc on one thread can wait for the other device's NCCL kernel, which waits for this thread.
    # (Production runs one process per GPU, where this cannot happen.)
    bar = threading.Barrier(world, timeout=120)

    def run(rank):
        try:
            h = capi.Handle(device=rank, max_endpoints=4 * S, max_pairs=1 << 17)
            h._ck(L.alz_comm_init(h.h, world, rank, idbuf), "alz_comm_init")
            h.load_tables(t.pod_ip, t.svc_ip)
            mine = ev[owner == rank]
            if overlap:
                mine = np.concatenate([mine, ev[:20_000][owner[:20_000] != rank]])
            h.submit(mine[: len(mine) // 2])
            h.submit(mine[len(mine) // 2:])
            h.sync()
            bar.wait()
            w1 = h.flush()
            w2 = h.flush()           # empty second window on every rank
            out[rank] = (w1, w2, h.stats())
            bar.wait()
            h.close()
        except Exception as e:   # noqa: BLE001
            errs.append((rank, repr(e)))

    th = [threading.Thread(target=run, args=(r,)) for r in range(world)]
    for x in th:
        x.start()
    for x in th:
        x.join(timeout=300)
    assert not errs, errs
    for r in range(world):
        w1, w2, st = out[r]
        assert edges_equal(w1, exp), f"rank {r}: " + explain_diff(w1, exp)
        assert len(w2) == 0
        # canonical order is the same on every rank
        assert w1.tobytes() == out[0][0].tobytes()
    assert sum(out[r][2]["events_in"] for r in range(world)) == N + (20_000 * (world - 1) if overlap else 0)
    assert sum(out[r][2]["rows_emitted"] for r in range(world)) == int(exp["count"].sum())
