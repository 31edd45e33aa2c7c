"""GPU: the window history and its rollups (docs/SPEC.md §12). alz_rollup(k) must equal, byte for byte and in
packed-key order, an oracle that saw the events of the newest k flushed windows and was never reset, and a numpy
sum of those windows' flushed rows. A handle without history must not change, and a rollup must leave the flush
output, the GNN pass and the next flush as they were."""
import ctypes as C
import threading

import numpy as np
import pytest

import oracle_lib as ol
from alaz_b200 import abi, capi
from helpers import edges_equal, explain_diff, pack_key

pytestmark = pytest.mark.gpu

TIMING = ("flush_local_us_last", "merge_us_last")


def _by_key(rows):
    keys = np.array([pack_key(e) for e in rows], dtype=np.uint64)
    return rows[np.argsort(keys, kind="stable")]


def _same(got, exp, what):
    exp = _by_key(exp)
    assert edges_equal(got, exp), f"{what}: " + explain_diff(got, exp)
    assert got.tobytes() == exp.tobytes(), what


def _numpy_rollup(windows):
    """Sum by packed key of flushed rows: u64 counters and u32 histogram cells, each wrapping."""
    rows = np.concatenate(windows) if windows else np.zeros(0, dtype=abi.EDGE_OUT)
    keys = np.array([pack_key(e) for e in rows], dtype=np.uint64)
    uk, first, inv = np.unique(keys, return_index=True, return_inverse=True)
    out = np.zeros(len(uk), dtype=abi.EDGE_OUT)
    for f in ("from_type", "to_type", "from", "to"):
        out[f] = rows[f][first]
    for f in ("count", "err5xx", "lat_sum_ns", "hist"):
        np.add.at(out[f], inv, rows[f])   # a field view: adds in place
    return out


def _rc_rollup(h, k, cap):
    out = np.zeros(max(cap, 1), dtype=abi.EDGE_OUT)
    n = C.c_size_t(0)
    rc = h.L.alz_rollup(h.h, k, out.ctypes.data_as(C.c_void_p), cap, C.byref(n))
    return rc, n.value, out[: n.value]


def _fetch(h):
    out = np.zeros(h.max_edges, dtype=abi.EDGE_OUT)
    n = C.c_size_t(0)
    h._ck(h.L.alz_window_fetch(h.h, out.ctypes.data_as(C.c_void_p), len(out), C.byref(n)), "alz_window_fetch")
    return out[: n.value]


def _scores(h, n):
    s = np.zeros(max(n, 1), dtype=np.float32)
    m = C.c_size_t(0)
    h._ck(h.L.alz_gnn_score(h.h, s.ctypes.data_as(C.c_void_p), n, C.byref(m)), "alz_gnn_score")
    return s[: m.value]


def test_rollup_equals_the_oracle_over_the_union_of_windows():
    S, per_window, n_windows = 1500, 200_000, 6
    t = ol.Topo(S, seed=2024, mix=abi.MIX_ALL)
    h = capi.Handle(max_endpoints=4 * S, max_pairs=1 << 16)
    h.history_init(8)
    assert h.history_info() == (0, 0)
    assert len(h.rollup(3)) == 0
    h.load_tables(t.pod_ip, t.svc_ip)
    ops, oracles, flushed = [], [], []   # oracles[j]: every event and table change from the start of window j on
    rng = np.random.default_rng(5)
    for w in range(n_windows):
        o = ol.Oracle()
        o.load_tables(t.pod_ip, t.svc_ip)
        for op, ip, id_ in ops:
            o.erase(abi.TABLE_POD, ip) if op == "erase" else o.upsert(abi.TABLE_POD, ip, id_)
        oracles.append(o)
        ev = t.events(w * per_window, per_window)
        cut = per_window // 3
        h.submit(ev[:cut])
        for o in oracles:
            o.process(ev[:cut], 4)
        churn = [("erase", int(t.pod_ip[k]), 0) for k in rng.integers(0, len(t.pod_ip), 20)]
        churn += [("upsert", int(t.pod_ip[k]), int(k)) for k in rng.integers(0, len(t.pod_ip), 20)]
        for op, ip, id_ in churn:
            h.erase(abi.TABLE_POD, ip) if op == "erase" else h.upsert(abi.TABLE_POD, ip, id_)
            for o in oracles:
                o.erase(abi.TABLE_POD, ip) if op == "erase" else o.upsert(abi.TABLE_POD, ip, id_)
        ops += churn
        h.commit()
        h.submit(ev[cut:])
        for o in oracles:
            o.process(ev[cut:], 4)
        flushed.append(h.flush())
        # k = 1 is the last flush
        assert h.rollup(1).tobytes() == flushed[-1].tobytes(), f"window {w}"
    held, newest = h.history_info()
    assert held == n_windows and newest == h.stats()["windows"] == n_windows
    for k in range(1, held + 1):
        got = h.rollup(k)
        _same(got, oracles[n_windows - k].edges(), f"k={k} vs oracle")
        assert got.tobytes() == _numpy_rollup(flushed[n_windows - k:]).tobytes(), f"k={k} vs numpy"
        p, n = h.rollup_device(k)
        assert n == len(got) and h.d2h(p, n, abi.EDGE_OUT).tobytes() == got.tobytes()
    assert h.rollup(100).tobytes() == h.rollup(held).tobytes()
    h.close()


def test_eviction_keeps_the_newest_depth_windows():
    S, per_window = 600, 60_000
    t = ol.Topo(S, seed=77, mix=abi.MIX_ALL)
    h = capi.Handle(max_endpoints=4 * S, max_pairs=1 << 15)
    h.history_init(3)
    h.load_tables(t.pod_ip, t.svc_ip)
    o = ol.Oracle()
    o.load_tables(t.pod_ip, t.svc_ip)
    for w in range(7):
        if w != 5:                       # window 6 of 7 is empty
            ev = t.events(w * per_window, per_window)
            h.submit(ev)
            if w >= 4:
                o.process(ev, 4)         # windows 5..7
        h.flush()
    held, newest = h.history_info()
    assert held == 3 and newest == h.stats()["windows"] == 7
    _same(h.rollup(10), o.edges(), "windows 5-7")
    o7 = ol.Oracle()
    o7.load_tables(t.pod_ip, t.svc_ip)
    o7.process(t.events(6 * per_window, per_window), 4)
    _same(h.rollup(2), o7.edges(), "windows 6-7: the empty window counts")
    h.close()


def test_time_cut_windows_roll_up_by_epoch():
    S, N = 800, 1_200_000
    t = ol.Topo(S, seed=909, mix=abi.MIX_ALL)
    ev = t.events(0, N)
    wt = ev["write_time_ns"].astype(np.uint64)
    fk, fu = np.uint64(int(wt[0]) - 12345), np.uint64(1_700_000_000_123_456_789)
    W = np.uint64((int(wt[-1]) - int(wt[0])) // 4 + 1)
    epoch = (wt + (fu - fk)) // W
    e0, e_last = int(epoch.min()), int(epoch.max())
    h = capi.Handle(max_endpoints=4 * S, max_pairs=1 << 16)
    h.load_tables(t.pod_ip, t.svc_ip)
    h.history_init(8)
    h.window_clock(int(fk), int(fu), int(W))
    for a, b in zip([0, 100_003, 350_000, 900_017], [100_003, 350_000, 900_017, N]):
        h.submit(ev[a:b])
    late = ev[:5000].copy()              # epoch e0 records that arrive while e0 + 1 is open
    for k, e in enumerate(range(e0, e_last + 1)):
        h.flush()
        if k == 0:
            h.submit(late)
    held, newest = h.history_info()
    assert held == e_last - e0 + 1 and newest == h.stats()["windows"]
    offset = e_last - newest             # epoch = ordinal + offset
    for k in range(1, held + 1):
        o = ol.Oracle()
        o.load_tables(t.pod_ip, t.svc_ip)
        o.process(ev[(epoch >= e_last - k + 1) & (epoch <= e_last)], 4)
        if newest - k + 1 + offset <= e0 + 1:
            o.process(late)
        _same(h.rollup(k), o.edges(), f"epochs [{e_last - k + 1}, {e_last}]")
    h.close()


def test_history_changes_nothing_without_being_asked():
    S, per_window = 1000, 150_000
    t = ol.Topo(S, seed=4242, mix=abi.MIX_ALL)
    a = capi.Handle(max_endpoints=4 * S, max_pairs=1 << 16)
    b = capi.Handle(max_endpoints=4 * S, max_pairs=1 << 16)
    b.history_init(4)
    for h in (a, b):
        h.load_tables(t.pod_ip, t.svc_ip)
    for w in range(6):
        ev = t.events(w * per_window, per_window)
        for h in (a, b):
            h.submit(ev)
        fa, fb = a.flush(), b.flush()
        assert fa.tobytes() == fb.tobytes(), f"window {w}"
        sa, sb = a.stats(), b.stats()
        assert {k: v for k, v in sa.items() if k not in TIMING} == {k: v for k, v in sb.items() if k not in TIMING}
        assert _scores(a, len(fa)).tobytes() == _scores(b, len(fb)).tobytes()
    # a rollup leaves the last window, its GNN scores, the open window and the next flush as they were
    last, scores = _fetch(b), _scores(b, len(fb))
    ev = t.events(6 * per_window, per_window)
    for h in (a, b):
        h.submit(ev[: per_window // 2])
    assert len(b.rollup(4)) > 0
    assert _fetch(b).tobytes() == last.tobytes() == fb.tobytes()
    assert _scores(b, len(last)).tobytes() == scores.tobytes()
    for h in (a, b):
        h.submit(ev[per_window // 2:])
    assert a.flush().tobytes() == b.flush().tobytes()
    a.close()
    b.close()


def test_errors_and_capacity():
    S = 400
    t = ol.Topo(S, seed=11, mix=abi.MIX_ALL)
    h = capi.Handle(max_endpoints=4 * S, max_pairs=1 << 16)
    L, n = h.L, C.c_size_t(0)
    h.load_tables(t.pod_ip, t.svc_ip)
    assert L.alz_rollup(h.h, 1, None, 0, C.byref(n)) == abi.E_STATE
    assert L.alz_rollup_device(h.h, 1, None, C.byref(n)) == abi.E_STATE
    held, newest = C.c_uint32(0), C.c_uint64(0)
    assert L.alz_history_info(h.h, C.byref(held), C.byref(newest)) == abi.E_STATE
    assert L.alz_history_init(h.h, 0) == abi.E_INVAL
    stride = (1 << 16) + 1
    assert L.alz_history_init(h.h, (1 << 32) // stride + 1) == abi.E_INVAL      # rows >= 2^32
    # rows just below 2^32 pass the check; 1.27 TB of ring does not fit a device: no history, and a retry works
    assert L.alz_history_init(h.h, ((1 << 32) - 1) // stride) == abi.E_NOMEM
    assert L.alz_history_info(h.h, C.byref(held), C.byref(newest)) == abi.E_STATE
    h.history_init(2)
    assert L.alz_history_init(h.h, 2) == abi.E_STATE
    assert L.alz_rollup(h.h, 0, None, 0, C.byref(n)) == abi.E_INVAL
    assert L.alz_rollup_device(h.h, 0, None, C.byref(n)) == abi.E_INVAL
    for w in range(2):
        h.submit(t.events(w * 50_000, 50_000))
        last = h.flush()
    full = h.rollup(2)
    assert len(full) > len(last) > 0
    rc, got_n, _ = _rc_rollup(h, 2, len(full) - 1)
    assert rc == abi.E_CAPACITY and got_n == len(full)
    rc, got_n, got = _rc_rollup(h, 2, len(full))
    assert rc == 0 and got.tobytes() == full.tobytes()
    # the test entry of the multi-rank merge runs the flush's merge but is no flush: the history stays
    blocks = np.zeros((2, len(last) + 1), dtype=abi.EDGE_OUT)
    half = len(last) // 2
    for r, part in enumerate((last[:half], last[half:])):
        hdr = blocks[r, :1].view(np.uint32)
        hdr[0], hdr[1], hdr[2] = 0xA1A2C0DE, len(part), 0
        blocks[r, 1:1 + len(part)] = part
    before = h.history_info()
    d = h.dev_alloc(blocks.nbytes)
    h.h2d(d, blocks)
    p = C.c_void_p()
    assert L.alz_merge_blocks_device(h.h, C.c_void_p(d), 2, len(last), C.byref(p), C.byref(n)) == 0
    h.dev_free(d)
    assert n.value == len(last)
    assert h.history_info() == before
    assert h.rollup(2).tobytes() == full.tobytes()
    h.close()


def _ngpu():
    import torch
    return torch.cuda.device_count() if torch.cuda.is_available() else 0


@pytest.mark.parametrize("overlap", [False, True])
@pytest.mark.parametrize("world", [2, 4, 8])
def test_multi_rank_rollups_are_local_and_equal_on_every_rank(world, overlap):
    if _ngpu() < world:
        pytest.skip(f"needs {world} GPUs")
    L = capi.load()
    S, per_window, n_windows, P = 2000, 300_000, 3, 10_000
    t = ol.Topo(S, seed=31, mix=abi.MIX_ALL)
    wins = [t.events(w * per_window, per_window) for w in range(n_windows)]
    o = ol.Oracle()
    o.load_tables(t.pod_ip, t.svc_ip)
    for ev in wins:
        o.process(ev, 4)
        for _ in range(world - 1 if overlap else 0):
            o.process(ev[:P])       # the first P events of every window reach every rank
    exp = o.edges()
    us = np.unique(np.concatenate([ev["saddr"] for ev in wins]))
    own_of = dict(zip(us.tolist(), [L.alz_owner_rank(int(s), world) for s in us]))
    owners = [np.array([own_of[int(s)] for s in ev["saddr"]]) for ev in wins]
    idbuf = (C.c_uint8 * abi.COMM_ID_BYTES)()
    assert L.alz_comm_unique_id(idbuf) == 0
    out, errs = [None] * world, []
    # one process drives every GPU: allocations and collectives are fenced apart (tests/test_gpu_multi.py)
    bar = threading.Barrier(world, timeout=120)

    def run(rank):
        try:
            h = capi.Handle(device=rank, max_endpoints=4 * S, max_pairs=1 << 17)
            h._ck(L.alz_comm_init(h.h, world, rank, idbuf), "alz_comm_init")
            h.history_init(4)
            h.load_tables(t.pod_ip, t.svc_ip)
            for ev, owner in zip(wins, owners):
                mine = ev[owner == rank]
                if overlap:
                    mine = np.concatenate([mine, ev[:P][owner[:P] != rank]])
                h.submit(mine)
                h.sync()
                bar.wait()
                h.flush()
                bar.wait()
            before = h.stats()["collective_bytes_last"]
            got = h.rollup(3)
            out[rank] = (got, h.history_info(), before, h.stats()["collective_bytes_last"])
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
        got, info, before, after = out[r]
        assert info == (3, 3)
        assert after == before
        assert got.tobytes() == out[0][0].tobytes(), f"rank {r}"
    _same(out[0][0], exp, "rollup(3) vs the single-rank oracle")
