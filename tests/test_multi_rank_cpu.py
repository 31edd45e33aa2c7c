"""CPU, world_size 2 over gloo: the multi-rank window merge as specified in SURVEY.md §8e /
alaz_b200/csrc/alz_comm.cu — shard events by alz_owner_rank(saddr), reduce each shard
independently, then ONE all-gather of fixed-size blocks (a header row {count, status} + the
rank's rows in ascending packed-key order); every rank places each row at its own index plus
its lower bounds in the other ranks' lists (the lists are disjoint when the caller partitions
by owner) and flags a key seen on two ranks. Flagged lists (overlapping shards: a prefix of the
events reaches every rank) are merged from the gathered rows alone: sort by key, one row per key
with the sums of its rows. The result on every rank must equal the single-rank oracle, bit for
bit. (The shards are reduced by the CPU oracle here; the CUDA merge is covered by
tests/test_gpu_merge.py and tests/test_gpu_multi.py.)"""
import os
import socket
import sys

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
N, P = 200_000, 20_000     # events; with overlapping shards the first P reach every rank


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _merge(lists, klists):
    """The merge after the all-gather: R sorted lists of rows and their keys -> (merged rows, dup)."""
    from alaz_b200 import abi
    merged = np.zeros(sum(len(l) for l in lists), dtype=abi.EDGE_OUT)
    dup = False
    for qi, (l, k) in enumerate(zip(lists, klists)):
        pos = np.arange(len(k))
        for pi, kp in enumerate(klists):
            if pi == qi:
                continue
            lb = np.searchsorted(kp, k, side="left")
            dup |= bool(np.any((lb < len(kp)) & (kp[np.minimum(lb, len(kp) - 1)] == k))) if len(kp) else False
            pos = pos + lb
        merged[pos] = l
    if not dup:
        return merged, False
    # a key on several ranks: sort all live rows by key, then one row per key. Type and id fields come from the
    # run's first row; count, err5xx and lat_sum_ns add modulo 2^64, each histogram cell modulo 2^32.
    rows, keys = np.concatenate(lists), np.concatenate(klists)
    order = np.argsort(keys, kind="stable")
    rows, keys = rows[order], keys[order]
    heads = np.flatnonzero(np.r_[True, keys[1:] != keys[:-1]])
    out = rows[heads]
    for f in ("count", "err5xx", "lat_sum_ns"):
        out[f] = np.add.reduceat(rows[f], heads, dtype=np.uint64)
    out["hist"] = np.add.reduceat(rows["hist"], heads, axis=0, dtype=np.uint32)
    return out, True


def _worker(rank, world, port, q):
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle_lib as ol
    from alaz_b200 import abi, capi
    from helpers import pack_key
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    L = capi.load()
    t = ol.Topo(300, seed=17, mix=abi.MIX_ALL)
    ev = t.events(0, N)
    owner = np.array([L.alz_owner_rank(int(s), world) for s in np.unique(ev["saddr"])])
    own_of = dict(zip(np.unique(ev["saddr"]).tolist(), owner.tolist()))
    mine = np.array([own_of[int(s)] == rank for s in ev["saddr"]])
    res = []
    for overlap in (False, True):
        shard = ev[mine]
        if overlap:
            shard = np.concatenate([shard, ev[:P][~mine[:P]]])
        o = ol.Oracle()
        o.load_tables(t.pod_ip, t.svc_ip)
        o.process(shard)
        local = o.edges()
        keys = np.array([pack_key(e) for e in local], dtype=np.uint64)
        order = np.argsort(keys)
        keys, local = keys[order], local[order]
        # block = header row + cap rows (cap would come from the previous window; here: a fixed generous size)
        cap = 16384
        assert len(local) <= cap
        block = np.zeros(cap + 1, dtype=abi.EDGE_OUT)
        hdr = block[:1].view(np.uint32)
        hdr[0], hdr[1], hdr[2] = 0xA1A2C0DE, len(local), 0
        block[1:1 + len(local)] = local
        # the single collective
        bufs = [torch.zeros(block.nbytes, dtype=torch.uint8) for _ in range(world)]
        dist.all_gather(bufs, torch.from_numpy(block.view(np.uint8).copy()))
        blocks = [b.numpy().view(abi.EDGE_OUT) for b in bufs]
        counts = [int(b[:1].view(np.uint32)[1]) for b in blocks]
        lists = [b[1:1 + n] for b, n in zip(blocks, counts)]
        klists = [np.array([pack_key(e) for e in l], dtype=np.uint64) for l in lists]
        merged, dup = _merge(lists, klists)
        assert dup == overlap
        can = np.array([pack_key(e) for e in merged], dtype=np.uint64)
        res.append((can.tobytes(), merged.tobytes(), len(shard)))
    q.put((rank, res))
    dist.destroy_process_group()


def test_two_rank_merge_equals_single_rank_oracle():
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle_lib as ol
    from alaz_b200 import abi
    from helpers import pack_key
    world, port = 2, _free_port()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    ps = [ctx.Process(target=_worker, args=(r, world, port, q)) for r in range(world)]
    for p in ps:
        p.start()
    res = [q.get(timeout=180) for _ in ps]
    for p in ps:
        p.join(timeout=60)
        assert p.exitcode == 0
    res.sort()
    t = ol.Topo(300, seed=17, mix=abi.MIX_ALL)
    ev = t.events(0, N)
    for s, overlap in enumerate((False, True)):
        r0, r1 = res[0][1][s], res[1][1][s]
        assert r0[0] == r1[0] and r0[1] == r1[1], f"ranks disagree after the merge (overlap={overlap})"
        assert 0 < r0[2] and 0 < r1[2] and r0[2] + r1[2] == N + (P * (world - 1) if overlap else 0)
        o = ol.Oracle()
        o.load_tables(t.pod_ip, t.svc_ip)
        o.process(ev)
        if overlap:
            for _ in range(world - 1):
                o.process(ev[:P])
        exp = o.edges()
        ek = np.array([pack_key(e) for e in exp], dtype=np.uint64)
        order = np.argsort(ek)
        ek, exp = ek[order], exp[order]
        can = np.frombuffer(r0[0], dtype=np.uint64)
        merged = np.frombuffer(r0[1], dtype=abi.EDGE_OUT)
        assert np.array_equal(can, ek)
        assert np.all(can[1:] > can[:-1])                      # canonical order, no key twice
        assert merged.tobytes() == exp.tobytes()
