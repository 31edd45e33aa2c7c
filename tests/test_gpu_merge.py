"""GPU, one device: the merge the multi-rank flush runs after its all-gather (alz_merge_blocks_device), on
R blocks built from oracle shards split by alz_owner_rank as tests/test_multi_rank_cpu.py builds them. The
merged rows must equal the single-rank oracle's edges in packed-key order, byte for byte, whether the
shards are disjoint or overlap (a prefix of the events reaches every rank); a block's failure status and a
block that overflows come back as the return code."""
import ctypes as C

import numpy as np
import pytest

import oracle_lib as ol
from alaz_b200 import abi, capi
from helpers import pack_key

pytestmark = pytest.mark.gpu

S, N, P = 300, 200_000, 20_000
BLOCK_ROWS = 16384
HDR_MAGIC = 0xA1A2C0DE


def _by_key(rows):
    keys = np.array([pack_key(e) for e in rows], dtype=np.uint64)
    order = np.argsort(keys)
    return rows[order], keys[order]


def _oracle(t, ev, repeat=None, times=0):
    o = ol.Oracle()
    o.load_tables(t.pod_ip, t.svc_ip)
    o.process(ev)
    for _ in range(times):
        o.process(repeat)
    return _by_key(o.edges())


def _blocks(t, ev, world, overlap):
    L = capi.load()
    us = np.unique(ev["saddr"])
    own_of = dict(zip(us.tolist(), [L.alz_owner_rank(int(s), world) for s in us]))
    owner = np.array([own_of[int(s)] for s in ev["saddr"]])
    blocks = np.zeros((world, BLOCK_ROWS + 1), dtype=abi.EDGE_OUT)
    for r in range(world):
        shard = ev[owner == r]
        if overlap:
            shard = np.concatenate([shard, ev[:P][owner[:P] != r]])
        rows, _ = _oracle(t, shard)
        assert len(rows) <= BLOCK_ROWS
        hdr = blocks[r, :1].view(np.uint32)
        hdr[0], hdr[1], hdr[2] = HDR_MAGIC, len(rows), 0
        blocks[r, 1:1 + len(rows)] = rows
    return blocks


def _merge(h, blocks):
    d = h.dev_alloc(blocks.nbytes)
    try:
        h.h2d(d, blocks)
        p, n = C.c_void_p(), C.c_size_t(0)
        rc = h.L.alz_merge_blocks_device(h.h, C.c_void_p(d), blocks.shape[0], BLOCK_ROWS, C.byref(p), C.byref(n))
        rows = h.d2h(p.value, n.value, abi.EDGE_OUT) if rc == 0 and n.value else np.zeros(0, dtype=abi.EDGE_OUT)
    finally:
        h.dev_free(d)
    return rc, rows


@pytest.fixture(scope="module")
def setup():
    t = ol.Topo(S, seed=17, mix=abi.MIX_ALL)
    h = capi.Handle(device=0, max_endpoints=4 * S, max_pairs=1 << 15, max_edges=1 << 17)
    yield t, t.events(0, N), h
    h.close()


@pytest.mark.parametrize("overlap", [False, True])
@pytest.mark.parametrize("world", [2, 3, 8])
def test_blocks_merge_to_the_single_rank_oracle(setup, world, overlap):
    t, ev, h = setup
    blocks = _blocks(t, ev, world, overlap)
    exp, ek = _oracle(t, ev, ev[:P], world - 1 if overlap else 0)
    rc, got = _merge(h, blocks)
    assert rc == 0
    keys = np.array([pack_key(e) for e in got], dtype=np.uint64)
    assert np.all(keys[1:] > keys[:-1])                    # ascending, no key twice
    assert np.array_equal(keys, ek)
    assert got.tobytes() == exp.tobytes()


def test_a_failed_block_status_is_returned(setup):
    t, ev, h = setup
    blocks = _blocks(t, ev, 3, False)
    blocks[1, :1].view(np.int32)[2] = abi.E_CUDA
    rc, _ = _merge(h, blocks)
    assert rc == abi.E_CUDA


def test_a_block_count_above_block_rows_is_a_capacity_error(setup):
    t, ev, h = setup
    blocks = _blocks(t, ev, 3, False)
    blocks[2, :1].view(np.uint32)[1] = BLOCK_ROWS + 1
    rc, _ = _merge(h, blocks)
    assert rc == abi.E_CAPACITY
