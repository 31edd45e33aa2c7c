"""Shared test helpers: golden-vector loading and edge-list comparison."""
import json
import os

import numpy as np

from alaz_b200 import abi

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")

_PROTO = {"UNKNOWN": 0, "HTTP": 1, "AMQP": 2, "POSTGRES": 3, "HTTP2": 4, "REDIS": 5,
          "KAFKA": 6, "MYSQL": 7, "MONGO": 8}
_TYPE = {"pod": abi.NODE_POD, "svc": abi.NODE_SVC, "outbound": abi.NODE_OUTBOUND}


def load_branches():
    with open(os.path.join(GOLDEN, "resolve_branches.json")) as f:
        g = json.load(f)
    recs = np.zeros(len(g["events"]), dtype=abi.L7_REC)
    for i, e in enumerate(g["events"]):
        p = e["proto"]
        mf = e["method"]
        if "tls" in e["flags"]:
            mf |= abi.MF_TLS
        if "reject" in e["flags"]:
            mf |= abi.MF_PAYLOAD_REJECT
        recs[i] = (abi.ip(e["saddr"]), abi.ip(e["daddr"]), 40000 + i, 80, e["status"],
                   _PROTO[p] if isinstance(p, str) else p, mf, e["dur"], 1000 + i)
    exp = np.zeros(len(g["expect_edges"]), dtype=abi.EDGE_OUT)
    for i, e in enumerate(g["expect_edges"]):
        def node(n):
            t = _TYPE[n[0]]
            return t, (abi.ip(n[1]) if t == abi.NODE_OUTBOUND else n[1])
        ft, fv = node(e["from"])
        tt, tv = node(e["to"])
        exp[i]["from_type"], exp[i]["from"], exp[i]["to_type"], exp[i]["to"] = ft, fv, tt, tv
        exp[i]["count"], exp[i]["err5xx"], exp[i]["lat_sum_ns"] = e["count"], e["err5xx"], e["lat_sum"]
        for b, c in e["hist"].items():
            exp[i]["hist"][int(b)] = c
    pods = {abi.ip(k): v for k, v in g["pods"].items()}
    svcs = {abi.ip(k): v for k, v in g["services"].items()}
    return pods, svcs, recs, sort_edges(exp), g["expect_stats"]


def sort_edges(e):
    order = np.lexsort((e["to"], e["to_type"], e["from"], e["from_type"]))
    return e[order]


def pack_key(e):
    """alz_device.cuh make_edge_key on the oracle's (from,to) representation."""
    ft, f, tt, t = int(e["from_type"]), int(e["from"]), int(e["to_type"]), int(e["to"])
    if ft == 0:          # pod is From (canonical for pod->pod too)
        rev, pod, ot, ov = 0, f, tt, t
    else:                # reversed row whose From is a service / outbound host
        rev, pod, ot, ov = 1, t, ft, f
    return (rev << 63) | (ot << 61) | (pod << 32) | ov


def edges_equal(a, b):
    """Bit-exact comparison of two alz_edge_out arrays (order-insensitive)."""
    a, b = sort_edges(np.asarray(a)), sort_edges(np.asarray(b))
    if len(a) != len(b):
        return False
    for f in ("from_type", "from", "to_type", "to", "count", "err5xx", "lat_sum_ns", "hist"):
        if not np.array_equal(a[f], b[f]):
            return False
    return True


def explain_diff(a, b, limit=5):
    a, b = sort_edges(np.asarray(a)), sort_edges(np.asarray(b))
    msgs = [f"len {len(a)} vs {len(b)}"]
    ka = {(int(x["from_type"]), int(x["from"]), int(x["to_type"]), int(x["to"])): x for x in a}
    kb = {(int(x["from_type"]), int(x["from"]), int(x["to_type"]), int(x["to"])): x for x in b}
    for k in list(ka.keys() - kb.keys())[:limit]:
        msgs.append(f"only in A: {k} count={int(ka[k]['count'])}")
    for k in list(kb.keys() - ka.keys())[:limit]:
        msgs.append(f"only in B: {k} count={int(kb[k]['count'])}")
    n = 0
    for k in ka.keys() & kb.keys():
        x, y = ka[k], kb[k]
        if x.tobytes() != y.tobytes():
            msgs.append(f"differs {k}: count {int(x['count'])}/{int(y['count'])} err {int(x['err5xx'])}/"
                        f"{int(y['err5xx'])} lat {int(x['lat_sum_ns'])}/{int(y['lat_sum_ns'])}")
            n += 1
            if n >= limit:
                break
    return "; ".join(msgs)


def pyref_edges(agg):
    """oracle/ref_py.Aggregator groups -> alz_edge_out array."""
    out = np.zeros(len(agg.groups), dtype=abi.EDGE_OUT)
    def node(t, uid):
        if t == "pod":
            return abi.NODE_POD, int(uid.split("-")[1])
        if t == "service":
            return abi.NODE_SVC, int(uid.split("-")[1])
        return abi.NODE_OUTBOUND, abi.ip(uid)
    for i, ((ft, fu, tt, tu), g) in enumerate(agg.groups.items()):
        a, b = node(ft, fu), node(tt, tu)
        out[i]["from_type"], out[i]["from"], out[i]["to_type"], out[i]["to"] = a[0], a[1], b[0], b[1]
        out[i]["count"], out[i]["err5xx"] = g["count"], g["err5xx"]
        out[i]["lat_sum_ns"] = g["lat_sum"] & 0xFFFFFFFFFFFFFFFF   # the accumulators are u64: sums are defined modulo 2^64 (docs/SPEC.md)
        out[i]["hist"] = g["hist"]
    return sort_edges(out)
