#!/usr/bin/env python
"""Cost of the window history (docs/SPEC.md §12) at the config-2 shape of bench.py: 10k services, max_edges = 2^20,
100M device-synthesised events per 1-window flush, history depth 60.

  python scripts/rollup_bench.py --out DIR [--depth 60] [--reps 10] [--events N] [--services S]

Flushes depth + 5 windows of distinct events through two handles, one with history and one without, alternating
which flushes first, then reports in DIR/rollup_bench.json:
  - rollup time of alz_rollup_device for k in {1, 10, 60}: host clock around the call (it ends in a stream
    synchronisation), median of --reps calls after one warm-up call per k;
  - rows in (the sum of the k windows' rows), rows out, algorithmic bytes (rows in x 296 read + rows out x 296
    written) and the resulting GB/s;
  - the phase split of one rollup per k (key extraction, sort, unique, sum) from a separate torch.profiler run;
  - flush time with history on and off: host clock around alz_window_flush_device + a synchronise, per window;
  - the card's name, power limit and maximum SM clock, read in the same run.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402  (its seed and capacity rules: the same shape as config 2)
from alaz_b200 import abi, capi  # noqa: E402

ROW = 296
KS = (1, 10, 60)
PHASES = (("keys", ("live_row_keys",)), ("sort", ("RadixSort", "Onesweep")),
          ("unique", ("flag_heads", "scatter_heads", "unique_count", "DeviceScan", "Scan")), ("sum", ("sum_runs",)))


def phase_of(name):
    for phase, marks in PHASES:
        if any(m in name for m in marks):
            return phase
    return "other"


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv"],
                       capture_output=True, text=True)
    return q.stdout.strip()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--depth", type=int, default=60)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--events", type=int, default=100_000_000)
    ap.add_argument("--services", type=int, default=10_000)
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("rollup_bench.py: no CUDA device")
    os.makedirs(a.out, exist_ok=True)
    S, N = a.services, a.events
    topo = capi.Topo(S, seed=bench.SEED)
    max_pairs = max(1 << 20, int(1.6 * topo.n_edges) + (1 << 19))   # bench.py's rules at one GPU
    max_edges = max(1 << 20, int(2.3 * topo.n_edges))

    def handle():
        h = capi.Handle(max_endpoints=4 * S, max_pairs=max_pairs, max_edges=max_edges, max_batch=1 << 22)
        h.load_tables(topo.pod_ip, topo.svc_ip)
        return h

    on, off = handle(), handle()
    on.history_init(a.depth)
    d_ev = on.dev_alloc(N * 32)
    n_windows = a.depth + 5
    rows, t_on, t_off = [], [], []
    for w in range(n_windows):
        topo.fill_device(on, w * N, N, d_ev)   # window w = events [w N, (w + 1) N) of the stream
        on.sync()
        order = (on, off) if w % 2 == 0 else (off, on)
        for h in order:
            h.submit_device(d_ev, N)
            h.sync()
            t0 = time.perf_counter()
            _, n = h.flush_device()
            h.sync()
            dt = time.perf_counter() - t0
            (t_on if h is on else t_off).append(dt)
        rows.append(n)
    held, newest = on.history_info()
    assert held == a.depth and newest == n_windows
    warm = 5                                   # the first flushes of a handle also load modules
    res = {
        "card": card(), "torch_device": torch.cuda.get_device_name(0),
        "shape": {"services": S, "events_per_window": N, "max_edges": max_edges, "max_pairs": max_pairs,
                  "depth": a.depth, "windows_flushed": n_windows, "ring_bytes": a.depth * (max_edges + 1) * ROW},
        "flush_ms": {"history_on_median": 1e3 * float(np.median(t_on[warm:])),
                     "history_off_median": 1e3 * float(np.median(t_off[warm:])),
                     "history_on_all": [1e3 * x for x in t_on], "history_off_all": [1e3 * x for x in t_off],
                     "timed": "host clock around alz_window_flush_device + synchronise, two handles alternating, "
                              f"median over windows {warm + 1}..{n_windows}"},
        "edges_per_window": rows, "rollup": {},
    }
    for k in KS:
        if k > held:
            continue
        rows_in = int(sum(rows[-k:]))
        _, n_out = on.rollup_device(k)         # warm-up: grows the scratch to this k
        ts = []
        for _ in range(a.reps):
            t0 = time.perf_counter()
            _, n_out = on.rollup_device(k)
            ts.append(time.perf_counter() - t0)
        med = float(np.median(ts))
        alg = (rows_in + n_out) * ROW
        res["rollup"][str(k)] = {"median_ms": 1e3 * med, "all_ms": [1e3 * x for x in ts], "rows_in": rows_in,
                                 "rows_out": int(n_out), "alg_bytes": alg, "alg_GBps": alg / med / 1e9}
    # phase split: a separate run under the profiler, one rollup per k
    from torch.profiler import ProfilerActivity, profile
    for k in KS:
        if k > held:
            continue
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
            on.rollup_device(k)
            torch.cuda.synchronize()
        split, kernels = {}, {}
        for e in prof.key_averages():
            us = getattr(e, "self_device_time_total", 0) or getattr(e, "self_cuda_time_total", 0)
            if us <= 0 or e.key.startswith(("cuda", "Memcpy", "Memset")):
                continue
            kernels[e.key] = kernels.get(e.key, 0.0) + us / 1e3
            split[phase_of(e.key)] = split.get(phase_of(e.key), 0.0) + us / 1e3
        res["rollup"][str(k)]["phase_ms"] = split
        res["rollup"][str(k)]["kernels_ms"] = kernels
        if k == max(x for x in KS if x <= held):
            prof.export_chrome_trace(os.path.join(a.out, f"rollup_k{k}.pt.trace.json"))
    on.dev_free(d_ev)
    on.close()
    off.close()
    topo.close()
    with open(os.path.join(a.out, "rollup_bench.json"), "w") as f:
        json.dump(res, f, indent=1)
    summary = {k: {x: v[x] for x in ("median_ms", "rows_in", "rows_out", "alg_GBps", "phase_ms")}
               for k, v in res["rollup"].items()}
    print(json.dumps({"card": res["card"], "flush_ms_on": res["flush_ms"]["history_on_median"],
                      "flush_ms_off": res["flush_ms"]["history_off_median"], "rollup": summary}))
    return 0


if __name__ == "__main__":
    sys.exit(main())
