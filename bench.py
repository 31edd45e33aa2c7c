#!/usr/bin/env python
"""bench.py — l7_req events/sec aggregated into the per-edge service graph.

One "step" = one window of the hot path over one batch of the synthetic stream:
alz_submit_l7_device (ingest kernel) + alz_window_flush_device (join of the distinct
socket pairs, canonical edge list; at N>1 the cross-rank merge with its single collective
on the per-edge accumulators) and, for the configs that name it, the GNN re-score of the
window. Every step ingests DIFFERENT events (window k = the next slice of the global
stream), so the hot-pair list a fold leaves behind is a prediction for the next window,
not a replay of it; the very first window (no history) is timed separately.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config 2|3|4|5]
                  [--dump-outputs DIR]

Configs are BASELINE.json's (index into `configs`):
  2 (default, the one `metric` is quoted on at N=1): 10k services / 100M events per GPU per step
  3: 50k services / 1B events per step + GNN pass each step, 1 GPU
  4: 100k services / 5B events per step over the ranks (1.25B each at 4 GPUs)
  5: 1M services / 10B events = ten 1-second windows of 1B events over the ranks, GNN re-score each window
At N>1 every rank ingests its own shard of the global stream (events owned by
alz_owner_rank(saddr)): weak scaling for config 2 (100M per rank), the named totals split
over the ranks for 4 and 5.

`--impl reference` times the CPU restatement of the reference aggregator (oracle/alz_oracle.c —
the Go binary cannot be built here, SURVEY.md §8c) on the box's host cores, on a bounded
sample of the same workload.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

METRIC = "l7_req events/sec aggregated (per-edge count/5xx/latency histogram)"
UNIT = "events/s"
ALG_BYTES_PER_EVENT = 32      # SURVEY.md §8d: each compact record read once
ALG_BYTES_PER_EDGE = 296      # each live edge row written once per window (alz_edge_out)
SEED = 0xA1A20001

CONFIGS = {
    # services, events per step (whole job), gnn inside the step, default steps/warmup, what BASELINE.json calls it
    2: dict(services=10_000, events=100_000_000, per_rank=True, gnn=False, steps=50, warmup=5,
            name="BASELINE.json configs[1]: 10k services / 100M l7_req events, hash-join + per-edge reduce"),
    3: dict(services=50_000, events=1_000_000_000, per_rank=True, gnn=True, steps=6, warmup=3,
            name="BASELINE.json configs[2]: 50k services / 1B events, 2-layer GraphSAGE d=64 pass over the CSR service graph"),
    4: dict(services=100_000, events=5_000_000_000, per_rank=False, gnn=False, steps=4, warmup=3,
            name="BASELINE.json configs[3]: 100k services / 5B events sharded by src hash, edge-accumulator collective"),
    5: dict(services=1_000_000, events=1_000_000_000, per_rank=False, gnn=True, steps=10, warmup=3,
            name="BASELINE.json configs[4]: 1M services / 10B events as ten 1-second windows of 1B events, GNN re-score each window"),
}


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None)
    ap.add_argument("--warmup", type=int, default=None)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", type=int, default=2, choices=sorted(CONFIGS))
    ap.add_argument("--services", type=int, default=None, help="override the config's service count")
    ap.add_argument("--events", type=int, default=None, help="override: events per GPU per step")
    ap.add_argument("--windows", type=int, default=None, help="distinct windows resident in HBM (rotated)")
    ap.add_argument("--cpu-sample", type=int, default=None, help="events per step timed on the CPU arm")
    ap.add_argument("--cpu-mode", default="faithful", choices=["faithful", "fair"],
                    help="--impl reference: which CPU arm is the line's value (both are reported)")
    ap.add_argument("--eager", action="store_true", help="ALZ_CFG_EAGER_JOIN plan")
    ap.add_argument("--no-smem-cache", action="store_true", help="ingest v1: global reductions only")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-gnn", action="store_true", help="skip the separate GNN-update timing (config 2)")
    ap.add_argument("--no-verify", action="store_true", help="skip the in-run parity check against the oracle")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the last timed step's edges (and GNN scores) to DIR/*.npy, see dump_outputs()")
    return ap.parse_args()


def resolve(args, world):
    c = CONFIGS[args.config]
    S = args.services or c["services"]
    if args.events:
        n_rank = args.events
    elif c["per_rank"]:
        n_rank = c["events"]
    else:
        n_rank = c["events"] // world
    steps = args.steps if args.steps is not None else c["steps"]
    warmup = args.warmup if args.warmup is not None else c["warmup"]
    if steps < 1:
        raise SystemExit("bench.py: --steps must be at least 1")
    return c, S, n_rank, steps, max(3, warmup)


def workload_text(c, S, n_rank, world, n_edges_topo):
    return (f"{c['name']}; as run: {S} services, {n_rank} events per GPU per step x {world} GPU(s) = "
            f"{n_rank * world} events per step, Zipf(1.1) over {n_edges_topo} socket pairs, 32-B compact records, "
            f"a different window of the stream every step")


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def measured_traffic(kernel, config):
    """dram__bytes_read.sum + dram__bytes_write.sum of one launch from a committed ncu --set full capture
    (profiles/traffic.json), or None: never a number that was not measured for this kernel and config."""
    p = os.path.join(ROOT, "profiles", "traffic.json")
    if not os.path.exists(p):
        return None
    try:
        return json.load(open(p)).get(f"{kernel}/config{config}")
    except Exception:
        return None


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.rows, self.p, self.index = [], None, index

    def start(self):
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                       "--format=csv,noheader,nounits", "-lms", "50"],
                                      stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.p = None

    def _read(self):
        for ln in self.p.stdout:
            self.rows.append([time.perf_counter()] + [x.strip() for x in ln.strip().split(",")])

    def mark(self):
        """Samples from here on are 'under load' (the timed regions); earlier ones are kept as a fallback."""
        self.t_mark = time.perf_counter()

    def stop(self):
        if not self.p:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.p.terminate()
        try:
            self.p.wait(timeout=2)
        except Exception:
            self.p.kill()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        t_mark = getattr(self, "t_mark", 0.0)
        loaded = [r for r in self.rows if r[0] >= t_mark]
        rows, scope = (loaded, "timed regions (device-resident steps + e2e steps)") if loaded else \
                      (self.rows, "whole run incl. warm-up (timed regions shorter than the sampling period)")
        sm, mx, reasons = [], None, set()
        for r in rows:
            try:
                sm.append(float(r[1]))
                mx = float(r[2])
                for n, v in zip(names, r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            except Exception:
                pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx,
                "reasons": sorted(reasons), "samples": len(sm), "scope": scope}


# ---------------------------------------------------------------------------------------------------
# CPU arms (the only place bench.py touches oracle/)
# ---------------------------------------------------------------------------------------------------
def cpu_arm(mode, services, n_events, nthreads, steps=1, warmup=0, first=0):
    """Time one CPU arm on events [first, first + n_events) of the workload stream. mode 'faithful' =
    oracle/alz_oracle.c (restatement of the Go data structures), 'fair' = oracle/alz_fastcpu.c."""
    import oracle_lib as ol
    t = ol.Topo(services, seed=SEED)
    ev = t.events(first, n_events)
    times, n_edges = [], 0
    for it in range(warmup + steps):
        if mode == "faithful":
            o = ol.Oracle()
            o.load_tables(t.pod_ip, t.svc_ip)
        else:
            o = ol.FastCpu(4 * services)
            o.load_tables(t.pod_ip, t.svc_ip)
        t0 = time.perf_counter()
        o.process(ev, nthreads)
        n_edges = len(o.edges())
        dt = time.perf_counter() - t0
        if it >= warmup:
            times.append(dt)
        o.close()
    sec = sum(times) / len(times)
    return n_events / sec, n_edges, sec


def cpu_baselines(services, sample, cores):
    out = {}
    for mode in ("faithful", "fair"):
        n = sample if mode == "faithful" else sample * 4
        v, _, sec = cpu_arm(mode, services, n, cores)
        out[mode] = {"value": v, "unit": UNIT, "cores": cores, "kind": "port",
                     "sample": f"first {n} events of the same stream per step, {cores} threads ({sec:.1f} s)"}
    return out


def run_reference(args, rank, world):
    if rank != 0:
        return
    c, S, n_rank, steps, warmup = resolve(args, world)
    cores = os.cpu_count() or 1
    import oracle_lib as ol
    t = ol.Topo(S, seed=SEED)
    n_edges_topo = t.n_edges
    t.close()
    if args.cpu_sample is None:   # bounded: ~400M events in total over all steps, 2M..32M per step
        args.cpu_sample = max(2_000_000, min(32_000_000, 400_000_000 // max(1, steps + warmup)))
    mode = args.cpu_mode
    v, n_edges, sec = cpu_arm(mode, S, args.cpu_sample, cores, steps, warmup)
    other = "fair" if mode == "faithful" else "faithful"
    v2, _, sec2 = cpu_arm(other, S, args.cpu_sample, cores, 1, 0)
    what = {"faithful": "restatement of aggregator/data.go's resolve/emit + group-by keeping the reference's data "
                        "structures (string keys, one heap row per event); the Go binary cannot be built here",
            "fair": "same semantics with integer keys, flat tables, per-thread accumulators, pinned threads"}
    line = {
        "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus,
        "steps": steps, "warmup": warmup, "ms_per_step": sec * 1e3, "higher_is_better": True,
        "scaling": "weak" if c["per_rank"] else "strong", "vs_baseline": None, "dtype": "u64/u32 integer",
        "data": "synthetic",
        "config": {"workload": workload_text(c, S, n_rank, world, n_edges_topo), "config": args.config},
        "cpu_baseline": {"value": v, "unit": UNIT, "cores": cores, "kind": "port", "mode": mode,
                         "what": what[mode],
                         "sample": f"a rate: each step times the first {args.cpu_sample} events of the workload "
                                   f"stream (not the full step), {cores} threads, tables preloaded",
                         "other_mode": {"mode": other, "value": v2, "what": what[other], "seconds": sec2}},
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------------
# GPU arm
# ---------------------------------------------------------------------------------------------------
def main():
    args = parse_args()
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return 0

    import torch
    import torch.distributed as dist
    from alaz_b200 import abi, capi

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the product has no CPU path (use --impl reference "
                         "for the CPU arm)")
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    c, S, N, steps, warmup = resolve(args, world)
    if args.cpu_sample is None:
        args.cpu_sample = 16_000_000
    with_gnn = c["gnn"]
    topo = capi.Topo(S, seed=SEED)
    flags = (abi.CFG_EAGER_JOIN if args.eager else 0) | (abi.CFG_NO_SMEM_CACHE if args.no_smem_cache else 0)
    # capacities: distinct pairs per rank per window (topology pairs it owns + unresolved sources), merged edges
    max_pairs = max(1 << 20, int(1.6 * topo.n_edges / (1 if world == 1 else world * 0.7)) + (1 << 19))
    # live edges: a topology pair shows up as a forward edge and, for the protocols that reverse (AMQP DELIVER, REDIS
    # PUSHED_EVENT), as a reversed one too: 1.9 edges per pair at config 2 (188,749 edges over 100k pairs)
    max_edges = max(1 << 20, int(2.3 * topo.n_edges))

    def new_handle():
        hh = capi.Handle(device=local_rank, max_endpoints=4 * S, max_pairs=max_pairs, max_edges=max_edges,
                         max_batch=1 << 22, flags=flags)
        hh.set_stream(stream.cuda_stream)
        hh.load_tables(topo.pod_ip, topo.svc_ip)
        return hh

    stream = torch.cuda.Stream()          # a real stream: handle 0 would mean "library's own"
    torch.cuda.set_stream(stream)
    h = new_handle()
    if world > 1:
        comm_setup(h, dist, rank, world, torch)

    # ---- inputs resident in HBM before the timed region: R distinct windows, rotated
    free_b, _ = torch.cuda.mem_get_info()
    R_want = args.windows or (4 if args.config == 2 else 10 if args.config == 5 else 2)
    R = args.windows or max(1, min(R_want, int((free_b * 0.55) // (N * 32))))
    if args.dump_outputs and R != R_want:
        # the last timed step reads window (warmup + steps - 1) % R: with fewer windows it would be other events
        raise SystemExit(f"bench.py: --dump-outputs needs all {R_want} input windows resident, only {R} fit "
                         f"in free device memory")
    d_win, first = [], 0
    for k in range(R):
        d = h.dev_alloc(N * 32)
        if world > 1:
            first += fill_owned(h, topo, d, N, world, rank, first)
        else:
            topo.fill_device(h, first, N, d)
            first += N
        d_win.append(d)
    h.sync()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def step(hh, k):
        hh.submit_device(d_win[k % R], N)
        out = hh.flush_device()
        if with_gnn:
            gnn_score_device(hh)
        return out

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    # warm-up also loads every kernel module, so the first-window timing below measures the window, not the loader
    for k in range(warmup):
        _, n_edges = step(h, k)
    barrier()

    # ---- first window of a fresh handle: no fold has run yet, the per-CTA table is filled first-come
    first_window_ms = None
    if world == 1:
        h1 = new_handle()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record(stream)
        step(h1, 0)
        e1.record(stream)
        torch.cuda.synchronize()
        first_window_ms = e0.elapsed_time(e1)
        h1.close()

    # ---- timed region
    launches0 = h.stats().get("kernel_launches", 0)
    barrier()
    sampler.mark()
    ev = [[torch.cuda.Event(enable_timing=True) for _ in range(4)] for _ in range(steps)]
    t_all0, t_all1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    p_scores = None
    t_all0.record(stream)
    for k in range(steps):
        ev[k][0].record(stream)
        h.submit_device(d_win[(warmup + k) % R], N)
        ev[k][1].record(stream)
        p_edges, n_edges = h.flush_device()
        ev[k][2].record(stream)
        if with_gnn:
            p_scores, n_scores = gnn_score_device(h)
        ev[k][3].record(stream)
    t_all1.record(stream)
    barrier()
    if args.dump_outputs and rank == 0:   # before verify_window: the next flush overwrites these device buffers
        if with_gnn and n_scores != n_edges:
            raise SystemExit(f"bench.py: {n_scores} GNN scores for {n_edges} edges")
        dump_outputs(args.dump_outputs, abi, torch, p_edges, n_edges, p_scores)
    total_ms = t_all0.elapsed_time(t_all1)
    ingest_ms = float(np.mean([e[0].elapsed_time(e[1]) for e in ev]))
    flush_ms = float(np.mean([e[1].elapsed_time(e[2]) for e in ev]))
    gnn_step_ms = float(np.mean([e[2].elapsed_time(e[3]) for e in ev])) if with_gnn else None
    st = h.stats()
    launches = st.get("kernel_launches", 0) - launches0

    tt = torch.tensor([total_ms, ingest_ms, flush_ms], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    total_ms, ingest_ms_max, flush_ms_max = (float(x) for x in tt.tolist())
    ms_per_step = total_ms / steps
    value = world * N / (ms_per_step * 1e-3)

    # ---- in-run parity: every rank holds byte-identical edges, and a sample of them matches the oracle
    verify = None
    if not args.no_verify:
        verify = verify_window(h, capi, abi, topo, d_win[(warmup + steps - 1) % R], N, S, world, rank,
                               dist if world > 1 else None, torch)

    # ---- end to end through the C ABI with host buffers (H2D + D2H inside the timed region)
    e2e = None
    if not args.no_e2e:
        e2e = run_e2e(h, capi, abi, d_win, N, steps, world, dist if world > 1 else None, torch)

    clocks = sampler.stop() if rank == 0 else None
    gnn_ms = None
    if not args.no_gnn and not with_gnn:
        gnn_ms = run_gnn(h, lambda: step(h, 0), torch)

    if rank == 0:
        peak, peak_src = peaks()
        kernel = "ingest_eager_kernel" if args.eager else ("ingest_pairs_kernel(v1)" if args.no_smem_cache
                                                           else "ingest_pairs_v8_kernel")
        alg_bytes = N * ALG_BYTES_PER_EVENT
        achieved = alg_bytes / (ingest_ms_max * 1e-3) / 1e9
        step_alg = N * ALG_BYTES_PER_EVENT + int(n_edges) * ALG_BYTES_PER_EDGE
        step_ms_no_gnn = ingest_ms_max + flush_ms_max
        step_achieved = step_alg / (step_ms_no_gnn * 1e-3) / 1e9
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": steps,
            "warmup": warmup, "ms_per_step": ms_per_step, "higher_is_better": True,
            "scaling": "weak" if c["per_rank"] else "strong", "vs_baseline": None, "dtype": "u64/u32 integer",
            "data": "synthetic",
            "config": {
                "workload": workload_text(c, S, N, world, topo.n_edges), "config": args.config,
                "plan": "eager-join" if args.eager else "reduce-per-socket-pair then join distinct pairs",
                "step": "alz_submit_l7_device + alz_window_flush_device" + (" + alz_gnn_score_device" if with_gnn else ""),
                "l2": f"inputs ({N * 32 / 1e9:.2f} GB per step, {R} distinct windows rotated) larger than L2; no explicit flush",
                "parallelism": f"dp{world} by alz_owner_rank(saddr)" if world > 1 else "single GPU",
                "live_edges": int(n_edges),
                "rows_emitted_per_step": int(st["rows_emitted"] // max(1, st["events_in"] // N)),
            },
            "roofline": {"bound": "hbm", "kernel": kernel, "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": achieved / peak, "peak_source": peak_src,
                         "traffic": measured_traffic(kernel, args.config) if world == 1 else None,
                         "kernel_ms": ingest_ms_max, "algorithmic_bytes_per_launch": alg_bytes,
                         "whole_step": {"what": "ingest + flush (fold, sort, gather" + (", cross-rank merge" if world > 1 else "") + ")",
                                        "ms": step_ms_no_gnn, "algorithmic_bytes": step_alg,
                                        "achieved": step_achieved, "frac": step_achieved / peak}},
            "phases_ms": {"ingest": ingest_ms_max, "flush": flush_ms_max, "gnn": gnn_step_ms,
                          "first_window_step": first_window_ms},
            "clocks": clocks,
            "gpu_launches": int(launches),
            "gpu_launches_what": "kernels of this library launched in the timed region (CUB sort/scan passes and memsets not counted)",
            "verify": verify,
            "e2e": e2e,
        }
        if world > 1:
            cs = h.stats()
            line["multi_gpu"] = {"collective_bytes_per_step": cs.get("collective_bytes_last", None),
                                 "flush_local_ms_last": cs.get("flush_local_us_last", 0) / 1000.0,
                                 "merge_ms_last": cs.get("merge_us_last", 0) / 1000.0,
                                 "what": "rank 0, last window: local part of the flush (fold, sort) and cross-rank part "
                                         "(gather rows, one ncclAllGather, merge kernel), device time between events"}
        if gnn_ms is not None:
            line["gnn_update"] = gnn_ms
        if not args.no_cpu:
            cores = os.cpu_count() or 1
            cb = cpu_baselines(S, args.cpu_sample, cores)
            line["cpu_baseline"] = dict(cb["faithful"], mode="faithful",
                                        what="restatement of aggregator/data.go keeping the reference's data "
                                             "structures, not the Go binary",
                                        fair=dict(cb["fair"], what="integer keys, flat tables, per-thread "
                                                                   "accumulators, pinned threads (oracle/alz_fastcpu.c)"))
        print(json.dumps(line), flush=True)
    for d in d_win:
        h.dev_free(d)
    topo.close()
    h.close()
    if world > 1:
        dist.destroy_process_group()
    return 0


class _DevView:
    """Zero-copy view of device memory owned by the library (__cuda_array_interface__), int32 words."""

    def __init__(self, ptr, n_words):
        self.__cuda_array_interface__ = {"shape": (int(n_words),), "typestr": "<i4", "data": (int(ptr), False),
                                         "version": 2}


def dev_view(torch, ptr, n_words):
    return torch.as_tensor(_DevView(ptr, n_words), device="cuda")


def gnn_score_device(h):
    p, n_out = C.c_void_p(), C.c_size_t(0)
    h._ck(h.L.alz_gnn_score_device(h.h, C.byref(p), C.byref(n_out)), "alz_gnn_score_device")
    return p.value, n_out.value


DUMP_MAX_EDGES = 1 << 16          # 71 float64 columns a row: at most 37 MB of edges.npy


def dump_outputs(out_dir, abi, torch, p_edges, n_edges, p_scores):
    """Writes what alz_window_flush_device (and alz_gnn_score_device) returned in the last timed step, so that two
    builds can be compared output for output. One float64 row per edge: from_type, to_type, from, to, count, err5xx,
    lat_sum_ns, hist[0..63], in the library's canonical edge order; above DUMP_MAX_EDGES edges a fixed seeded sample
    of the rows (edge_rows.npy says which). scores.npy: float32 GNN scores of the same rows."""
    os.makedirs(out_dir, exist_ok=True)
    n = int(n_edges)
    rows = np.arange(n)
    if n > DUMP_MAX_EDGES:
        rows = np.sort(np.random.default_rng(SEED).choice(n, DUMP_MAX_EDGES, replace=False))
    idx = torch.from_numpy(rows).to("cuda")
    words = abi.EDGE_OUT.itemsize // 4
    e = np.zeros(0, dtype=abi.EDGE_OUT)
    if n:
        sel = dev_view(torch, p_edges, n * words).view(n, words).index_select(0, idx)
        e = sel.cpu().numpy().view(abi.EDGE_OUT).reshape(-1)
    cols = [e[f].astype(np.float64)[:, None] for f in ("from_type", "to_type", "from", "to", "count", "err5xx",
                                                        "lat_sum_ns")]
    np.save(os.path.join(out_dir, "edges.npy"), np.hstack(cols + [e["hist"].astype(np.float64)]))
    np.save(os.path.join(out_dir, "edge_rows.npy"), rows.astype(np.float64))
    np.save(os.path.join(out_dir, "n_edges.npy"), np.array([n], dtype=np.float64))
    if p_scores is not None:
        s = dev_view(torch, p_scores, n).index_select(0, idx).cpu().numpy().view(np.float32) if n else \
            np.zeros(0, dtype=np.float32)
        np.save(os.path.join(out_dir, "scores.npy"), s)


def verify_window(h, capi, abi, topo, d_ev, N, S, world, rank, dist, torch):
    """Re-run one window and check it: (a) every rank's merged edge array is byte-identical (64-bit sums over
    the device buffer, all-gathered); (b) on every rank, the edges whose source pod falls in a 1/64 sample are
    bit-exact against the CPU oracle run on this rank's events of those sources."""
    import oracle_lib as ol
    from helpers import edges_equal, explain_diff
    h.submit_device(d_ev, N)
    p_edges, n = h.flush_device()
    res = {"edges": int(n)}
    if n == 0:
        return res
    nbytes = n * abi.EDGE_OUT.itemsize
    words = nbytes // 4
    t = dev_view(torch, p_edges, words).to(torch.int64)
    idx = torch.arange(1, words + 1, dtype=torch.int64, device="cuda")
    sig = torch.stack([t.sum(), (t * idx).sum(), torch.tensor(n, dtype=torch.int64, device="cuda")])
    if world > 1:
        sigs = [torch.zeros_like(sig) for _ in range(world)]
        dist.all_gather(sigs, sig)
        same = all(bool((s == sigs[0]).all()) for s in sigs)
        res["ranks_identical"] = same
        if not same:
            raise SystemExit(f"bench.py: rank {rank}: merged edges differ between ranks")
    # (b) sample: sources whose pod id % 64 == 5
    edges = h.d2h(p_edges, n, abi.EDGE_OUT)
    pod_ids = np.arange(len(topo.pod_ip))
    sample_ids = pod_ids[pod_ids % 64 == 5]
    if world > 1:
        # this rank's events are those of the sources it owns: only their edges can be checked against them
        own = np.array([h.L.alz_owner_rank(int(ip), world) for ip in topo.pod_ip[sample_ids]])
        sample_ids = sample_ids[own == rank]
    sample_ips = np.sort(topo.pod_ip[sample_ids])
    rec = dev_view(torch, d_ev, N * 8)
    sad = rec.view(N, 8)[:, 0]
    ips_t = torch.from_numpy(sample_ips.astype(np.int64)).to("cuda")
    sad64 = sad.to(torch.int64) & 0xFFFFFFFF
    pos = torch.searchsorted(ips_t, sad64).clamp_(max=len(sample_ips) - 1)
    mask = ips_t[pos] == sad64
    sel = rec.view(N, 8)[mask].contiguous().cpu().numpy().view(abi.L7_REC).reshape(-1)
    del rec, sad, sad64, pos, mask
    o = ol.Oracle()
    o.load_tables(topo.pod_ip, topo.svc_ip)
    o.process(sel, min(16, os.cpu_count() or 1))
    exp = o.edges()
    o.close()
    in_sample = np.zeros(len(topo.pod_ip) + 1, dtype=bool)
    in_sample[sample_ids] = True

    def pick(e):
        # edges every contribution of which comes from a sampled source: the pod end resolved from saddr is
        # sampled, and for pod<->pod edges (which a reversed row of the other pod can also feed) both ends are
        f_pod, t_pod = e["from_type"] == abi.NODE_POD, e["to_type"] == abi.NODE_POD
        fs = f_pod & in_sample[np.minimum(e["from"], len(in_sample) - 1)] & (e["from"] < len(topo.pod_ip))
        ts = t_pod & in_sample[np.minimum(e["to"], len(in_sample) - 1)] & (e["to"] < len(topo.pod_ip))
        return e[np.where(f_pod & t_pod, fs & ts, fs | ts)]

    got_s, exp_s = pick(edges), pick(exp)
    ok = edges_equal(got_s, exp_s)
    res.update({"sampled_events": int(len(sel)), "sampled_edges": int(len(exp_s)), "oracle_match": bool(ok)})
    flag = torch.tensor([1 if ok else 0], dtype=torch.int64, device="cuda")
    if world > 1:
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    if int(flag.item()) != 1:
        raise SystemExit(f"bench.py: rank {rank}: sampled edges differ from the oracle: " + explain_diff(got_s, exp_s))
    res["oracle_match_all_ranks"] = True
    return res


def run_e2e(h, capi, abi, d_win, N, steps_dev, world, dist, torch):
    """Same metric through alz_submit_l7_packed / alz_window_flush with HOST buffers: every step copies that
    step's records host->device from pinned memory and the window's edge rows device->host."""
    from alaz_b200 import capi as _c
    W = min(2, len(d_win))
    pins, n_ovf = [], 0
    for k in range(W):
        got = h.d2h(d_win[k], N, abi.L7_REC)                 # host copy of the very same stream
        r16, ovf = _c.pack_l7(got)                           # what the Go reader would fill: 16-B packed records
        del got
        pin = capi.PinnedBuffer(N, abi.L7_REC16, handle=h)   # NUMA-local to this GPU
        pin.array[:] = r16
        pov = None
        if len(ovf):
            pov = capi.PinnedBuffer(len(ovf), np.uint64, handle=h)
            pov.array[:] = ovf
        n_ovf = max(n_ovf, len(ovf))
        pins.append((pin, pov, len(ovf)))
        del r16
    out = capi.PinnedBuffer(h.max_edges, abi.EDGE_OUT, handle=h)
    n_out = C.c_size_t(0)
    steps = max(3, min(steps_dev, 6))

    def one(k):
        pin, pov, no = pins[k % W]
        h.submit_packed_ptr(pin.ptr, N, pov.ptr if pov is not None else None, no)
        h._ck(h.L.alz_window_flush(h.h, C.c_void_p(out.ptr), h.max_edges, C.byref(n_out)), "alz_window_flush")

    one(0); one(1)
    if dist is not None:
        dist.barrier()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for k in range(steps):
        one(k)
    torch.cuda.synchronize()
    dt = (time.perf_counter() - t0) / steps
    t = torch.tensor([dt], dtype=torch.float64, device="cuda")
    if dist is not None:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    dt = float(t.item())
    res = {"value": world * N / dt, "unit": UNIT, "h2d_bytes_per_step": N * 16 + n_ovf * 8,
           "d2h_bytes_per_step": int(n_out.value) * abi.EDGE_OUT.itemsize, "ms_per_step": dt * 1e3,
           "steps": steps, "record_bytes": 16,
           "api": "alz_submit_l7_packed (16-B records in pinned host memory next to the GPU) + alz_window_flush "
                  "(edge rows to host); wall clock, max over ranks"}
    for pin, pov, _ in pins:
        pin.free()
        if pov is not None:
            pov.free()
    out.free()
    return res


def run_gnn(h, step, torch):
    """GNN-update ms = CSR build + 2 GraphSAGE layers + edge scoring over the flushed window (device time)."""
    step()
    p, n_out = C.c_void_p(), C.c_size_t(0)
    rc = h.L.alz_gnn_score_device(h.h, C.byref(p), C.byref(n_out))
    if rc != 0:
        return None
    stream = torch.cuda.current_stream()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    reps = 5
    e0.record(stream)
    for _ in range(reps):
        h.L.alz_gnn_score_device(h.h, C.byref(p), C.byref(n_out))
    e1.record(stream)
    torch.cuda.synchronize()
    return {"ms": e0.elapsed_time(e1) / reps, "edges": int(n_out.value), "layers": 2, "d": 64,
            "what": "node set + CSR build + 2x GraphSAGE-mean + edge scores, replicated per rank"}


def comm_setup(h, dist, rank, world, torch):
    from alaz_b200 import abi
    idbuf = (C.c_uint8 * abi.COMM_ID_BYTES)()
    if rank == 0:
        h._ck(h.L.alz_comm_unique_id(idbuf), "alz_comm_unique_id")
    t = torch.tensor(list(bytes(idbuf)), dtype=torch.uint8, device="cuda")
    dist.broadcast(t, 0)
    raw = bytes(t.cpu().tolist())
    idbuf = (C.c_uint8 * abi.COMM_ID_BYTES).from_buffer_copy(raw)
    h._ck(h.L.alz_comm_init(h.h, world, rank, idbuf), "alz_comm_init")


def fill_owned(h, topo, d_ev, N, world, rank, first):
    """Fill d_ev with the next N events of the global stream (from index `first` on) that this rank owns;
    returns how many global events were scanned."""
    if topo.dev is None:
        topo.to_device(h)
    n_written, n_scanned = C.c_uint64(0), C.c_uint64(0)
    h._ck(h.L.alz_synth_dev_fill_owned(h.h, topo.dev, first, world, rank, C.c_void_p(d_ev), N,
                                       C.byref(n_written), C.byref(n_scanned)), "alz_synth_dev_fill_owned")
    assert n_written.value == N
    return n_scanned.value


if __name__ == "__main__":
    sys.exit(main())
