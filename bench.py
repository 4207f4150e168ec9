#!/usr/bin/env python
"""Benchmark of the DistEGNN hot path on B200 (contract: see the task statement / DESIGN.md §Measurement).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload synth1m] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

One "step" = one complete FastEGNN forward (4 layers, all virtual-node all-reduces) over the WHOLE graph
(all partitions concurrently, one per GPU), inputs resident in HBM, CSR preprocessing cached.
metric = graph-steps/s (BASELINE.json), `edges_per_sec` = Σ_p E_p × graph-steps/s.

  value     device-timed (CUDA events, max over ranks), inputs resident, L2 flushed between steps
  e2e       same metric through the public API with HOST (pinned) inputs: H2D of every input, CSR build,
            forward, D2H of both outputs inside the timed region
  roofline  the edge-aggregation kernel (dominant): algorithmic bytes E·284+N·536 per launch ÷ its
            CUDA-event duration, against the measured HBM copy peak (MEASURED_PEAKS.json)
  roofline_virtual  the real<->virtual kernel (compute-bound): logical FLOP per launch ÷ its duration against the
            measured sustained bf16 tensor peak
  cpu_baseline  the reference's own CPU PyTorch path (oracle/_ref = the unmodified models/FastEGNN.py installed by
            oracle/build_ref.py; the oracle port if that copy is absent) on this box's host cores, on a bounded
            sample of the same workload (rank 0, N=1 only)
  dist_parity   (N>1) before the timed region every rank runs small instances of BASELINE configs 3/4/5 through the same
            CUDA path + exchange and rank 0 checks them against the partitioned float64 oracle; a miss fails the run

--impl reference times ONLY the CPU path, at FULL size: the whole 1M-node graph (N>1: the block-diagonal union of the
N partitions, identical arithmetic to N-rank DistEGNN — BASELINE.md §3), 1 warm-up + as many timed forwards as fit
--ref-budget-s; `steps` reports how many were timed.

--dump-outputs DIR writes what the last timed step returned, node_loc.npy [N, 3] and virtual_loc.npy [B, 3, C]; inputs
and weights are generated from fixed seeds, so two builds run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

from distegnn_b200 import synth  # noqa: E402

METRIC = "graph_steps_per_sec"
UNIT = "graph-steps/s"
N_LAYERS = 4


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="synth1m", choices=list(synth.WORKLOADS))
    ap.add_argument("--split-mode", default="random", choices=["random", "kmeans"])
    ap.add_argument("--nodes", type=int, default=None, help="override node count (debug)")
    ap.add_argument("--cpu-sample-nodes", type=int, default=100_000)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-train", action="store_true", help="skip the secondary forward+backward measurement")
    ap.add_argument("--cuda-graph", default="auto", choices=["auto", "on", "off"],
                    help="replay the forward (collectives included) as a CUDA graph in the timed region; auto = on for "
                         "N>1 (latency-bound regime), off for N=1")
    ap.add_argument("--ref-budget-s", type=float, default=420.0,
                    help="--impl reference: wall-clock budget for full-size CPU forwards (1 warm-up + timed steps)")
    ap.add_argument("--no-dist-parity", action="store_true", help="skip the multi-GPU parity cases before the timed region")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps write the outputs of the last one as DIR/<name>.npy (float32; with N>1 "
                         "ranks one file per rank), for comparing two builds on the same seeded inputs")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    return a


DUMP_MAX_BYTES = 64 * 10 ** 6


def dump_outputs(d: str, outputs, rank: int, world: int) -> None:
    """Write each output as DIR/<name>.npy in float32 (DIR/<name>.rank<r>.npy with N>1 ranks).  If the outputs exceed
    DUMP_MAX_BYTES in all, each keeps a seeded sample of its rows (in order), the same from run to run."""
    os.makedirs(d, exist_ok=True)
    total = world * sum(t.numel() * 4 for t in outputs.values())
    for name, t in outputs.items():
        t = t.detach().float().cpu()
        if total > DUMP_MAX_BYTES:
            keep = max(1, t.shape[0] * DUMP_MAX_BYTES // total)
            rows = torch.randperm(t.shape[0], generator=torch.Generator().manual_seed(rank))[:keep].sort().values
            t = t[rows]
        np.save(os.path.join(d, name + ("" if world == 1 else f".rank{rank}") + ".npy"), t.numpy())


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def tensor_peak():
    """Sustained bf16/fp16 tensor peak in TFLOP/s (the kernel is timed inside a long step)."""
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["bf16_tflops_sustained"]), "measured (MEASURED_PEAKS.json bf16_tflops_sustained)"
        except Exception:
            pass
    return 1400.0, "fallback (B200_PROFILING.md, sustained)"


def virtual_kernel_flops(n_nodes: int, channels: int) -> int:
    """Logical FLOP of one real<->virtual launch: per (node, channel) row three 64x64 layers (W2v and the two
    coordinate heads' hidden layers, 2*64*64 each) and the two 64-wide head projections."""
    return n_nodes * channels * (3 * 2 * 64 * 64 + 2 * 2 * 64)


def edge_kernel_bytes(n_nodes: int, n_edges: int) -> int:
    """Algorithmic bytes of one edge-stage launch (SURVEY §8d): per edge row+col ids 8 B, edge_attr 8 B,
    neighbour feature row 256 B, neighbour coordinate 12 B; per node own feature row + coordinate read
    268 B and the aggregated [64]+[3] written 268 B."""
    return n_edges * 284 + n_nodes * 536


class ClockSampler(threading.Thread):
    """Samples SM clock + throttle reasons of this rank's GPU during the timed region (NVML)."""

    def __init__(self, index: int):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.max_mhz = index, [], set(), None
        self._halt = threading.Event()
        self.ok = False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception as e:  # pragma: no cover
            self.err = repr(e)

    def run(self):
        if not self.ok:
            return
        nv = self.nv
        names = {getattr(nv, k): k for k in dir(nv) if k.startswith("nvmlClocksEventReason")
                 or k.startswith("nvmlClocksThrottleReason")}
        while not self._halt.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                mask = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                for bit, name in names.items():
                    if isinstance(bit, int) and bit and mask & bit:
                        self.reasons.add(name.replace("nvmlClocksEventReason", "").replace(
                            "nvmlClocksThrottleReason", ""))
            except Exception:
                pass
            time.sleep(0.1)

    def stop(self):
        self._halt.set()
        self.join(timeout=2)
        s = sorted(self.samples)
        reasons = sorted(r for r in self.reasons if r not in ("None", "GpuIdle", "ApplicationsClocksSetting"))
        return {"sm_mhz": (s[len(s) // 2] if s else None), "sm_max_mhz": self.max_mhz,
                "reasons": reasons, "samples": len(s)}


def model_dims(w: synth.Workload):
    return dict(node_feat_nf=w.node_feat_nf, node_attr_nf=w.node_attr_nf, edge_attr_nf=w.edge_attr_nf,
                virtual_channels=w.virtual_channels, n_layers=N_LAYERS, normalize=w.normalize)


def make_state_dict(w: synth.Workload):
    """Random-init weights of the architecture (same distributions as the reference's init)."""
    from distegnn_b200 import FastEGNN
    torch.manual_seed(0)
    m = FastEGNN(hidden_nf=64, world_size=1, **model_dims(w))
    return m.state_dict()


# ------------------------------------------------------------------------------------------------
# CPU arm: the reference's own PyTorch path on host cores (oracle/_ref; the oracle port if that copy is absent)
# ------------------------------------------------------------------------------------------------
_THREADS = None


def cpu_forward_fn(w: synth.Workload, sd):
    """(fn(inp) -> (out, X), kind): kind "reference" = the unmodified models/FastEGNN.py from oracle/_ref."""
    from oracle import ref_loader
    if ref_loader.available():
        def fn(inp):
            return ref_loader.reference_forward(sd, normalize=w.normalize, n_layers=N_LAYERS, **inp)
        return fn, "reference"
    from oracle import fastegnn_oracle as orc

    def fn(inp):
        with torch.no_grad():
            return orc.forward(sd, **inp, normalize=w.normalize)
    return fn, "port"


def pick_threads(w: synth.Workload, sd) -> int:
    """The reference's CPU path is plain PyTorch; its speed depends heavily on the intra-op thread count (on a
    128-thread host all threads is far from the best).  Probe a few counts on a small graph and keep the fastest —
    this makes the CPU baseline as strong as the host allows."""
    global _THREADS
    if _THREADS is not None:
        return _THREADS
    fn, _ = cpu_forward_fn(w, sd)
    ncpu = os.cpu_count() or 1
    cands = sorted({c for c in (4, 8, 16, 32, 64, ncpu) if c <= ncpu})
    inp = synth.make_partitions(w, n_nodes=min(20000, w.n_nodes), seed=1)[0]
    best, best_t = cands[0], float("inf")
    for c in cands:
        torch.set_num_threads(c)
        fn(inp)
        t0 = time.perf_counter()
        fn(inp)
        dt = time.perf_counter() - t0
        if dt < best_t:
            best, best_t = c, dt
    _THREADS = best
    torch.set_num_threads(best)
    return best


def cpu_reference_time(w: synth.Workload, sd, sample_nodes: int, repeats: int):
    """Best-of-`repeats` forward time of the CPU path on a `sample_nodes` sub-cloud of the same density."""
    fn, kind = cpu_forward_fn(w, sd)
    cores = pick_threads(w, sd)
    torch.set_num_threads(cores)
    n = min(sample_nodes, w.n_nodes)
    inp = synth.make_partitions(w, n_nodes=n, seed=0)[0]
    e = int(inp["edge_index"].shape[1])
    best = float("inf")
    fn(inp)                                                     # warm-up
    for _ in range(repeats):
        t0 = time.perf_counter()
        fn(inp)
        best = min(best, time.perf_counter() - t0)
    return best, n, e, cores, kind


def cpu_model_name():
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name"):
                return line.split(":", 1)[1].strip()
    except Exception:
        pass
    return "unknown"


def union_graph(w: synth.Workload, world: int, split_mode: str, n_nodes: int):
    """The graph the CPU arm evaluates: the whole graph for one partition, else the block-diagonal union of the `world`
    partitions (no cross edges, one graph id, the global loc_mean) — identical arithmetic to `world`-rank DistEGNN
    (SURVEY §8c(i), BASELINE.md §3).  Returns (forward kwargs, Σ_p E_p, nodes)."""
    parts = synth.make_partitions(w, world_size=world, split_mode=split_mode, seed=0, n_nodes=n_nodes)
    if world == 1:
        inp = parts[0]
    else:
        from oracle import fastegnn_oracle as orc
        inp = dict(orc.block_diagonal(parts)["merged"], loc_mean=parts[0]["loc_mean"])
    return inp, int(inp["edge_index"].shape[1]), int(inp["node_loc"].shape[0])


def run_reference(args, w, rank, world):
    if rank != 0:
        return
    sd = {k: v.clone() for k, v in make_state_dict(w).items()}
    full_nodes = args.nodes or w.n_nodes
    fn, kind = cpu_forward_fn(w, sd)
    t_begin = time.perf_counter()
    cores = pick_threads(w, sd)
    inp, e_total, n_total = union_graph(w, world, args.split_mode, full_nodes)
    t_setup = time.perf_counter() - t_begin
    # 1 warm-up + timed FULL-SIZE forwards until the budget is spent (at least one, at most --steps)
    t0 = time.perf_counter()
    fn(inp)
    t_warm = time.perf_counter() - t0
    times = []
    while len(times) < args.steps:
        if times and (time.perf_counter() - t0) + max(times) > args.ref_budget_s:
            break
        t1 = time.perf_counter()
        out, X = fn(inp)
        times.append(time.perf_counter() - t1)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"node_loc": out, "virtual_loc": X}, rank, 1)
    t_step = sum(times) / len(times)
    value = 1.0 / t_step
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": len(times), "steps_requested": args.steps, "warmup": 1, "warmup_requested": args.warmup,
        "ms_per_step": t_step * 1e3, "best_ms_per_step": min(times) * 1e3, "step_seconds": [round(t, 3) for t in times],
        "warmup_seconds": round(t_warm, 3), "setup_seconds": round(t_setup, 2), "budget_s": args.ref_budget_s,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic", "edges_per_sec": e_total * value,
        "config": {"workload": f"{w.name}: {full_nodes} nodes radius graph r={w.radius} (expected degree "
                               f"{w.degree}), C={w.virtual_channels}, F={w.node_feat_nf}, Na={w.node_attr_nf}, "
                               f"{N_LAYERS} layers, hidden 64, normalize={w.normalize}",
                   "partitions": world, "split_mode": args.split_mode if world > 1 else "none",
                   "nodes_total": n_total, "edges_total_sum_p": e_total,
                   "graph": "whole graph" if world == 1 else f"block-diagonal union of the {world} partitions "
                            "(identical arithmetic to DistEGNN on that many ranks)"},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": kind, "cpu": cpu_model_name(),
                         "host_threads": os.cpu_count(),
                         "sample": f"FULL-SIZE forward ({n_total} nodes / {e_total} edges) of "
                                   + ("the unmodified reference models/FastEGNN.py (oracle/_ref, PyG global_mean_pool stub)"
                                      if kind == "reference" else "the oracle port of the reference's op sequence")
                                   + f", torch CPU fp32 no_grad, {cores} threads (fastest of a thread-count probe on this "
                                     f"{os.cpu_count()}-thread host), 1 warm-up + {len(times)} timed forward(s) within a "
                                     f"{args.ref_budget_s:.0f} s budget (mean reported)"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------
def run_ours(args, w, rank, world, local_rank):
    import torch.distributed as dist
    from distegnn_b200 import FastEGNN
    from distegnn_b200.backend import cuda_backend
    assert torch.cuda.is_available(), "bench.py --impl ours needs a CUDA device (no CPU fallback)"
    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    full_nodes = args.nodes or w.n_nodes
    t0 = time.perf_counter()
    host = synth.make_partitions(w, world_size=world, split_mode=args.split_mode, seed=0,
                                 n_nodes=full_nodes, only_rank=rank)[rank]
    t_gen = time.perf_counter() - t0
    pinned = {k: (v.pin_memory() if v is not None else None) for k, v in host.items()}
    N, E = int(host["node_loc"].shape[0]), int(host["edge_index"].shape[1])

    sd = make_state_dict(w)
    model = FastEGNN(hidden_nf=64, world_size=world, **model_dims(w))
    model.load_state_dict(sd)
    model = model.to(dev).eval()
    be = cuda_backend()
    inp = {k: (v.to(dev) if v is not None else None) for k, v in host.items()}
    flush_buf = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x: float) -> float:
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def sum_over_ranks(x: float) -> float:
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return float(t.item())

    # ---- multi-GPU parity BEFORE anything is timed (VERDICT r01 #1): small instances of BASELINE configs 3, 4 and 5 through
    # the same kernels + exchange (+ CUDA graph) as the timed path, checked on rank 0 against the partitioned float64 oracle
    dist_parity = None
    if world > 1 and not args.no_dist_parity:
        from oracle import dist_check
        cases = [dist_check.check_case("fluid113k", 30_000, "random", dev, cuda_graph=True),        # config 3 (small)
                 dist_check.check_case("fluid113k", 30_000, "kmeans", dev, cuda_graph=False),       # config 4 (small)
                 dist_check.check_case("synth1m", 40_000, "random", dev, cuda_graph=True),          # config 5 (small)
                 dist_check.check_case("synth1m", 8_000, "random", dev, grads=True)]                # training path
        dist_parity = {
            "pass": all(c["pass"] for c in cases),
            "abs": max(c.get("abs", 0.0) for c in cases), "rel_disp": max(c.get("rel_disp", 0.0) for c in cases),
            "virtual": max(c.get("virtual", 0.0) for c in cases),
            "bit_identical_across_ranks": all(c.get("bit_identical_across_ranks", True) for c in cases),
            "grads_worst": max(c.get("grads_worst", 0.0) for c in cases), "cases": cases,
            "oracle": "oracle.fastegnn_oracle.forward_partitions in float64 on the same partitions (pinned to the "
                      "reference's own world_size=2 run by tests/test_oracle_golden.py)"}
        if rank == 0:
            print("[bench] dist_parity " + json.dumps(dist_parity), file=sys.stderr, flush=True)
        if not dist_parity["pass"]:
            if rank == 0:
                print(json.dumps({"metric": METRIC, "value": None, "unit": UNIT, "n_gpus": world,
                                  "error": "multi-GPU parity check failed", "dist_parity": dist_parity}), flush=True)
            dist.barrier()
            dist.destroy_process_group()
            sys.exit(3)

    with torch.no_grad():
        # ---- warm-up (also builds + caches the CSR) ----
        t0 = time.perf_counter()
        model(**inp)
        torch.cuda.synchronize()
        t_first = time.perf_counter() - t0
        for _ in range(max(args.warmup - 1, 0)):
            model(**inp)
        # ---- timed: K steps, per-step CUDA events, L2 flushed between steps ----
        use_graph = args.cuda_graph == "on" or (args.cuda_graph == "auto" and world > 1)
        if use_graph and world > 1 and not model._comm:
            use_graph = False                             # torch.distributed fallback of the sync cannot be captured
        timing = []
        if use_graph:
            # per-kernel durations (roofline) come from 3 eager steps; the timed region replays the captured graph
            model._timing = timing
            for _ in range(3):
                flush_buf.zero_()
                model(**inp)
            model._timing = None
            model.cuda_graph = True
            model(**inp)                                  # capture
            model(**inp)                                  # first replay
        sampler = ClockSampler(local_rank)
        if not use_graph:
            model._timing = timing
        evs = []
        barrier()
        sampler.start()
        launches0 = be.launches
        wall0 = time.perf_counter()
        for _ in range(args.steps):
            flush_buf.zero_()
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record()
            out, X = model(**inp)
            e.record()
            evs.append((s, e))
        barrier()
        wall = time.perf_counter() - wall0
        launches = be.launches - launches0
        clocks = sampler.stop()
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, {"node_loc": out, "virtual_loc": X}, rank, world)
        t_dev = sum(s.elapsed_time(e) for s, e in evs) * 1e-3
        model._timing = None
        model.cuda_graph = False                          # e2e below uses fresh device tensors every step
        t_edge = sum(t[1].elapsed_time(t[2]) for t in timing) * 1e-3 / max(len(timing), 1)
        t_virt = sum(t[2].elapsed_time(t[3]) for t in timing) * 1e-3 / max(len(timing), 1)
        t_node = sum(t[3].elapsed_time(t[4]) for t in timing) * 1e-3 / max(len(timing), 1)
        t_upd = sum(t[4].elapsed_time(t[5]) for t in timing) * 1e-3 / max(len(timing), 1)

        # ---- e2e: host (pinned) inputs -> H2D -> CSR build -> forward -> D2H, every step ----
        e2e = None
        if not args.no_e2e:
            h2d = sum(v.numel() * v.element_size() for v in pinned.values() if v is not None)
            out_host = torch.empty(N, 3, dtype=torch.float32).pin_memory()
            X_host = torch.empty(int(host["loc_mean"].shape[0]), 3, w.virtual_channels).pin_memory()
            d2h = out_host.numel() * 4 + X_host.numel() * 4

            def e2e_step():
                d = {k: (v.to(dev, non_blocking=True) if v is not None else None) for k, v in pinned.items()}
                o, xv = model(**d)
                out_host.copy_(o, non_blocking=True)
                X_host.copy_(xv, non_blocking=True)

            e2e_step()
            barrier()
            n_e2e = max(3, min(args.steps, 5))
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            w0 = time.perf_counter()
            s.record()
            for _ in range(n_e2e):
                e2e_step()
            e.record()
            barrier()
            t_e2e_wall = (time.perf_counter() - w0) / n_e2e
            t_e2e = max(s.elapsed_time(e) * 1e-3 / n_e2e, 0.0)
            t_e2e = max_over_ranks(max(t_e2e, 0.0))
            # same bytes every step, but the H2D of step i+1 is issued on a copy stream while step i computes (what a
            # prefetching loader with pinned memory does); reported NEXT TO the serialised number, never instead of it
            copy_stream = torch.cuda.Stream(device=dev)

            def prefetch():
                with torch.cuda.stream(copy_stream):
                    d = {k: (v.to(dev, non_blocking=True) if v is not None else None) for k, v in pinned.items()}
                    ev = torch.cuda.Event()
                    ev.record(copy_stream)
                return d, ev

            def consume(d, ev):
                cur = torch.cuda.current_stream(dev)
                cur.wait_event(ev)
                for v in d.values():
                    if v is not None:
                        v.record_stream(cur)
                o, xv = model(**d)
                out_host.copy_(o, non_blocking=True)
                X_host.copy_(xv, non_blocking=True)

            nxt = prefetch()
            consume(*nxt)
            barrier()
            nxt = prefetch()
            s2, e2 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s2.record()
            for i in range(n_e2e):
                cur_in = nxt
                if i + 1 < n_e2e:
                    nxt = prefetch()
                consume(*cur_in)
            e2.record()
            barrier()
            t_pipe = max_over_ranks(s2.elapsed_time(e2) * 1e-3 / n_e2e)
            # graph built ON THE DEVICE from the positions (SURVEY §8 f-2): only node tensors cross PCIe; every step ONE C-ABI call
            # turns the positions into int32 CSR + edge lengths (distegnn_b200.partition.radius_graph_csr in capacity mode: no
            # host read of the edge count, no COO->CSR sort) — what a rollout does; the reference builds the graph on the host
            # with PyG radius_graph before the step
            from distegnn_b200.partition import radius_graph_csr
            node_keys = [k for k in pinned if k not in ("edge_index", "edge_attr")]
            h2d_nodes = sum(pinned[k].numel() * pinned[k].element_size() for k in node_keys if pinned[k] is not None)
            cap = int(E * 1.1) + 1024

            def from_positions_step():
                d = {k: (pinned[k].to(dev, non_blocking=True) if pinned[k] is not None else None) for k in node_keys}
                g, ea = radius_graph_csr(d["node_loc"], w.radius, edge_attr_nf=w.edge_attr_nf, capacity=cap)
                o, xv = model(edge_index=g, edge_attr=ea, **d)
                out_host.copy_(o, non_blocking=True)
                X_host.copy_(xv, non_blocking=True)
                return g

            g_last = from_positions_step()
            barrier()
            s3, e3 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s3.record()
            for _ in range(n_e2e):
                g_last = from_positions_step()
            e3.record()
            barrier()
            t_pos = max_over_ranks(s3.elapsed_time(e3) * 1e-3 / n_e2e)
            pos_overflow = bool(g_last.overflowed())
            # pre-sorted CSR shard (SURVEY §8 f-4): int32 col + rowptr + CSR-ordered edge_attr from pinned memory, no sort.
            # Local failures must not desynchronise the ranks: the collectives below run unconditionally.
            import tempfile
            t_shard_local, shard_bytes = float("nan"), 0
            try:
                from distegnn_b200.shards import read_shard, shard_from_forward_inputs, write_shard
                with tempfile.TemporaryDirectory() as td:
                    sp = os.path.join(td, f"rank{rank}.shard")
                    write_shard(sp, shard_from_forward_inputs(host))
                    shard = read_shard(sp).pinned()
                shard_bytes = shard.nbytes()

                def from_shard_step():
                    o, xv = model(**shard.to(dev))
                    out_host.copy_(o, non_blocking=True)
                    X_host.copy_(xv, non_blocking=True)

                from_shard_step()
                torch.cuda.synchronize()
                s4, e4 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                s4.record()
                for _ in range(n_e2e):
                    from_shard_step()
                e4.record()
                torch.cuda.synchronize()
                t_shard_local = s4.elapsed_time(e4) * 1e-3 / n_e2e
            except Exception as ex:                       # noqa: BLE001 — reported in the JSON line, never fatal for the bench
                print(f"[bench] from_shard leg failed on rank {rank}: {ex!r}", file=sys.stderr, flush=True)
            barrier()
            t_shard = max_over_ranks(t_shard_local if t_shard_local == t_shard_local else 1e30)
            shard_bytes_total = int(sum_over_ranks(shard_bytes))
            e2e = {"value": 1.0 / t_e2e, "unit": UNIT, "h2d_bytes_per_step": int(sum_over_ranks(h2d)),
                   "from_shard": None if t_shard >= 1e29 else {
                                  "value": 1.0 / t_shard, "ms_per_step": t_shard * 1e3,
                                  "h2d_bytes_per_step": shard_bytes_total,
                                  "note": "inputs from the binary shard format (distegnn_b200/shards.py): graph already CSR "
                                          "by destination with int32 ids, edge_attr in CSR order; H2D, forward, D2H — no sort"},
                   "from_positions": {"value": 1.0 / t_pos, "ms_per_step": t_pos * 1e3,
                                      "h2d_bytes_per_step": int(sum_over_ranks(h2d_nodes)),
                                      "edge_capacity_overflow": pos_overflow,
                                      "note": "node tensors H2D, graph built on the device straight into int32 CSR + edge "
                                              "lengths (one C-ABI call, no host sync, no sort), forward, D2H"},
                   "pipelined": {"value": 1.0 / t_pipe, "ms_per_step": t_pipe * 1e3,
                                 "note": "same per-step copies, H2D of step i+1 overlapped with the forward of step i "
                                         "on a copy stream (the first H2D of the timed region is not hidden)"},
                   "d2h_bytes_per_step": int(sum_over_ranks(d2h)), "ms_per_step": t_e2e * 1e3,
                   "wall_ms_per_step": max_over_ranks(t_e2e_wall) * 1e3,
                   "includes": "H2D of all inputs from pinned host memory, CSR build, forward, D2H of outputs"}

    # ---- secondary: train step = forward + backward through the fused kernels (SURVEY §8d, row f-1) ----
    train = None
    if not args.no_train:
        model.train()
        target = (inp["node_loc"] + 0.01 * inp["node_vel"]).detach()
        for p_ in model.parameters():
            p_.grad = None

        def train_step():
            o, xv = model(**inp)
            loss = torch.nn.functional.mse_loss(o, target) + 1e-3 * xv.square().mean()
            loss.backward()

        train_step()
        barrier()
        n_tr = max(2, min(args.steps, 3))
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        for _ in range(n_tr):
            train_step()
        e.record()
        barrier()
        t_tr = max_over_ranks(s.elapsed_time(e) * 1e-3 / n_tr)
        train = {"value": 1.0 / t_tr, "unit": "train-steps/s", "ms_per_step": t_tr * 1e3, "steps": n_tr,
                 "peak_mem_gb": round(torch.cuda.max_memory_allocated(dev) / 2 ** 30, 2),
                 "includes": "forward (sm_100a kernels, activations kept per layer) + backward (hand-written kernels for every "
                             "stage: edge and real<->virtual on tcgen05, node stage / embedding / virtual update as fp32 "
                             "tile kernels; packed gradient exchange); no optimizer step"}
        model.eval()
        for p_ in model.parameters():
            p_.grad = None

    t_step = max_over_ranks(t_dev / args.steps)
    e_total = int(sum_over_ranks(E))
    n_total = int(sum_over_ranks(N))
    t_edge_max = max_over_ranks(t_edge)
    peak, peak_src = peaks()
    bytes_edge = edge_kernel_bytes(N, E)
    achieved = bytes_edge / t_edge / 1e9 if t_edge > 0 else 0.0
    traffic = None
    tr_path = os.path.join(ROOT, "profiles", "edge_kernel_traffic.json")
    if os.path.exists(tr_path) and world == 1:
        try:
            tj = json.load(open(tr_path))
            if tj.get("workload") == w.name and tj.get("n_nodes") == full_nodes:
                traffic = tj.get("dram_bytes_per_launch")
        except Exception:
            pass

    tpeak, tpeak_src = tensor_peak()
    flops_virt = virtual_kernel_flops(N, w.virtual_channels)
    t_virt_max, t_node_max, t_upd_max = max_over_ranks(t_virt), max_over_ranks(t_node), max_over_ranks(t_upd)
    collective = "none (single partition)" if world == 1 else (
        "p2p-fused: push over NVLink peer memory inside the virtual-node update kernel (csrc/comm.cuh)" if model._comm
        else "torch.distributed all_reduce (NCCL)")
    if rank == 0:
        line = {
            "metric": METRIC, "value": 1.0 / t_step, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": t_step * 1e3, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "edges_per_sec": e_total / t_step, "edge_layers_per_sec": e_total * N_LAYERS / t_step,
            "config": {
                "workload": f"{w.name}: {full_nodes} nodes radius graph r={w.radius} (expected degree "
                            f"{w.degree}), C={w.virtual_channels}, F={w.node_feat_nf}, Na={w.node_attr_nf}, "
                            f"{N_LAYERS} layers, hidden 64, normalize={w.normalize}",
                "partitions": world, "split_mode": args.split_mode if world > 1 else "none",
                "nodes_total": n_total, "edges_total_sum_p": e_total, "nodes_rank0": N, "edges_rank0": E,
                "l2": "256 MiB buffer written between timed steps (L2 flush); per-step CUDA events",
                "csr": "cached (built once in warm-up; included in e2e)",
                "cuda_graph": bool(use_graph),
                "graph_gen_s": round(t_gen, 2), "first_forward_s": round(t_first, 3)},
            "clocks": clocks,
            "e2e": e2e,
            "train_step": train,
            "gpu_launches": launches,
            "roofline": {"bound": "hbm", "kernel": "edge_layer_cs_kernel", "achieved": achieved, "peak": peak,
                         "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
                         "bytes_per_launch": bytes_edge, "ms_per_launch": t_edge * 1e3, "peak_source": peak_src,
                         "note": "rank-0 kernel; algorithmic bytes = E*284 + N*536 (SURVEY §8d)"},
            "roofline_virtual": {"bound": "tensor", "kernel": "virtual_layer_t16_kernel",
                                 "achieved": flops_virt / t_virt / 1e12 if t_virt > 0 else 0.0, "peak": tpeak,
                                 "unit": "TFLOP/s", "frac": (flops_virt / t_virt / 1e12 / tpeak) if t_virt > 0 else 0.0,
                                 "flops_per_launch": flops_virt, "ms_per_launch": t_virt * 1e3, "peak_source": tpeak_src,
                                 "note": "rank-0 kernel; LOGICAL flops (3 64x64 layers + 2 head dots per node-channel row); "
                                         "each layer runs as 3 fp16-split products on tcgen05, so the tensor pipe does 3x "
                                         "this; the kernel is bound by instruction issue of its SiLU epilogues (ncu)"},
            "kernel_ms": {"edge": t_edge_max * 1e3, "virtual": t_virt_max * 1e3, "node": t_node_max * 1e3,
                          "sync_update": t_upd_max * 1e3,
                          "note": "CUDA-event durations per launch (mean over layers and steps, eager launches)",
                          "wall_ms_per_step": wall / args.steps * 1e3},
            "collective": collective,
            "dist_parity": dist_parity,
        }
    else:
        line = None

    # ---- CPU baseline beside it (rank 0, N=1 only) ----
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        t, n, e, cores, kind = cpu_reference_time(w, {k: v.cpu() for k, v in sd.items()}, args.cpu_sample_nodes, 2)
        eps = e / t
        full_edges_est = e * (full_nodes / n)
        line["cpu_baseline"] = {
            "value": eps / full_edges_est, "unit": UNIT, "cores": cores, "kind": kind, "cpu": cpu_model_name(),
            "edges_per_sec": eps, "sample_seconds": t,
            "sample": ("the unmodified reference models/FastEGNN.py (oracle/_ref)" if kind == "reference"
                       else "oracle port (reference op sequence)")
                      + f", torch CPU fp32, {cores} threads = fastest of a thread-count "
                      f"probe on this {os.cpu_count()}-thread host: forward on a {n}-node/"
                      f"{e}-edge sub-cloud of the same density, best of 2 after warm-up; rate scaled by "
                      f"node ratio {full_nodes / n:.1f}x to the full graph (the full-size measurement is "
                      f"`bench.py --impl reference`)"}
    if rank == 0:
        print(json.dumps(line), flush=True)
    if world > 1:
        model.release_comm()
        dist.barrier()
        dist.destroy_process_group()


def main():
    args = parse()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("--gpus N>1 must be launched with torch.distributed.run (one rank per GPU)")
    w = synth.WORKLOADS[args.workload]
    if args.impl == "reference":
        run_reference(args, w, rank, world)
    else:
        run_ours(args, w, rank, world, local_rank)


if __name__ == "__main__":
    main()
