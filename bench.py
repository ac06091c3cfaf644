"""bench.py — graphs/sec through GPSLayer forward+backward on PCQM4M-shaped synthetic batches.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload NAME] [--dump-outputs DIR]
    python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...

A *step* is one GPSLayer forward+backward (training mode, BatchNorm batch statistics, dropout as
configured by configs/GPS/pcqm4m-GPS+RWSE.yaml: dropout 0.0, attn_dropout 0.5) over one synthetic
256-graph PCQM4Mv2-shaped mini-batch per GPU (SURVEY.md 8d, config C3).  For N > 1 every rank
processes its own mini-batch (weak scaling) and the parameter gradients are all-reduced over NCCL
inside the step.  One JSON line is printed by rank 0.

  value     graphs/s with inputs resident in HBM, CUDA-event timed per step, L2 flushed between steps
  e2e       same metric through the public API with HOST (pinned) inputs: H2D of x/edge_attr/
            edge_index/batch, graph build, fwd+bwd, D2H of x_out and grad_x inside the timed region
  roofline  dominant kernel of the step, timed live with CUDA events around its C-ABI stage call
  cpu_baseline  the reference's own GPSLayer (oracle/_ref run verbatim under oracle/ref_shim.py; the
            oracle port if the files are absent) on the host cores, bounded sample of the same workload

--dump-outputs DIR writes what the last timed step returned to its caller (x_out, edge_out, grad_x, grad_edge_attr,
grad.<parameter>) as float32 DIR/<name>.npy.  Inputs, weights and dropout streams are seeded, so two builds run with
the same arguments can be compared array by array.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

WORKLOADS = {
    # name: (shape key, local, global, heads, dropout, attn_dropout, config file it mirrors)
    "pcqm4m-small": ("pcqm4m-small", "CustomGatedGCN", "Transformer", 4, 0.0, 0.5, "configs/GPS/pcqm4m-GPS+RWSE.yaml"),
    "zinc-gatedgcn": ("zinc-gatedgcn", "CustomGatedGCN", "Transformer", 4, 0.0, 0.5, "configs/GPS/zinc-GPS+RWSE.yaml"),
    "zinc-gine": ("zinc-gine", "GINE", "Transformer", 4, 0.0, 0.5, "configs/GPS/zinc-GPS+RWSE.yaml"),
    "zinc-gcn": ("zinc-gine", "GCN", "Transformer", 4, 0.2, 0.0,
                 "layer settings of configs/GPS/webkb-tex-GPS.yaml (GCN+Transformer d=64 H=4) on the ZINC-shaped batch"),
    "code2": ("code2", "CustomGatedGCN", "Transformer", 4, 0.2, 0.2, "configs/GPS/ogbg-code2-GPS.yaml"),
    "pcqm4m-medium-performer": ("pcqm4m-medium-performer", "CustomGatedGCN", "Performer", 16, 0.1, 0.1,
                                "configs/GPS/pcqm4m-GPSmedium+RWSE.yaml (Performer as BASELINE.json asks)"),
}
NUM_BATCHES = 8          # rotating distinct batches
L2_FLUSH_BYTES = 256 << 20
DUMP_LIMIT_BYTES = 64 << 20


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        p = json.load(open(path))
        return dict(hbm=p["hbm_gbs"], tensor=p["bf16_tflops"], tensor_sustained=p["bf16_tflops_sustained"],
                    source="measured (MEASURED_PEAKS.json)")
    return dict(hbm=6650.0, tensor=1590.0, tensor_sustained=1400.0, source="fallback (B200_PROFILING.md)")


class ClockSampler:
    """SM clock / throttle-reason sampling DURING the timed region (B200_PROFILING.md recipe).

    The timed region of this benchmark is tens of milliseconds, far below nvidia-smi's loop period, so the
    same counters are read through NVML (nvidia_ml_py) from a thread every ~2 ms; nvidia-smi is the fallback."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self.thr = None
        self.nvml = None
        try:
            import pynvml
            pynvml.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(vis.split(",")[index]) if vis and vis.split(",")[index].isdigit() else index
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM))
            self.nvml = pynvml
        except Exception:
            self.nvml = None

    def _loop_nvml(self):
        n = self.nvml
        bits = {"hw_slowdown": getattr(n, "nvmlClocksEventReasonHwSlowdown", 0x8),
                "hw_thermal_slowdown": getattr(n, "nvmlClocksEventReasonHwThermalSlowdown", 0x40),
                "sw_thermal_slowdown": getattr(n, "nvmlClocksEventReasonSwThermalSlowdown", 0x20),
                "sw_power_cap": getattr(n, "nvmlClocksEventReasonSwPowerCap", 0x4)}
        get_reasons = getattr(n, "nvmlDeviceGetCurrentClocksEventReasons", None) or \
            getattr(n, "nvmlDeviceGetCurrentClocksThrottleReasons", None)
        while not self._stop.is_set():
            try:
                self.samples.append(float(n.nvmlDeviceGetClockInfo(self.handle, n.NVML_CLOCK_SM)))
                if get_reasons is not None:
                    r = int(get_reasons(self.handle))
                    for name, bit in bits.items():
                        if r & bit:
                            self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.002)

    def start(self):
        if self.nvml is not None:
            self.thr = threading.Thread(target=self._loop_nvml, daemon=True)
            self.thr.start()
            return
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thr = threading.Thread(target=self._read, daemon=True)
            self.thr.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.nvml is not None:
            self._stop.set()
            if self.thr is not None:
                self.thr.join(timeout=1)
            sm = sorted(self.samples)
            return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": self.max_mhz,
                    "reasons": sorted(self.reasons), "samples": len(sm), "source": "nvml, 2 ms period"}
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [t.strip() for t in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for nm, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm), "source": "nvidia-smi -lms 20"}


def make_workload(name, seed, device=None):
    import graphgps_b200
    shape, local, glob, heads, drop, adrop, _ = WORKLOADS[name]
    spec = graphgps_b200.SHAPES[shape]
    batches = [graphgps_b200.make_batch(shape, seed=seed * 1000 + i) for i in range(NUM_BATCHES)]
    return spec, local, glob, heads, drop, adrop, batches


# ================================================================================ reference arm
def cpu_reference_layer(spec, local, glob, heads, drop, adrop):
    """The reference's own GPSLayer on the CPU (oracle/_ref verbatim under the shim) or the port."""
    from oracle.ref_shim import find_reference_layer_dir, load_reference
    torch.manual_seed(0)
    if find_reference_layer_dir() is not None:
        ref = load_reference()
        return ref.GPSLayer(spec.dim, local, glob, heads, dropout=drop, attn_dropout=adrop), "reference"
    from oracle.gps_oracle import OracleGPSLayer
    return OracleGPSLayer(spec.dim, local, glob, heads, dropout=drop, attn_dropout=adrop), "port"


def pick_cpu_threads(layer, batches, local):
    """Thread count that makes the reference fastest on this host (torch's default of one thread per
    logical core is ~50x slower than 8-16 threads on a 128-core box for these small ops)."""
    cores = os.cpu_count() or 1
    best, best_t = 1, float("inf")
    for nt in [c for c in (4, 8, 16, 32, 64) if c <= cores] + ([cores] if cores < 4 else []):
        torch.set_num_threads(nt)
        t = min(time_cpu(layer, batches, 1, 1, local))
        if t < best_t:
            best, best_t = nt, t
        elif t > 1.5 * best_t:
            break
    torch.set_num_threads(best)
    return best


def time_cpu(layer, batches, steps, warmup, local):
    layer.train()
    times = []
    for it in range(warmup + steps):
        b = batches[it % len(batches)].clone()
        b.x.requires_grad_(True)
        b.edge_attr.requires_grad_(True)
        for p in layer.parameters():
            p.grad = None
        t0 = time.perf_counter()
        out = layer(b)
        loss = out.x.sum() + (out.edge_attr.sum() if local == "CustomGatedGCN" else 0.0)
        loss.backward()
        t1 = time.perf_counter()
        if it >= warmup:
            times.append(t1 - t0)
    return times


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    spec, local, glob, heads, drop, adrop, batches = make_workload(args.workload, seed=0)
    layer, kind = cpu_reference_layer(spec, local, glob, heads, drop, adrop)
    cores = pick_cpu_threads(layer, batches, local)
    steps = min(args.steps, 20)   # bounded sample: ~0.05-0.25 s per step at C3 (each step is one full batch fwd+bwd)
    times = time_cpu(layer, batches, steps, args.warmup, local)
    total = sum(times)
    B = spec.num_graphs
    value = B * len(times) / total
    out = {
        "impl": "reference", "metric": "graphs/sec GPSLayer fwd+bwd", "value": value, "unit": "graphs/s",
        "n_gpus": args.gpus, "steps": len(times), "warmup": args.warmup,
        "ms_per_step": 1e3 * total / len(times), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args.workload, spec, local, glob, heads, drop, adrop, 1),
        "cpu_baseline": {"value": value, "unit": "graphs/s", "cores": cores, "kind": kind,
                         "sample": f"{len(times)} steps of one {B}-graph batch fwd+bwd, torch fp32, {cores} threads "
                                   f"(fastest of 4..64 on a {os.cpu_count()}-core host)"},
        "e2e": {"value": value, "unit": "graphs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(out), flush=True)


def workload_config(name, spec, local, glob, heads, drop, adrop, n_gpus):
    return {"workload": f"{name}: one GPSLayer({local}+{glob}) fwd+bwd, d={spec.dim} H={heads}, "
                        f"{spec.num_graphs} graphs/GPU (~{spec.n_mean:.0f} nodes/graph), dropout={drop} "
                        f"attn_dropout={adrop}; mirrors {WORKLOADS[name][6]}",
            "graphs_per_gpu": spec.num_graphs, "global_batch": spec.num_graphs * n_gpus,
            "parallelism": f"dp{n_gpus}", "l2": f"flushed between steps ({L2_FLUSH_BYTES >> 20} MiB write) and "
                                                f"{NUM_BATCHES} rotating batches"}


# ================================================================================ our arm
def dump_outputs(path, out, x_in, e_in, layer, gated):
    """Writes one step's layer outputs, input gradients and parameter gradients as float32 .npy files; beyond
    DUMP_LIMIT_BYTES in all, every array keeps the same share of its rows, chosen with a fixed seed."""
    import numpy as np
    arrays = {"x_out": out.x, "grad_x": x_in.grad}
    if gated:
        arrays["edge_out"] = out.edge_attr
    if e_in.grad is not None:
        arrays["grad_edge_attr"] = e_in.grad
    arrays.update({"grad." + n: p.grad for n, p in layer.named_parameters() if p.grad is not None})
    arrays = {k: v.detach().float().cpu() for k, v in arrays.items()}
    total = sum(v.numel() * 4 for v in arrays.values())
    if total > DUMP_LIMIT_BYTES:
        gen = torch.Generator().manual_seed(0)
        for k, v in arrays.items():
            keep = max(1, v.shape[0] * DUMP_LIMIT_BYTES // total)
            arrays[k] = v[torch.randperm(v.shape[0], generator=gen)[:keep].sort().values]
    os.makedirs(path, exist_ok=True)
    for k, v in arrays.items():
        np.save(os.path.join(path, k + ".npy"), v.numpy())


def trace(msg):
    """GPS_BENCH_TRACE=1: stage markers on stderr (+ a watchdog that dumps every thread's stack if a stage hangs)."""
    if os.environ.get("GPS_BENCH_TRACE") == "1":
        import faulthandler
        faulthandler.cancel_dump_traceback_later()
        faulthandler.dump_traceback_later(int(os.environ.get("GPS_BENCH_TRACE_TIMEOUT", "120")), exit=True)
        sys.stderr.write(f"[bench rank {os.environ.get('RANK', '0')} {time.strftime('%H:%M:%S')}] {msg}\n")
        sys.stderr.flush()


def run_ours(args):
    import graphgps_b200
    from graphgps_b200 import _lib
    from graphgps_b200.graph import graph_of

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs a GPU: graphgps_b200 has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)
    lib = _lib.load()

    spec, local, glob, heads, drop, adrop, cpu_batches = make_workload(args.workload, seed=rank)
    torch.manual_seed(0)
    layer = graphgps_b200.GPSLayer(spec.dim, local, glob, heads, dropout=drop, attn_dropout=adrop,
                                   precision=args.precision).to(dev).train()
    params = [p for p in layer.parameters()]
    gated = local == "CustomGatedGCN"

    dev_batches = [b.clone().to(dev) for b in cpu_batches]
    for b in dev_batches:
        graph_of(b)                     # structure is per-batch, amortised over the L layers of a model
    gen = torch.Generator().manual_seed(1)
    cts = [(torch.randn(b.x.shape, generator=gen).to(dev), torch.randn(b.edge_attr.shape, generator=gen).to(dev))
           for b in cpu_batches]
    flush = torch.empty(L2_FLUSH_BYTES, dtype=torch.uint8, device=dev)
    # Static gradient bucket (graphgps_b200.dp.GradBucket): every p.grad is a view of one flat buffer that the backward
    # pass accumulates into, so CUDA-graph replays and the collective see the same memory.  For N > 1 the bucket is
    # all-reduced in place (NCCL AVG): the early segment (FFN / out-proj / norms) on a communication stream as soon as
    # the library signals it, under the rest of the backward pass; the late segment at the end.
    from graphgps_b200.dp import GradBucket
    bucket = GradBucket([layer])
    if world > 1:
        bucket.enable_overlap()
        dist.all_reduce(torch.zeros(1, device=dev))      # communicator up before any capture

    def allreduce_grads(overlap=True):
        if world > 1:
            if overlap:
                bucket.allreduce_overlapped()
            else:
                bucket.allreduce()

    def step(i, bobj=None, reduce=True):
        b = bobj if bobj is not None else dev_batches[i % NUM_BATCHES]
        ctx, cte = cts[i % NUM_BATCHES]
        bb = graphgps_b200.GraphBatch(x=b.x.detach().requires_grad_(True), edge_index=b.edge_index,
                                      edge_attr=b.edge_attr.detach().requires_grad_(True), batch=b.batch,
                                      num_graphs=b.num_graphs)
        if "_gps_b200_graph" in b.__dict__:
            bb.__dict__["_gps_b200_graph"] = b.__dict__["_gps_b200_graph"]
        bucket.zero_()
        x_in = bb.x
        out = layer(bb)
        if gated:
            torch.autograd.backward([out.x, out.edge_attr], [ctx, cte])
        else:
            torch.autograd.backward([out.x], [ctx])
        if reduce:
            allreduce_grads()
        return out, x_in, bb.edge_attr

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---------------- device-resident timing
    # Eager warm-up (also sizes the shared workspace), then one CUDA graph per rotating batch: a replay
    # re-executes the captured kernel sequence (forward + backward of the layer) with no host work.
    trace("eager warm-up")
    for i in range(max(args.warmup, NUM_BATCHES)):
        step(i)
    barrier()
    trace("capture")
    graphs = None
    graphs_local = None            # the same step without the collectives (N > 1: exposes the all-reduce cost)
    results = None                 # per graph: the (out, x_in, e_in) its replays overwrite
    launches_per_step = None
    collective_in_graph = False

    def capture_all(reduce):
        out, res = [], []
        nonlocal launches_per_step
        for i in range(NUM_BATCHES):
            g = torch.cuda.CUDAGraph()
            l0 = lib.gps_launch_count()
            with torch.cuda.graph(g, capture_error_mode="thread_local"):
                res.append(step(i, reduce=reduce))
            launches_per_step = lib.gps_launch_count() - l0
            out.append(g)
        return out, res

    if args.graph:
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for i in range(NUM_BATCHES):
                step(i, reduce=True)
        torch.cuda.current_stream().wait_stream(side)
        barrier()
        if world > 1 and os.environ.get("GPS_BENCH_NCCL_IN_GRAPH") == "1":
            try:     # NCCL collectives captured in the same graph as the step (measured: ~0.5 ms of host time per launch)
                graphs, results = capture_all(True)
                collective_in_graph = True
            except Exception as e:   # noqa: BLE001
                sys.stderr.write(f"[bench] capturing the collectives failed ({e!r}); they run after each replay\n")
                graphs = None
                torch.cuda.synchronize()
        # default: the graph holds fwd+bwd and records the gradient-group events as external event nodes; the
        # collectives are enqueued after each replay and wait on those events (overlap without NCCL graph nodes)
        graphs_local, results_local = capture_all(False)
        if graphs is None:
            graphs, results = graphs_local, results_local

    def run_step(i):
        if graphs is None:
            return step(i)
        graphs[i % NUM_BATCHES].replay()
        if world > 1 and not collective_in_graph:
            allreduce_grads()
        return results[i % NUM_BATCHES]

    trace("graph warm-up")
    for i in range(args.warmup):
        run_step(i)
    barrier()
    trace("timed region")
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    evs = []
    l0 = lib.gps_launch_count()
    host_t0 = time.perf_counter()
    for i in range(args.steps):
        flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        last = run_step(i)
        e1.record()
        evs.append((e0, e1))
    host_ms = (time.perf_counter() - host_t0) * 1e3 / args.steps   # host enqueue time per step (no sync inside)
    barrier()
    launches = launches_per_step if graphs is not None else (lib.gps_launch_count() - l0) // max(1, args.steps)
    ms = sum(a.elapsed_time(b) for a, b in evs)
    clocks = sampler.stop() if rank == 0 else None
    t = torch.tensor([ms], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_total = float(t.item())
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, *last, layer, gated)

    # N > 1: the same replays without the collectives -> what the all-reduce still costs after overlap
    trace("no-collective replays")
    local_ms = None
    if world > 1 and graphs_local is not None:
        for i in range(args.warmup):
            graphs_local[i % NUM_BATCHES].replay()
        barrier()
        le = []
        for i in range(args.steps):
            flush.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            graphs_local[i % NUM_BATCHES].replay()
            e1.record()
            le.append((e0, e1))
        barrier()
        tl = torch.tensor([sum(a.elapsed_time(b) for a, b in le)], device=dev, dtype=torch.float64)
        dist.all_reduce(tl, op=dist.ReduceOp.MAX)
        local_ms = float(tl.item()) / args.steps

    # eager (no CUDA graph) number for the same loop, reported alongside
    trace("eager timing")
    eager_ms = None
    if graphs is not None:
        for i in range(3):
            step(i)
        barrier()
        ee = []
        for i in range(min(args.steps, 20)):
            flush.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            step(i)
            e1.record()
            ee.append((e0, e1))
        barrier()
        eager_ms = sum(a.elapsed_time(b) for a, b in ee) / len(ee)

    # ---------------- end-to-end through the public API with host buffers
    # Every step: H2D of that step's x / edge_attr / edge_index / batch from pinned host memory, graph-structure
    # build, layer forward + backward, D2H of x_out and grad_x into pinned host memory.  The copies run on their
    # own streams (PCIe is full duplex), two steps deep, so step k+1's inputs travel while step k computes; the
    # timed region spans the first H2D to the last D2H (device events), i.e. it includes every byte moved.
    trace("e2e")
    pinned = [b.clone().pin_memory() for b in cpu_batches]
    static = [b.clone().to(dev) for b in cpu_batches]
    host_x = [torch.empty(b.x.shape).pin_memory() for b in cpu_batches]
    host_g = [torch.empty(b.x.shape).pin_memory() for b in cpu_batches]
    h2d = sum(t.numel() * t.element_size() for t in (pinned[0].x, pinned[0].edge_index, pinned[0].edge_attr, pinned[0].batch))
    d2h = 2 * pinned[0].x.numel() * 4
    outs = [None] * NUM_BATCHES

    def e2e_body(i):
        sb = static[i]
        bb = graphgps_b200.GraphBatch(x=sb.x.detach().requires_grad_(True), edge_index=sb.edge_index,
                                      edge_attr=sb.edge_attr.detach().requires_grad_(True), batch=sb.batch,
                                      num_graphs=sb.num_graphs)     # no cached structure: gps_graph_build runs
        bucket.zero_()
        x_in = bb.x
        out = layer(bb)
        ctx, cte = cts[i]
        if gated:
            torch.autograd.backward([out.x, out.edge_attr], [ctx, cte])
        else:
            torch.autograd.backward([out.x], [ctx])
        return out.x.detach(), x_in.grad

    e2e_graphs = None
    for i in range(NUM_BATCHES):
        outs[i] = e2e_body(i)
    barrier()
    if args.graph:
        e2e_graphs = []
        for i in range(NUM_BATCHES):
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, capture_error_mode="thread_local"):
                outs[i] = e2e_body(i)
            e2e_graphs.append(g)
    s_h2d, s_d2h, s_cmp = torch.cuda.Stream(), torch.cuda.Stream(), torch.cuda.current_stream()

    def e2e_run(nsteps):
        ev_in = [torch.cuda.Event() for _ in range(nsteps)]
        ev_cmp = [torch.cuda.Event() for _ in range(nsteps)]
        ev_out = [torch.cuda.Event() for _ in range(nsteps)]
        e_start, e_end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

        def h2d_step(k):
            i = k % NUM_BATCHES
            with torch.cuda.stream(s_h2d):
                if k >= NUM_BATCHES:
                    s_h2d.wait_event(ev_cmp[k - NUM_BATCHES])      # buffers of batch i are free again
                for name in ("x", "edge_index", "edge_attr", "batch"):
                    getattr(static[i], name).copy_(getattr(pinned[i], name), non_blocking=True)
                ev_in[k].record(s_h2d)

        e_start.record(s_h2d)
        for k in range(min(2, nsteps)):
            h2d_step(k)
        for k in range(nsteps):
            i = k % NUM_BATCHES
            s_cmp.wait_event(ev_in[k])
            if k >= NUM_BATCHES:
                s_cmp.wait_event(ev_out[k - NUM_BATCHES])           # previous results of batch i were read out
            if e2e_graphs is not None:
                e2e_graphs[i].replay()
            else:
                outs[i] = e2e_body(i)
            allreduce_grads(overlap=False)   # the early-gradient event lives inside the captured graph here
            ev_cmp[k].record(s_cmp)
            with torch.cuda.stream(s_d2h):
                s_d2h.wait_event(ev_cmp[k])
                host_x[i].copy_(outs[i][0], non_blocking=True)
                host_g[i].copy_(outs[i][1], non_blocking=True)
                ev_out[k].record(s_d2h)
            if k + 2 < nsteps:
                h2d_step(k + 2)
        e_end.record(s_d2h)
        torch.cuda.synchronize()
        return e_start.elapsed_time(e_end)

    e2e_run(min(4, args.steps))
    barrier()
    e_ms = e2e_run(args.steps)
    t = torch.tensor([e_ms], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e_ms_total = float(t.item())

    trace("roofline probe")
    roof = roofline_probe(lib, layer, dev_batches[0], spec, heads, args) if rank == 0 else None
    trace("stack")

    # ---------------- the model's layer stack (gps_model.py:100,105-108): L GPSLayers back to back, fwd+bwd, as
    # ONE captured CUDA graph over a resident batch (graph structure shared by all layers).  Measured last and
    # guarded, so a failure here can only drop this extra key.
    stack = None
    if args.graph and spec.layers > 1:
        try:
            torch.manual_seed(1)
            gstack = graphgps_b200.GPSStack(spec.layers, spec.dim, local, glob, heads, dropout=drop, attn_dropout=adrop,
                                            precision=args.precision).to(dev).train()
            sbucket = gstack.make_grad_bucket(overlap=world > 1)
            coll = (lambda: sbucket.allreduce_overlapped()) if world > 1 else (lambda: None)
            steps_c = [gstack.capture(dev_batches[i], cts[i][0], cts[i][1] if gated else None, bucket=sbucket)
                       for i in range(2)]
            for i in range(4):
                steps_c[i % 2].replay()
                coll()
            barrier()
            se = []
            nst = min(args.steps, 50)
            for i in range(nst):
                flush.zero_()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                steps_c[i % 2].replay()
                coll()
                e1.record()
                se.append((e0, e1))
            barrier()
            ts = torch.tensor([sum(a.elapsed_time(b) for a, b in se)], device=dev, dtype=torch.float64)
            if world > 1:
                dist.all_reduce(ts, op=dist.ReduceOp.MAX)
            sms = float(ts.item()) / nst
            stack = {"layers": spec.layers, "measured": True, "ms_per_step": sms, "ms_per_layer": sms / spec.layers,
                     "graphs_per_s": spec.num_graphs * world / (sms * 1e-3),
                     "how": f"graphgps_b200.GPSStack: {spec.layers} GPSLayers fwd+bwd in one captured CUDA graph per rank "
                            f"(shared graph structure, plane hand-off between layers, one gradient bucket"
                            + (", per-layer all-reduce segments overlapped with the backward of the layers below" if world > 1 else "")
                            + f"), batch resident, L2 flushed between steps, {nst} steps, max over ranks"}
        except Exception as e:   # noqa: BLE001 - the headline numbers above must survive
            stack = {"layers": spec.layers, "measured": False, "error": repr(e)[:300]}

    trace("report")
    if rank == 0:
        B = spec.num_graphs
        value = B * world * args.steps / (ms_total * 1e-3)
        e2e_value = B * world * args.steps / (e_ms_total * 1e-3)
        ref_layer, kind = cpu_reference_layer(spec, local, glob, heads, drop, adrop)
        cores = pick_cpu_threads(ref_layer, cpu_batches, local)
        ct = time_cpu(ref_layer, cpu_batches, 8, 2, local)
        cpu_value = B * len(ct) / sum(ct)
        out = {
            "metric": "graphs/sec GPSLayer fwd+bwd", "value": value, "unit": "graphs/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_total / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32" if args.precision == "fp32" else "bf16", "data": "synthetic",
            "config": workload_config(args.workload, spec, local, glob, heads, drop, adrop, world),
            "e2e": {"value": e2e_value, "unit": "graphs/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "ms_per_step": e_ms_total / args.steps,
                    "how": "pinned host -> H2D -> graph build + fwd + bwd -> D2H(x_out, grad_x); copies on their own "
                           "streams, 2 steps deep; first H2D to last D2H by device events"},
            "gpu_launches": int(launches), "host_enqueue_ms_per_step": host_ms,
            "gemm_fallbacks": int(lib.gps_fallback_count()),
            "allreduce": (None if world == 1 else {
                "bytes": int(bucket.flat.numel() * 4), "in_graph": bool(collective_in_graph),
                "how": "in-place NCCL AVG on the static gradient bucket, three segments per layer on a communication stream, "
                       "each released by an event the backward pass records when that gradient group is final",
                "ms_per_step_without_collectives": local_ms,
                "exposed_ms_per_step": (None if local_ms is None else ms_total / args.steps - local_ms)}),
            "execution": ("CUDA graph replay (one captured fwd+bwd"
                          + ("+all-reduce" if collective_in_graph else "") + " graph per rotating batch shape)"
                          if args.graph else "eager launches"),
            "eager": ({"ms_per_step": eager_ms, "value": B * world / (eager_ms * 1e-3)} if eager_ms else None),
            "clocks": clocks, "roofline": roof,
            "cpu_baseline": {"value": cpu_value, "unit": "graphs/s", "cores": cores, "kind": kind,
                             "sample": f"{len(ct)} steps of one {B}-graph batch fwd+bwd (same workload), "
                                       f"torch fp32, {cores} threads (fastest of 4..64 on a {os.cpu_count()}-core host)"},
            "stack": stack if stack and stack.get("measured") else dict(
                stack or {}, layers=spec.layers, measured=False, graphs_per_s=value / spec.layers,
                how="single-layer value / L (not measured as a stack)"),
        }
        print(json.dumps(out), flush=True)
    if world > 1:
        # destroy_process_group() blocks forever while captured CUDA graphs that contain NCCL kernels are alive
        # (observed with torch 2.11 / NCCL 2.28): release them, synchronise, and leave without the collective teardown
        trace("teardown")
        torch.cuda.synchronize()
        dist.barrier()
        sys.stdout.flush()
        sys.stderr.flush()
        os._exit(0)


def roofline_probe(lib, layer, b, spec, heads, args):
    """Times the step's two headline kernels live (CUDA events around their C-ABI stage calls, L2 flushed, host
    launch latency hidden behind a spin kernel): the longest single kernel of the step — the data-gradient GEMM
    g_x = gY1[N,7d] . Wcat[7d,d] (tensor bound, 2*N*7d*d flop) — and the GatedGCN gather-reduce (HBM bound,
    4*(5N+2E)*d algorithmic bytes, SURVEY.md 8d).  `traffic` = DRAM bytes per launch of the same kernels from the
    committed `ncu --set full` capture (profiles/r1_roofline_traffic.json)."""
    import ctypes as C
    from graphgps_b200.graph import graph_of
    pk = peaks()
    gs = graph_of(b)
    dev = b.x.device
    N, E, d = gs.N, gs.E, spec.dim
    stream = torch.cuda.current_stream().cuda_stream
    flush = torch.empty(L2_FLUSH_BYTES, dtype=torch.uint8, device=dev)
    # DRAM bytes per launch from the committed `ncu --set full` capture of THIS workload (null when none was taken)
    traffic = {}
    tpath = os.path.join(ROOT, "profiles", "r2_roofline_traffic.json")
    if os.path.exists(tpath):
        traffic = json.load(open(tpath)).get(f"{args.workload}:{args.precision}", {})
    res = {}

    def timeit(fn, reps=10):
        for _ in range(3):
            fn()
        tot = 0.0
        for _ in range(reps):
            flush.zero_()
            torch.cuda._sleep(300000)   # GPU busy while the host enqueues: the events bracket only the kernel
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            torch.cuda.synchronize()
            tot += e0.elapsed_time(e1)
        return tot / reps * 1e-3

    prec = 0 if args.precision == "fp32" else 1
    Wy = 7 * d
    W = torch.randn(Wy, d, device=dev) / d ** 0.5
    gY = torch.randn(N, Wy, device=dev)
    gx = torch.zeros(N, d, device=dev)

    def planes(t):   # bf16 hi/lo operand planes, as the producing kernels of the layer write them
        r, c = t.shape
        ld = (c + 7) // 8 * 8
        buf = torch.zeros(2, r, ld, dtype=torch.bfloat16, device=dev)
        _ = lib.gps_to_planes(t.data_ptr(), t.stride(0), r, c, buf[0].data_ptr(), buf[1].data_ptr() if prec == 0 else 0, ld, stream)
        return buf, ld

    gYp, ldg = planes(gY)
    Wp, ldw = planes(W)
    # split-K 4 accumulates atomically into gx (the layer zeroes it with a memset that is not part of the kernel)
    t_g = timeit(lambda: lib.gps_gemm_planes(gYp[0].data_ptr(), gYp[1].data_ptr() if prec == 0 else 0, ldg, 0,
                                             Wp[0].data_ptr(), Wp[1].data_ptr() if prec == 0 else 0, ldw, 1,
                                             gx.data_ptr(), d, 0, 0, 0, N, d, Wy, 4, prec, 0, stream))
    flops = 2.0 * N * Wy * d
    res["gemm"] = {"bound": "tensor", "achieved": flops / t_g / 1e12, "peak": pk["tensor"], "unit": "TFLOP/s",
                   "frac": flops / t_g / 1e12 / pk["tensor"], "traffic": traffic.get("gemm_dgrad_x"), "seconds": t_g,
                   "kernel": "k_gemm_tma data gradient g_x[N,d] = gY1[N,7d] x Wcat[7d,d] (TMA-fed tcgen05 on bf16 hi/lo planes, "
                             + ("3 MMAs per product" if prec == 0 else "1 MMA per product") + ", split-K 4)",
                   "algorithmic_flops": flops, "peak_source": pk["source"]}
    Y = torch.randn(N, Wy, device=dev)
    Ce = torch.randn(E, d, device=dev)
    xt = torch.empty(N, d, device=dev)
    sx = torch.zeros(2, d, device=dev, dtype=torch.float64)
    se = torch.zeros(2, d, device=dev, dtype=torch.float64)
    t_s = timeit(lambda: lib.gps_gatedgcn_aggregate_forward(C.byref(gs.desc), d, Y.data_ptr(), Y.data_ptr() + 4 * d,
                                                            Y.data_ptr() + 8 * d, Y.data_ptr() + 12 * d, Wy,
                                                            Ce.data_ptr(), xt.data_ptr(), sx.data_ptr(), se.data_ptr(),
                                                            stream))
    nbytes = 4.0 * (5 * N + 2 * E) * d
    res["scatter"] = {"bound": "hbm", "achieved": nbytes / t_s / 1e9, "peak": pk["hbm"], "unit": "GB/s",
                      "frac": nbytes / t_s / 1e9 / pk["hbm"], "traffic": traffic.get("gatedgcn_fwd"), "seconds": t_s,
                      "kernel": "k_gatedgcn_fwd CSR segmented gather-reduce (+BatchNorm column sums)",
                      "algorithmic_bytes": nbytes, "peak_source": pk["source"]}
    dom = "gemm" if t_g >= t_s else "scatter"
    out = dict(res[dom])
    out["other"] = res["scatter" if dom == "gemm" else "gemm"]
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="pcqm4m-small", choices=sorted(WORKLOADS))
    ap.add_argument("--precision", default="fp32", choices=["fp32", "bf16"])
    ap.add_argument("--no-graph", dest="graph", action="store_false", help="time eager launches instead of CUDA-graph replays")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's outputs and gradients as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
