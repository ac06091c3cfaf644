"""Cost of the EquivStableLapPE edge gate at the pcqm4m-GPS-ESLapPE shape: one GPSLayer (CustomGatedGCN+Transformer,
d=304, 4 heads, 256 graphs, dropout 0, attn_dropout 0.5), forward + backward, with and without equivstable_pe, same
weights, timed alternately in one process.

Each variant's step is captured once as a CUDA graph; the timed loop replays ES and plain in turn, overwriting a 256 MB
buffer before every step so neither finds its working set in the 126 MB L2, and times each replay with device events.
Kernel launches per step come from gps_launch_count() over one eager step of each.  Prints one JSON line (GPU name and
power limit read in the same run) and, with --out, writes it to that file.

    python tools/bench_eslappe.py --steps 200 --out profiles/bench_eslappe.json
    python tools/bench_eslappe.py --profile profiles/eslappe_kernels.txt   # torch.profiler, separate run

--profile replays each variant 20 times under torch.profiler (no timing) and writes the per-kernel device time of
both, so the extra time of the ES step can be attributed.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

import graphgps_b200  # noqa: E402
from graphgps_b200 import _lib  # noqa: E402
from graphgps_b200.batch import add_equivstable_pe, make_batch  # noqa: E402
from graphgps_b200.graph import graph_of  # noqa: E402


def power_limit():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        return out or "unknown"
    except Exception:
        return "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--out", default=None)
    ap.add_argument("--profile", default=None, help="write a torch.profiler kernel table of both variants here")
    args = ap.parse_args()
    dev = "cuda:0"
    torch.manual_seed(0)
    es = graphgps_b200.GPSLayer(304, "CustomGatedGCN", "Transformer", 4, dropout=0.0, attn_dropout=0.5,
                                equivstable_pe=True).to(dev).train()
    plain = graphgps_b200.GPSLayer(304, "CustomGatedGCN", "Transformer", 4, dropout=0.0, attn_dropout=0.5).to(dev).train()
    plain.load_state_dict({k: v for k, v in es.state_dict().items() if "mlp_r_ij" not in k}, strict=True)
    b = make_batch("pcqm4m-small", seed=1)
    add_equivstable_pe(b, seed=2, scale=0.3)
    b = b.to(dev)
    graph_of(b)
    g = torch.Generator().manual_seed(3)
    ct_x, ct_e = torch.randn(b.x.shape, generator=g).to(dev), torch.randn(b.edge_attr.shape, generator=g).to(dev)
    x_in = b.x.detach().clone().requires_grad_(True)
    e_in = b.edge_attr.detach().clone().requires_grad_(True)
    pe_in = b.pe_EquivStableLapPE.detach().clone().requires_grad_(True)
    lib = _lib.load()

    def body(layer):
        bb = graphgps_b200.GraphBatch(x=x_in, edge_index=b.edge_index, edge_attr=e_in, batch=b.batch,
                                      num_graphs=b.num_graphs, pe_EquivStableLapPE=pe_in)
        bb.__dict__["_gps_b200_graph"] = graph_of(b)
        for t in [x_in, e_in, pe_in] + list(layer.parameters()):
            t.grad = None
        out = layer(bb)
        torch.autograd.backward([out.x, out.edge_attr], [ct_x, ct_e])

    launches, graphs = {}, {}
    side = torch.cuda.Stream(device=dev)
    for name, layer in (("es", es), ("plain", plain)):
        side.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(side):
            for _ in range(3):
                body(layer)
            torch.cuda.synchronize()
            n0 = lib.gps_launch_count()
            body(layer)
            torch.cuda.synchronize()
            launches[name] = int(lib.gps_launch_count() - n0)
        torch.cuda.current_stream(dev).wait_stream(side)
        gr = torch.cuda.CUDAGraph()
        with torch.cuda.graph(gr, capture_error_mode="thread_local"):
            body(layer)
        graphs[name] = gr
    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=dev)
    if args.profile:
        from torch.profiler import ProfilerActivity, profile
        lines = [f"gpu: {torch.cuda.get_device_name(0)}, power limit {power_limit()}; 20 replays per variant, L2 overwritten"
                 " before each; device time per kernel summed over the 20 replays (us)"]
        for name in ("es", "plain"):
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                for _ in range(20):
                    flush.fill_(1.0)
                    graphs[name].replay()
                torch.cuda.synchronize()
            rows = [(e.key, e.device_time_total, e.count) for e in prof.key_averages() if e.device_time_total > 0
                    and "fill" not in e.key.lower()]
            rows.sort(key=lambda r: -r[1])
            lines.append(f"\n== {name}: total {sum(r[1] for r in rows) / 20:.1f} us of kernel time per step")
            lines += [f"{t / 20:10.1f} us/step  x{c // 20:<3d} {k[:150]}" for k, t, c in rows]
        os.makedirs(os.path.dirname(os.path.abspath(args.profile)), exist_ok=True)
        with open(args.profile, "w") as f:
            f.write("\n".join(lines) + "\n")
        print("\n".join(lines[:40]))
        return
    times = {"es": [], "plain": []}
    for i in range(args.warmup + args.steps):
        for name in (("es", "plain") if i % 2 == 0 else ("plain", "es")):
            flush.fill_(float(i))
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            graphs[name].replay()
            e1.record()
            e1.synchronize()
            if i >= args.warmup:
                times[name].append(e0.elapsed_time(e1))
    med = {k: statistics.median(v) for k, v in times.items()}
    res = {"workload": "pcqm4m-GPS-ESLapPE layer: CustomGatedGCN+Transformer d=304 H=4 B=256 dropout 0 attn_dropout 0.5,"
                       " fwd+bwd, CUDA-graph replay, L2 overwritten before each step",
           "N": b.num_nodes, "E": b.num_edges, "steps": args.steps,
           "es_step_ms_median": round(med["es"], 4), "plain_step_ms_median": round(med["plain"], 4),
           "es_over_plain": round(med["es"] / med["plain"], 4),
           "es_step_ms_p10_p90": [round(sorted(times["es"])[len(times["es"]) // 10], 4),
                                  round(sorted(times["es"])[len(times["es"]) * 9 // 10], 4)],
           "plain_step_ms_p10_p90": [round(sorted(times["plain"])[len(times["plain"]) // 10], 4),
                                     round(sorted(times["plain"])[len(times["plain"]) * 9 // 10], 4)],
           "launches_per_step": launches, "extra_launches": launches["es"] - launches["plain"],
           "gpu": torch.cuda.get_device_name(0), "power_limit": power_limit()}
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
