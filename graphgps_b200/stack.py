"""The GPSLayer stack of a GPSModel as one component (SURVEY.md section 8 f1).

The reference builds `self.layers = torch.nn.Sequential(*[GPSLayer(...)] * L)` and runs it over ONE batch object
(graphgps/network/gps_model.py:85-100, 105-108).  `GPSStack` is that container for the B200 layers plus what the
stack can share that a single layer cannot:
  * the CSR/CSC graph structure is built once per batch and cached on the batch object (graph.py), so all L layers and
    their backward passes reuse it;
  * layer l writes the bf16 hi/lo operand planes of its outputs next to x / edge_attr and layer l+1 consumes them, so no
    layer after the first converts its inputs (ABI-3 plane hand-off, gps_layer.py::_handoff_args); weights are re-packed
    into planes only when a parameter changed (once per optimiser step);
  * one static gradient bucket over all layers (dp.GradBucket) whose per-layer segments are all-reduced while the
    layers below are still in their backward pass;
  * `capture()` records forward + backward (+ the collectives) of the whole stack into one CUDA graph per batch shape.
The same hand-off happens automatically inside an unmodified GPSModel once `graphgym.install()` has rebound GPSLayer:
consecutive layers find the planes on the batch object.
Not folded (measured design decision, DESIGN.md): layer l's norm2 into layer l+1's first GEMM - the TMA-fed GEMM reads
operand planes as stored, so the BatchNorm would have to be folded into a per-step rescale of the weight planes, which
moves as many bytes as the `bn_combine` pass it would remove.
"""
from __future__ import annotations

import torch
import torch.nn as nn

from .dp import GradBucket
from .gps_layer import GPSLayer


class GPSStack(nn.Module):
    def __init__(self, num_layers, dim_h, local_gnn_type, global_model_type, num_heads, **layer_kwargs):
        super().__init__()
        self.layers = nn.ModuleList([GPSLayer(dim_h, local_gnn_type, global_model_type, num_heads, **layer_kwargs)
                                     for _ in range(num_layers)])

    @classmethod
    def from_layers(cls, layers):
        self = cls.__new__(cls)
        nn.Module.__init__(self)
        self.layers = nn.ModuleList(list(layers))
        return self

    def forward(self, batch):
        for layer in self.layers:          # gps_model.py:105-108: each layer consumes the previous layer's batch
            batch = layer(batch)
        return batch

    def make_grad_bucket(self, overlap=False):
        bucket = GradBucket(list(self.layers))
        return bucket.enable_overlap() if overlap else bucket

    def capture(self, batch, ct_x, ct_e=None, bucket=None, collective=None, warmup=2):
        """Records `bucket.zero_(); out = stack(batch); backward(out, cotangents); collective()` into one CUDA graph.

        `batch` must be resident on the GPU with its graph structure already built (graph.graph_of); its x / edge_attr
        (and pe_EquivStableLapPE when present, for equivstable_pe layers) are the graph's static inputs (copy new data
        into them before replay()).  Returns a CapturedStep."""
        from .batch import GraphBatch
        from .graph import graph_of
        gs = graph_of(batch)
        x_in = batch.x.detach().requires_grad_(True)
        e_in = batch.edge_attr.detach().requires_grad_(True) if getattr(batch, "edge_attr", None) is not None else None
        pe = getattr(batch, "pe_EquivStableLapPE", None)
        pe_in = pe.detach().requires_grad_(True) if pe is not None else None
        extra = {"pe_EquivStableLapPE": pe_in} if pe_in is not None else {}
        params = [p for p in self.parameters()]
        res = {}

        def body():
            bb = GraphBatch(x=x_in, edge_index=batch.edge_index, edge_attr=e_in, batch=batch.batch,
                            num_graphs=batch.num_graphs, **extra)
            bb.__dict__["_gps_b200_graph"] = gs
            x_in.grad = None
            if e_in is not None:
                e_in.grad = None
            if pe_in is not None:
                pe_in.grad = None
            if bucket is not None:
                bucket.zero_()
            else:
                for p in params:
                    p.grad = None
            out = self(bb)
            outs, cts = [out.x], [ct_x]
            if ct_e is not None:
                outs.append(out.edge_attr)
                cts.append(ct_e)
            torch.autograd.backward(outs, cts)
            if collective is not None:
                collective()
            res["x"], res["e"] = out.x.detach(), (out.edge_attr.detach() if ct_e is not None else None)

        dev = batch.x.device
        side = torch.cuda.Stream(device=dev)
        side.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(side):
            for _ in range(warmup):
                body()
        torch.cuda.current_stream(dev).wait_stream(side)
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, capture_error_mode="thread_local"):
            body()
        return CapturedStep(g, x_in, e_in, res["x"], res["e"], pe_in)


class CapturedStep:
    """One captured forward+backward of a GPSStack: static inputs, outputs and input gradients."""

    def __init__(self, graph, x_in, e_in, x_out, e_out, pe_in=None):
        self.graph, self.x_in, self.e_in, self.x_out, self.e_out = graph, x_in, e_in, x_out, e_out
        self.pe_in = pe_in

    def replay(self):
        self.graph.replay()

    @property
    def grad_x(self):
        return self.x_in.grad

    @property
    def grad_e(self):
        return self.e_in.grad if self.e_in is not None else None

    @property
    def grad_pe(self):
        """Gradient w.r.t. the batch's pe_EquivStableLapPE summed over the layers (None without one)."""
        return self.pe_in.grad if self.pe_in is not None else None
