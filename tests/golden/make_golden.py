"""Generates tests/golden/*.pt from the REFERENCE ITSELF (its own layer files run verbatim under
oracle/ref_shim.py, fp64), so the fixtures pin both the oracle and the CUDA path on the GPU box,
where /root/reference does not exist.

    python tests/golden/make_golden.py          # needs /root/reference (authoring container)

Each fixture holds: config, inputs (x, edge_index, edge_attr, batch), the module state_dict (fp32),
the cotangents used for the backward pass, and the reference's outputs / input gradients /
parameter gradients / updated BatchNorm running statistics (computed in fp64, stored as fp32).

It also writes tests/golden/reference/*.pt: the reference's fp64 results for the weights and inputs that
tests/test_oracle.py::test_oracle_equals_reference_live and
tests/test_layer_gpu.py::test_three_layer_stack_matches_reference_stack build from fixed seeds, kept as
tests/util.sample_summary (seeded sample + full-tensor sums), with summaries of those weights and inputs so a
drift of the seeded construction is reported as such.
"""
import os
import zlib
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from graphgps_b200.batch import make_batch, batch_from_lists  # noqa: E402
from oracle.gps_oracle import OracleGPSLayer  # noqa: E402
from oracle.ref_shim import load_reference  # noqa: E402

sys.path.insert(0, os.path.join(ROOT, "tests"))
from util import sample_summary  # noqa: E402

HERE = os.path.dirname(os.path.abspath(__file__))

CASES = [
    # name, local, global, shape, d, heads, act, num_graphs, training
    ("gatedgcn_transformer_relu", "CustomGatedGCN", "Transformer", "zinc-gatedgcn", 64, 4, "relu", 6, True),
    ("gatedgcn_transformer_gelu", "CustomGatedGCN", "Transformer", "pcqm4m-small", 48, 4, "gelu", 12, True),
    ("gatedgcn_transformer_hd76", "CustomGatedGCN", "Transformer", "pcqm4m-small", 152, 2, "relu", 8, True),
    ("gine_transformer_relu", "GINE", "Transformer", "zinc-gine", 64, 4, "relu", 6, True),
    ("gatedgcn_none_relu", "CustomGatedGCN", "None", "zinc-gatedgcn", 32, 4, "relu", 5, True),
    ("none_transformer_relu", "None", "Transformer", "zinc-gine", 32, 2, "relu", 5, True),
    ("gine_none_gelu", "GINE", "None", "zinc-gine", 32, 4, "gelu", 5, True),
    ("gatedgcn_transformer_eval", "CustomGatedGCN", "Transformer", "zinc-gatedgcn", 64, 4, "relu", 6, False),
    ("gatedgcn_performer_relu", "CustomGatedGCN", "Performer", "zinc-gatedgcn", 64, 4, "relu", 6, True),
    ("code2_gatedgcn_transformer", "CustomGatedGCN", "Transformer", "code2", 32, 4, "relu", 3, True),
    # GCN: the aggregation is PyG's GCNConv (third party) as restated in oracle/ref_shim.py; the composition is the
    # reference's own gps_layer.py
    ("gcn_transformer_relu", "GCN", "Transformer", "zinc-gine", 64, 4, "relu", 6, True),
    ("gcn_transformer_hd76", "GCN", "Transformer", "pcqm4m-small", 152, 2, "gelu", 8, True),
]


def run_case(ref, name, local, glob, shape, d, heads, act, B, training):
    torch.manual_seed(zlib.crc32(name.encode()) % (2 ** 31))
    layer = ref.GPSLayer(d, local, glob, heads, act=act)
    # non-trivial BatchNorm affine + running stats so they are actually exercised
    with torch.no_grad():
        for m in layer.modules():
            if isinstance(m, torch.nn.BatchNorm1d):
                m.weight.uniform_(0.5, 1.5)
                m.bias.uniform_(-0.3, 0.3)
                m.running_mean.uniform_(-0.2, 0.2)
                m.running_var.uniform_(0.6, 1.4)
        if local == "GCN":
            layer.local_model.bias.uniform_(-0.3, 0.3)   # PyG initialises it to zero
    state = {k: v.clone() for k, v in layer.state_dict().items()}
    batch = make_batch(shape, seed=11, dim=d, num_graphs=B)
    fix = {"config": dict(name=name, local=local, glob=glob, d=d, heads=heads, act=act, training=training),
           "x": batch.x.clone(), "edge_index": batch.edge_index.clone(), "edge_attr": batch.edge_attr.clone(),
           "batch": batch.batch.clone(), "num_graphs": B, "state": state}
    layer = layer.double()
    layer.train(training)
    b = batch.clone()
    b.x = b.x.double().requires_grad_(True)
    b.edge_attr = b.edge_attr.double().requires_grad_(True)
    x_in, e_in = b.x, b.edge_attr
    out = layer(b)
    g = torch.Generator().manual_seed(5)
    ct_x = torch.randn(out.x.shape, generator=g)
    fix["ct_x"] = ct_x
    fix["out_x"] = out.x.detach().float()
    loss = (out.x * ct_x.double()).sum()
    if local == "CustomGatedGCN":
        ct_e = torch.randn(out.edge_attr.shape, generator=g)
        fix["ct_e"] = ct_e
        fix["out_e"] = out.edge_attr.detach().float()
        loss = loss + (out.edge_attr * ct_e.double()).sum()
    if training:
        loss.backward()
        fix["grad_x"] = x_in.grad.float()
        if e_in.grad is not None:
            fix["grad_e"] = e_in.grad.float()
        fix["grad_params"] = {n: p.grad.float() for n, p in layer.named_parameters() if p.grad is not None}
    fix["state_after"] = {k: v.detach().float() if v.is_floating_point() else v.clone()
                          for k, v in layer.state_dict().items() if "running" in k or "num_batches" in k}
    return fix


LIVE_CASES = [("CustomGatedGCN", "Transformer"), ("GINE", "Transformer"), ("CustomGatedGCN", "Performer"),
              ("None", "Transformer"), ("GINE", "None"), ("GCN", "Transformer"), ("GCN", "None")]


def reference_live(ref):
    """The reference layer (fp64) on the oracle's seeded weights: d=32, H=4, 7 ZINC-shaped graphs, loss sum(x_out^2)."""
    out = {}
    for local, glob in LIVE_CASES:
        torch.manual_seed(3)
        state = OracleGPSLayer(32, local, glob, 4).double().state_dict()
        R = ref.GPSLayer(32, local, glob, 4).double()
        R.load_state_dict(state, strict=True)
        b = make_batch("zinc-gatedgcn", seed=5, dim=32, num_graphs=7, dtype=torch.float64)
        inputs = {"x": b.x, "edge_attr": b.edge_attr, "edge_index": b.edge_index, "batch": b.batch}
        b.x.requires_grad_(True)
        b.edge_attr.requires_grad_(True)
        x_in = b.x
        o = R(b)
        (o.x ** 2).sum().backward()
        grads = {n: p.grad for n, p in R.named_parameters() if p.grad is not None}
        out[f"{local}-{glob}"] = {"state": sample_summary(state, 4), "inputs": sample_summary(inputs, 16),
                                  "outputs": sample_summary({"x": o.x}, 256),
                                  "grad_x": sample_summary({"grad_x": x_in.grad}, 256),
                                  "grads": sample_summary(grads, 32)}
    return out


def reference_stack(ref):
    """Three chained reference layers (fp64) on the oracle's seeded weights: d=64, H=4, 24 ZINC-shaped graphs."""
    d, heads, L = 64, 4, 3
    torch.manual_seed(11)
    states = [OracleGPSLayer(d, "CustomGatedGCN", "Transformer", heads).state_dict() for _ in range(L)]
    layers = []
    for st in states:
        R = ref.GPSLayer(d, "CustomGatedGCN", "Transformer", heads)
        R.load_state_dict(st, strict=True)
        layers.append(R.double())
    b = make_batch("zinc-gatedgcn", seed=13, dim=d, num_graphs=24)
    g = torch.Generator().manual_seed(6)
    ct_x, ct_e = torch.randn(b.x.shape, generator=g), torch.randn(b.edge_attr.shape, generator=g)
    inputs = {"x": b.x, "edge_attr": b.edge_attr, "edge_index": b.edge_index, "batch": b.batch, "ct_x": ct_x, "ct_e": ct_e}
    b.x, b.edge_attr = b.x.double().requires_grad_(True), b.edge_attr.double().requires_grad_(True)
    x_in, e_in = b.x, b.edge_attr
    for R in layers:
        b = R(b)
    ((b.x * ct_x.double()).sum() + (b.edge_attr * ct_e.double()).sum()).backward()
    grads = {f"{li}.{n}": p.grad for li, R in enumerate(layers) for n, p in R.named_parameters() if p.grad is not None}
    return {"state": sample_summary({f"{li}.{k}": v for li, st in enumerate(states) for k, v in st.items()}, 4),
            "inputs": sample_summary(inputs, 16),
            "outputs": sample_summary({"x": b.x, "e": b.edge_attr, "gx": x_in.grad, "ge": e_in.grad}, 256),
            "grads": sample_summary(grads, 32)}


def main():
    ref = load_reference("/root/reference/graphgps/layer")
    only = set(sys.argv[1:])   # optional: regenerate just the named fixtures
    for case in CASES:
        if only and case[0] not in only:
            continue
        fix = run_case(ref, *case)
        path = os.path.join(HERE, case[0] + ".pt")
        torch.save(fix, path)
        print(case[0], "N", fix["x"].shape[0], "E", fix["edge_index"].shape[1], f"{os.path.getsize(path)/1e3:.0f} kB")
    os.makedirs(os.path.join(HERE, "reference"), exist_ok=True)
    for name, make in (("oracle_live", reference_live), ("stack3", reference_stack)):
        if only and name not in only:
            continue
        path = os.path.join(HERE, "reference", name + ".pt")
        torch.save(make(ref), path)
        print("reference/" + name, f"{os.path.getsize(path)/1e3:.0f} kB")


if __name__ == "__main__":
    main()
