"""Generates the EquivStableLapPE fixtures from the REFERENCE ITSELF (its own layer files run verbatim under
oracle/ref_shim.py, fp64), as tests/golden/make_golden.py does for the plain layer.

    python tests/golden/make_golden_eslappe.py      # needs the reference's layer files (see oracle/ref_shim.py)

Writes tests/golden/eslappe/<case>.pt (not tests/golden/*.pt: the existing parametrised tests load every file there as
a plain-layer case) and tests/golden/reference/eslappe_live.pt.  Each fixture holds what a make_golden.py fixture holds
plus the batch's pe_EquivStableLapPE (graphgps_b200.batch.add_equivstable_pe, scaled per case so that the default-init
gates spread instead of saturating), its gradient, and the reference layer's state_dict key order.  Every file stays
below 1 MB.
"""
import os
import sys
import zlib

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from graphgps_b200.batch import add_equivstable_pe, make_batch  # noqa: E402
from oracle.ref_shim import load_reference  # noqa: E402
from es_oracle import OracleGPSLayerES  # noqa: E402
from util import sample_summary  # noqa: E402

HERE = os.path.dirname(os.path.abspath(__file__))

# name, local, global, shape, d, heads, act, num_graphs, training, PE scale.  The scale puts the mean r_ij near 8 for
# each shape, where the default-init gates spread (std > 0.03) without saturating; at full scale most sit near 0 or 1.
ES_CASES = [
    ("es_gatedgcn_transformer_relu", "CustomGatedGCN", "Transformer", "zinc-gatedgcn", 64, 4, "relu", 4, True, 3.0),
    ("es_gatedgcn_transformer_gelu", "CustomGatedGCN", "Transformer", "pcqm4m-small", 48, 4, "gelu", 12, True, 3.0),
    ("es_gatedgcn_transformer_hd76", "CustomGatedGCN", "Transformer", "pcqm4m-small", 76, 1, "relu", 4, True, 1.4),
    ("es_gatedgcn_performer_relu", "CustomGatedGCN", "Performer", "zinc-gatedgcn", 48, 2, "relu", 5, True, 2.0),
    ("es_gatedgcn_none_relu", "CustomGatedGCN", "None", "zinc-gatedgcn", 32, 4, "relu", 5, True, 3.0),
    ("es_gatedgcn_transformer_eval", "CustomGatedGCN", "Transformer", "zinc-gatedgcn", 64, 4, "relu", 6, False, 2.0),
]
ES_LIVE_CASES = [("CustomGatedGCN", "Transformer", "relu"), ("CustomGatedGCN", "Transformer", "gelu"),
                 ("CustomGatedGCN", "Performer", "relu"), ("CustomGatedGCN", "None", "relu"), ("GCN", "Transformer", "relu")]
ES_LIVE_PE_SCALE = 3.0


def run_case(ref, name, local, glob, shape, d, heads, act, B, training, pe_scale):
    torch.manual_seed(zlib.crc32(name.encode()) % (2 ** 31))
    layer = ref.GPSLayer(d, local, glob, heads, act=act, equivstable_pe=True)
    with torch.no_grad():   # non-trivial BatchNorm affine + running stats so they are actually exercised
        for m in layer.modules():
            if isinstance(m, torch.nn.BatchNorm1d):
                m.weight.uniform_(0.5, 1.5)
                m.bias.uniform_(-0.3, 0.3)
                m.running_mean.uniform_(-0.2, 0.2)
                m.running_var.uniform_(0.6, 1.4)
    state = {k: v.clone() for k, v in layer.state_dict().items()}
    batch = make_batch(shape, seed=11, dim=d, num_graphs=B)
    add_equivstable_pe(batch, d, seed=12, scale=pe_scale)
    fix = {"config": dict(name=name, local=local, glob=glob, d=d, heads=heads, act=act, training=training,
                          equivstable_pe=True, pe_scale=pe_scale),
           "x": batch.x.clone(), "edge_index": batch.edge_index.clone(), "edge_attr": batch.edge_attr.clone(),
           "batch": batch.batch.clone(), "num_graphs": B, "state": state, "state_keys": list(state.keys()),
           "pe": batch.pe_EquivStableLapPE.clone()}
    layer = layer.double().train(training)
    b = batch.clone()
    b.x = b.x.double().requires_grad_(True)
    b.edge_attr = b.edge_attr.double().requires_grad_(True)
    b.pe_EquivStableLapPE = b.pe_EquivStableLapPE.double().requires_grad_(True)
    x_in, e_in, pe_in = b.x, b.edge_attr, b.pe_EquivStableLapPE
    out = layer(b)
    g = torch.Generator().manual_seed(5)
    ct_x, ct_e = torch.randn(out.x.shape, generator=g), torch.randn(out.edge_attr.shape, generator=g)
    fix.update(ct_x=ct_x, ct_e=ct_e, out_x=out.x.detach().float(), out_e=out.edge_attr.detach().float())
    if training:
        ((out.x * ct_x.double()).sum() + (out.edge_attr * ct_e.double()).sum()).backward()
        fix["grad_x"], fix["grad_e"], fix["grad_pe"] = x_in.grad.float(), e_in.grad.float(), pe_in.grad.float()
        fix["grad_params"] = {n: p.grad.float() for n, p in layer.named_parameters() if p.grad is not None}
    fix["state_after"] = {k: v.detach().float() if v.is_floating_point() else v.clone()
                          for k, v in layer.state_dict().items() if "running" in k or "num_batches" in k}
    return fix


def reference_eslappe_live(ref):
    """The reference layer with equivstable_pe=True (fp64) on the ES oracle's seeded weights: d=32, H=4, 7 ZINC-shaped
    graphs, PE from add_equivstable_pe(seed=6, scale=3), loss = <x_out, ct_x> + <e_out, ct_e> with seeded cotangents
    (with sum(x_out^2) the PE gradient nearly vanishes and would pin nothing)."""
    out = {}
    for local, glob, act in ES_LIVE_CASES:
        torch.manual_seed(3)
        state = OracleGPSLayerES(32, local, glob, 4, act=act).double().state_dict()
        R = ref.GPSLayer(32, local, glob, 4, act=act, equivstable_pe=True).double()
        R.load_state_dict(state, strict=True)
        b = make_batch("zinc-gatedgcn", seed=5, dim=32, num_graphs=7, dtype=torch.float64)
        add_equivstable_pe(b, 32, seed=6, scale=ES_LIVE_PE_SCALE)
        g = torch.Generator().manual_seed(7)
        ct_x, ct_e = torch.randn(b.x.shape, generator=g).double(), torch.randn(b.edge_attr.shape, generator=g).double()
        inputs = {"x": b.x, "edge_attr": b.edge_attr, "edge_index": b.edge_index, "batch": b.batch,
                  "pe": b.pe_EquivStableLapPE}
        for t in (b.x, b.edge_attr, b.pe_EquivStableLapPE):
            t.requires_grad_(True)
        x_in, e_in, pe_in = b.x, b.edge_attr, b.pe_EquivStableLapPE
        o = R(b)
        loss = (o.x * ct_x).sum()
        outs = {"x": o.x}
        if local == "CustomGatedGCN":
            loss = loss + (o.edge_attr * ct_e).sum()
            outs["e"] = o.edge_attr
        loss.backward()
        grads = {n: p.grad for n, p in R.named_parameters() if p.grad is not None}
        gin = {"grad_x": x_in.grad}
        if local == "CustomGatedGCN":
            gin["grad_e"], gin["grad_pe"] = e_in.grad, pe_in.grad
        out[f"{local}-{glob}-{act}"] = {"state": sample_summary(state, 4), "inputs": sample_summary(inputs, 16),
                                        "outputs": sample_summary(outs, 256), "grad_in": sample_summary(gin, 256),
                                        "grads": sample_summary(grads, 32), "state_keys": list(R.state_dict().keys())}
    return out


def main():
    ref = load_reference()
    only = set(sys.argv[1:])   # optional: regenerate just the named fixtures
    os.makedirs(os.path.join(HERE, "eslappe"), exist_ok=True)
    for case in ES_CASES:
        if only and case[0] not in only:
            continue
        fix = run_case(ref, *case)
        path = os.path.join(HERE, "eslappe", case[0] + ".pt")
        torch.save(fix, path)
        print("eslappe/" + case[0], "N", fix["x"].shape[0], "E", fix["edge_index"].shape[1],
              f"{os.path.getsize(path)/1e3:.0f} kB")
    if not only or "eslappe_live" in only:
        path = os.path.join(HERE, "reference", "eslappe_live.pt")
        torch.save(reference_eslappe_live(ref), path)
        print("reference/eslappe_live", f"{os.path.getsize(path)/1e3:.0f} kB")


if __name__ == "__main__":
    main()
