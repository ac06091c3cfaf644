"""CPU: EquivStableLapPE (GPSLayer(..., equivstable_pe=True)).  Pins the oracle's gated GatedGCN against the
reference's own layer files (tests/golden/reference/eslappe_live.pt) and the ES fixtures (tests/golden/eslappe/, written by tests/golden/make_golden_eslappe.py),
checks the drop-in's state_dict against the reference's key order, and the constructor contract."""
import pytest
import torch

import graphgps_b200
from graphgps_b200.batch import add_equivstable_pe, make_batch
from es_oracle import OracleGPSLayerES
from es_util import es_batch, es_golden_names, es_l2_errors, load_es_golden, run_es_layer
from util import check_summary, compare, load_reference_golden

LIVE = [("CustomGatedGCN", "Transformer", "relu"), ("CustomGatedGCN", "Transformer", "gelu"),
        ("CustomGatedGCN", "Performer", "relu"), ("CustomGatedGCN", "None", "relu"), ("GCN", "Transformer", "relu")]


def _oracle(fix):
    cfg = fix["config"]
    layer = OracleGPSLayerES(cfg["d"], cfg["local"], cfg["glob"], cfg["heads"], act=cfg["act"])
    layer.load_state_dict(fix["state"], strict=True)
    return layer


def test_es_fixtures_exist():
    assert len(es_golden_names()) >= 6


@pytest.mark.parametrize("local,glob,act", LIVE)
def test_oracle_equals_reference_live_es(local, glob, act):
    """Oracle fp64 vs the reference's layer files in fp64 on the same seeded weights, batch, PE and cotangents:
    outputs to 1e-10, gradients (PE gradient included) to 1e-9."""
    fix = load_reference_golden("eslappe_live")[f"{local}-{glob}-{act}"]
    torch.manual_seed(3)
    O = OracleGPSLayerES(32, local, glob, 4, act=act).double()
    b = make_batch("zinc-gatedgcn", seed=5, dim=32, num_graphs=7, dtype=torch.float64)
    add_equivstable_pe(b, 32, seed=6, scale=3.0)
    g = torch.Generator().manual_seed(7)
    ct_x, ct_e = torch.randn(b.x.shape, generator=g).double(), torch.randn(b.edge_attr.shape, generator=g).double()
    check_summary(O.state_dict(), fix["state"], 1e-12, "seeded weights differ from make_golden.py's", scaled=True)
    check_summary({"x": b.x, "edge_attr": b.edge_attr, "edge_index": b.edge_index, "batch": b.batch,
                   "pe": b.pe_EquivStableLapPE}, fix["inputs"], 1e-12, "seeded batch differs from make_golden.py's",
                  scaled=True)
    assert sorted(O.state_dict().keys()) == sorted(fix["state_keys"])
    for t in (b.x, b.edge_attr, b.pe_EquivStableLapPE):
        t.requires_grad_(True)
    x_in, e_in, pe_in = b.x, b.edge_attr, b.pe_EquivStableLapPE
    o = O(b)
    loss = (o.x * ct_x).sum()
    outs = {"x": o.x}
    if local == "CustomGatedGCN":
        loss = loss + (o.edge_attr * ct_e).sum()
        outs["e"] = o.edge_attr
    loss.backward()
    check_summary(outs, fix["outputs"], 1e-10, "oracle vs reference outputs")
    gin = {"grad_x": x_in.grad}
    if local == "CustomGatedGCN":
        gin["grad_e"], gin["grad_pe"] = e_in.grad, pe_in.grad
        assert float(pe_in.grad.abs().max()) > 1e-3   # the cotangents exercise the gate's gradient
    check_summary(gin, fix["grad_in"], 1e-9, "oracle vs reference input gradients")
    check_summary({n: p.grad for n, p in O.named_parameters() if p.grad is not None}, fix["grads"], 1e-9,
                  "oracle vs reference parameter gradients")


@pytest.mark.parametrize("name", es_golden_names())
def test_oracle_matches_es_golden_fp64(name):
    fix = load_es_golden(name)
    cfg = fix["config"]
    layer = _oracle(fix).double().train(cfg["training"])
    res = run_es_layer(layer, es_batch(fix, dtype=torch.float64), fix, backward=cfg["training"])
    compare(res, fix, 2e-6, f"oracle fp64 vs ES golden {name}")
    if cfg["training"]:
        errs = es_l2_errors(res, fix)
        assert max(errs.values()) < 1e-6, errs


@pytest.mark.parametrize("name", es_golden_names())
def test_oracle_fp32_close_to_es_golden(name):
    fix = load_es_golden(name)
    cfg = fix["config"]
    layer = _oracle(fix).train(cfg["training"])
    res = run_es_layer(layer, es_batch(fix), fix, backward=cfg["training"])
    compare(res, fix, 5e-4, f"oracle fp32 vs ES golden {name}")
    if cfg["training"]:
        errs = es_l2_errors(res, fix)
        assert max(errs.values()) < 1e-3, errs


@pytest.mark.parametrize("name", es_golden_names())
def test_es_golden_gates_spread(name):
    """The fixtures' PE (scaled per case in make_golden.py) keeps the default-init gates away from saturation, so their gradient paths are
    exercised: std(gate) > 0.03 and at most 1 % of the edges above 0.999."""
    fix = load_es_golden(name)
    layer = _oracle(fix).double()
    pe = fix["pe"].double()
    src, dst = fix["edge_index"]
    with torch.no_grad():
        gate = layer.local_model.mlp_r_ij(((pe[dst] - pe[src]) ** 2).sum(-1, keepdim=True)).squeeze(1)
    assert float(gate.std()) > 0.03 and float((gate > 0.999).double().mean()) <= 0.01, (float(gate.std()),
                                                                                        float(gate.max()))


@pytest.mark.parametrize("name", es_golden_names())
def test_state_dict_keys_order_and_shapes_match_reference(name):
    fix = load_es_golden(name)
    cfg = fix["config"]
    ours = graphgps_b200.GPSLayer(cfg["d"], cfg["local"], cfg["glob"], cfg["heads"], act=cfg["act"],
                                  equivstable_pe=True)
    sd = ours.state_dict()
    assert list(sd.keys()) == fix["state_keys"]
    for k in sd:
        assert tuple(sd[k].shape) == tuple(fix["state"][k].shape), k
    ours.load_state_dict(fix["state"], strict=True)
    assert tuple(ours.local_model.mlp_r_ij[0].weight.shape) == (cfg["d"], 1)
    assert tuple(ours.local_model.mlp_r_ij[2].weight.shape) == (1, cfg["d"])


def test_constructor_equivstable_pe():
    G = graphgps_b200.GPSLayer
    es = G(64, "CustomGatedGCN", "Transformer", 4, equivstable_pe=True)
    assert "local_model.mlp_r_ij.0.weight" in es.state_dict()
    gcn = G(64, "GCN", "Transformer", 4, equivstable_pe=True)          # accepted and not read, as in the reference
    assert set(gcn.state_dict()) == set(G(64, "GCN", "Transformer", 4).state_dict())
    G(64, "None", "Transformer", 4, equivstable_pe=True)
    with pytest.raises(NotImplementedError, match="GINEConvESLapPE"):
        G(64, "GINE", "Transformer", 4, equivstable_pe=True)
    # the plain layer keeps its parameter list
    assert not any("mlp_r_ij" in k for k in G(64, "CustomGatedGCN", "Transformer", 4).state_dict())


def test_missing_pe_raises_before_any_device_work():
    layer = graphgps_b200.GPSLayer(32, "CustomGatedGCN", "Transformer", 4, equivstable_pe=True)
    b = make_batch("zinc-gatedgcn", dim=32, num_graphs=2)
    with pytest.raises(RuntimeError, match="no CPU fallback"):   # CPU tensors are refused first
        layer(b)


def test_add_equivstable_pe_leaves_batch_unchanged():
    a = make_batch("zinc-gatedgcn", seed=3, dim=16, num_graphs=4)
    b = make_batch("zinc-gatedgcn", seed=3, dim=16, num_graphs=4)
    add_equivstable_pe(b, seed=1)
    assert torch.equal(a.x, b.x) and torch.equal(a.edge_attr, b.edge_attr)
    pe = b.pe_EquivStableLapPE
    assert pe.shape == (b.num_nodes, 16) and pe.dtype == torch.float32
    assert torch.equal(pe, add_equivstable_pe(make_batch("zinc-gatedgcn", seed=3, dim=16, num_graphs=4), seed=1)
                       .pe_EquivStableLapPE)


def test_graphgym_register_passes_equivstable_pe(monkeypatch):
    import sys
    import types
    from graphgps_b200 import graphgym

    registry = {}
    ns = types.SimpleNamespace
    cfg = ns(gt=ns(layer_type="CustomGatedGCN+Transformer", n_heads=4, dropout=0.0, attn_dropout=0.5,
                   layer_norm=False, batch_norm=True), gnn=ns(act="relu"), posenc_EquivStableLapPE=ns(enable=True))
    for name, attrs in (("torch_geometric", {}), ("torch_geometric.graphgym", {}),
                        ("torch_geometric.graphgym.register",
                         {"register_layer": lambda k, m=None: registry.setdefault(k, m)}),
                        ("torch_geometric.graphgym.config", {"cfg": cfg})):
        m = types.ModuleType(name)
        m.__dict__.update(attrs)
        monkeypatch.setitem(sys.modules, name, m)
    cls = graphgym.register("gpslayer_b200_es")
    layer = cls(ns(dim_out=32))
    assert layer.equivstable_pe and "local_model.mlp_r_ij.2.bias" in layer.state_dict()
