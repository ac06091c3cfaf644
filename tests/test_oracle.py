"""CPU: pins the oracle (oracle/gps_oracle.py) against the committed golden fixtures (outputs of the
reference's own layer files, fp64, run under oracle/ref_shim.py by tests/golden/make_golden.py).  Also the
published parameter-count KATs (README.md:77-79)."""
import pytest
import torch

from oracle.gps_oracle import OracleGPSLayer, param_count
from graphgps_b200.batch import make_batch
from util import check_summary, compare, golden_batch, golden_names, load_golden, load_reference_golden, run_layer


@pytest.mark.parametrize("name", golden_names())
def test_oracle_matches_golden_fp64(name):
    fix = load_golden(name)
    cfg = fix["config"]
    layer = OracleGPSLayer(cfg["d"], cfg["local"], cfg["glob"], cfg["heads"], act=cfg["act"])
    layer.load_state_dict(fix["state"], strict=True)
    layer = layer.double().train(cfg["training"])
    res = run_layer(layer, golden_batch(fix, dtype=torch.float64), fix, backward=cfg["training"])
    compare(res, fix, 2e-6, f"oracle fp64 vs golden {name}")   # goldens are stored as fp32


@pytest.mark.parametrize("name", golden_names())
def test_oracle_fp32_close_to_golden(name):
    fix = load_golden(name)
    cfg = fix["config"]
    layer = OracleGPSLayer(cfg["d"], cfg["local"], cfg["glob"], cfg["heads"], act=cfg["act"])
    layer.load_state_dict(fix["state"], strict=True)
    layer.train(cfg["training"])
    res = run_layer(layer, golden_batch(fix), fix, backward=cfg["training"])
    compare(res, fix, 5e-4, f"oracle fp32 vs golden {name}")


@pytest.mark.parametrize("local,glob", [("CustomGatedGCN", "Transformer"), ("GINE", "Transformer"),
                                        ("CustomGatedGCN", "Performer"), ("None", "Transformer"),
                                        ("GINE", "None"), ("GCN", "Transformer"), ("GCN", "None")])
def test_oracle_equals_reference_live(local, glob):
    """The oracle in fp64 against the reference's own layer files run in fp64 on the same seeded weights and batch
    (tests/golden/reference/oracle_live.pt, written by make_golden.py): outputs to 1e-10, gradients to 1e-9."""
    fix = load_reference_golden("oracle_live")[f"{local}-{glob}"]
    torch.manual_seed(3)
    O = OracleGPSLayer(32, local, glob, 4).double()
    b = make_batch("zinc-gatedgcn", seed=5, dim=32, num_graphs=7, dtype=torch.float64)
    check_summary(O.state_dict(), fix["state"], 1e-12, "seeded weights differ from make_golden.py's", scaled=True)
    check_summary({"x": b.x, "edge_attr": b.edge_attr, "edge_index": b.edge_index, "batch": b.batch}, fix["inputs"],
                  1e-12, "seeded batch differs from make_golden.py's", scaled=True)
    b.x.requires_grad_(True)
    b.edge_attr.requires_grad_(True)
    x_in = b.x
    o = O(b)
    (o.x ** 2).sum().backward()
    check_summary({"x": o.x}, fix["outputs"], 1e-10, "oracle vs reference outputs")
    check_summary({"grad_x": x_in.grad}, fix["grad_x"], 1e-9, "oracle vs reference input gradient")
    check_summary({n: p.grad for n, p in O.named_parameters() if p.grad is not None}, fix["grads"], 1e-9,
                  "oracle vs reference parameter gradients")


def test_gcn_restatements_agree_with_self_loops_and_isolated_nodes():
    """GCNConv is third-party (PyG 2.2): the shim's message-passing restatement (gcn_norm +
    add_remaining_self_loops + propagate) and the oracle's dense one must agree, including on graphs with
    explicit self-loop edges (replaced by the single unit loop), duplicate edges and isolated nodes."""
    from oracle.gps_oracle import OracleGCN
    from oracle.ref_shim import _GCNConv
    torch.manual_seed(0)
    N, d = 9, 8
    ei = torch.tensor([[0, 1, 1, 2, 2, 3, 3, 3, 5, 6, 6, 0], [1, 0, 1, 2, 3, 2, 3, 4, 5, 7, 7, 1]])  # loops at 1,2,3,5; dup 6->7, 0->1
    A, B = _GCNConv(d, d).double(), OracleGCN(d).double()
    with torch.no_grad():
        A.bias.uniform_(-1, 1)
    B.load_state_dict(A.state_dict(), strict=True)
    x1 = torch.randn(N, d, dtype=torch.float64, requires_grad=True)
    x2 = x1.detach().clone().requires_grad_(True)
    y1, y2 = A(x1, ei), B(x2, ei)
    assert (y1 - y2).abs().max() < 1e-12
    (y1 ** 2).sum().backward()
    (y2 ** 2).sum().backward()
    assert (x1.grad - x2.grad).abs().max() < 1e-12
    assert (A.lin.weight.grad - B.lin.weight.grad).abs().max() < 1e-12
    # node 8 is isolated: deg = 1 -> h = x W^T + b
    assert (y2[8] - (B.lin(x2[8]) + B.bias)).abs().max() < 1e-12


def test_parameter_count_kats():
    """Published totals pin the layer's tensor shapes (SURVEY.md section 4): per-layer counts
    13d^2+22d (GatedGCN+Transformer), 10d^2+15d (GINE+Transformer)."""
    for d, h in ((304, 4), (384, 16), (256, 8)):
        assert param_count(OracleGPSLayer(d, "CustomGatedGCN", "Transformer", h)) == 13 * d * d + 22 * d
    assert param_count(OracleGPSLayer(64, "GINE", "Transformer", 4)) == 10 * 64 * 64 + 15 * 64
    # GatedGCN+Performer at d=256, H=4: inner = 64*4 = 256 -> 13d^2+19d (no q/k/v biases)
    assert param_count(OracleGPSLayer(256, "CustomGatedGCN", "Performer", 4)) == 13 * 256 * 256 + 19 * 256
    # GPS-small body: 5 layers of d=304 = 6,040,480 of the published 6,152,001 (rest: encoders + head)
    assert 5 * (13 * 304 * 304 + 22 * 304) == 6040480
