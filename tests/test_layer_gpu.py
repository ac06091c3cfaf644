"""GPU parity tests (run on the B200 box): the CUDA path, called through the C ABI, against
(i) the committed golden fixtures (reference-verbatim, fp64), (ii) the oracle on the same seeded
inputs, (iii) torch restatements of single stages, and (iv) size-independent properties at the
BASELINE sizes.  Tolerances: 1e-3 for precision="fp32", 1e-2 for "bf16" (BASELINE.json north_star),
measured as max|a-b| / max(1, max|b|) on BatchNorm-normalised outputs."""
import ctypes as C

import pytest
import torch

import graphgps_b200
from graphgps_b200 import _lib
from graphgps_b200.batch import batch_from_lists, make_batch
from graphgps_b200.graph import GraphStructure, graph_of
from oracle.gps_oracle import OracleGPSLayer
from util import (check_summary, compare, golden_batch, golden_names, load_golden, load_reference_golden, rel_err,
                  rel_l2, run_layer)

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
TOL = {"fp32": 1e-3, "bf16": 1e-2}
# Gradient fallback criterion (util.compare): relative L2 when ReLU-kink flips defeat the max-abs one.
# bf16 rounding (2^-9 per product operand, ~12 chained single-pass products between the loss and the first weight
# gradient) also flips ~0.3% of the ReLU masks.  Round 1 allowed 15% everywhere, which could hide a defect; measured on
# B200 (round 2): weight gradients 3.5-4.3e-2 relative L2 at the BASELINE sizes and up to 9e-2 on the small golden
# batches (120-300 rows per BatchNorm column); the near-cancelling column sums (bias / BatchNorm-bias gradients) up to
# 7.2e-2 (local_model.bn_node_x.bias).  Bounds: 8e-2 at the BASELINE sizes (GRAD_L2_FULL), 1e-1 on the goldens; the bias gradients are
# exact fp32 column sums in both modes.  A wrong operand or a missing term shows up as O(1).  Smooth-activation
# (GELU) cases are held to the strict max-abs tolerance in test_layer_gelu_strict_gradients_full_size.
# util.compare reports raw max-abs errors beside the scaled ones.
GRAD_L2 = {"fp32": 5e-3, "bf16": 1e-1}
GRAD_L2_FULL = {"fp32": 5e-3, "bf16": 8e-2}   # BASELINE-size batches (thousands of rows per BatchNorm column)


def _stream():
    return torch.cuda.current_stream().cuda_stream


# ------------------------------------------------------------------------------- graph structure
@pytest.mark.parametrize("shape,B", [("pcqm4m-small", 64), ("code2", 8), ("zinc-gine", 1)])
def test_graph_build_matches_sort(shape, B):
    b = make_batch(shape, seed=1, dim=8, num_graphs=B).to(DEV)
    gs = GraphStructure(b.edge_index, b.batch, B)
    torch.cuda.synchronize()
    src, dst = b.edge_index[0].cpu(), b.edge_index[1].cpu()
    E, N = src.numel(), b.num_nodes
    order = torch.argsort(dst * E + torch.arange(E), stable=True)     # by dst, ties by edge id
    assert torch.equal(gs.dst_eid.cpu().long(), order)
    assert torch.equal(gs.dst_src.cpu().long(), src[order])
    assert torch.equal(gs.dst_ptr.cpu().long(), torch.cat([torch.zeros(1, dtype=torch.long),
                                                           torch.bincount(dst, minlength=N).cumsum(0)]))
    order_s = torch.argsort(src * E + torch.arange(E), stable=True)
    assert torch.equal(gs.src_eid.cpu().long(), order_s)
    assert torch.equal(gs.src_dst.cpu().long(), dst[order_s])
    assert torch.equal(gs.graph_ptr.cpu().long(), b.ptr.cpu())


def test_graph_build_empty_graphs_and_no_edges():
    b = batch_from_lists([3, 0, 2, 0], [[(0, 1), (1, 0), (2, 2)], [], [], []], d=8).to(DEV)
    gs = GraphStructure(b.edge_index, b.batch, 4)
    assert gs.graph_ptr.cpu().tolist() == [0, 3, 3, 5, 5]
    assert gs.dst_ptr.cpu().tolist() == [0, 1, 2, 3, 3, 3]


# ------------------------------------------------------------------------------- single stages
@pytest.mark.parametrize("M,N,K", [(3620, 2128, 304), (7455, 304, 304), (130, 64, 64), (1, 4, 4), (333, 608, 304)])
def test_linear_forward(M, N, K):
    lib = _lib.load()
    g = torch.Generator(device="cpu").manual_seed(0)
    A = torch.randn(M, K, generator=g).to(DEV)
    W = (torch.randn(N, K, generator=g) / K ** 0.5).to(DEV)
    bias = torch.randn(N, generator=g).to(DEV)
    Cc = torch.empty(M, N, device=DEV)
    rc = lib.gps_linear_forward(A.data_ptr(), K, W.data_ptr(), K, bias.data_ptr(), Cc.data_ptr(), N, M, N, K, -1, 0,
                                _stream())
    _lib.check(rc, "gps_linear_forward")
    ref = (A.double() @ W.double().t() + bias.double()).float()
    assert rel_err(Cc.cpu(), ref.cpu()) < 1e-4


@pytest.mark.parametrize("shape,d", [("pcqm4m-small", 304), ("zinc-gatedgcn", 64), ("code2", 256)])
def test_gatedgcn_aggregate_forward(shape, d):
    lib = _lib.load()
    b = make_batch(shape, seed=2, dim=d, num_graphs=16).to(DEV)
    gs = graph_of(b)
    N, E = b.num_nodes, b.num_edges
    Y = torch.randn(N, 4 * d, device=DEV)
    Ce = torch.randn(E, d, device=DEV)
    src, dst = b.edge_index
    Ax, Bx, Dx, Ex = (Y[:, i * d:(i + 1) * d].double() for i in range(4))
    e_ij = Dx[dst] + Ex[src] + Ce.double()
    sig = torch.sigmoid(e_ij)
    num = torch.zeros(N, d, device=DEV, dtype=torch.float64).index_add_(0, dst, sig * Bx[src])
    den = torch.zeros(N, d, device=DEV, dtype=torch.float64).index_add_(0, dst, sig)
    xt_ref = Ax + num / (den + 1e-6)
    xt = torch.empty(N, d, device=DEV)
    sx = torch.zeros(2, d, device=DEV, dtype=torch.float64)
    se = torch.zeros(2, d, device=DEV, dtype=torch.float64)
    rc = lib.gps_gatedgcn_aggregate_forward(C.byref(gs.desc), d, Y.data_ptr(), Y.data_ptr() + 4 * d,
                                            Y.data_ptr() + 8 * d, Y.data_ptr() + 12 * d, 4 * d, Ce.data_ptr(),
                                            xt.data_ptr(), sx.data_ptr(), se.data_ptr(), _stream())
    _lib.check(rc, "gatedgcn_aggregate")
    assert rel_err(xt.cpu(), xt_ref.cpu()) < 2e-5
    assert rel_err(Ce.cpu(), e_ij.cpu()) < 1e-5
    assert rel_err(sx[0].cpu(), xt_ref.sum(0).cpu()) < 1e-4 and rel_err(sx[1].cpu(), (xt_ref ** 2).sum(0).cpu()) < 1e-4
    assert rel_err(se[0].cpu(), e_ij.sum(0).cpu()) < 1e-4 and rel_err(se[1].cpu(), (e_ij ** 2).sum(0).cpu()) < 1e-4


def _dense_attention_ref(Q, K, V, ptr, H):
    outs = []
    N, D = Q.shape
    hd = D // H
    for g in range(len(ptr) - 1):
        s, e = int(ptr[g]), int(ptr[g + 1])
        if e == s:
            continue
        q = Q[s:e].view(e - s, H, hd).transpose(0, 1)
        k = K[s:e].view(e - s, H, hd).transpose(0, 1)
        v = V[s:e].view(e - s, H, hd).transpose(0, 1)
        p = torch.softmax(q @ k.transpose(1, 2) / hd ** 0.5, dim=-1)
        outs.append((p @ v).transpose(0, 1).reshape(e - s, D))
    return torch.cat(outs)


@pytest.mark.parametrize("shape,H,hd,B", [("pcqm4m-small", 4, 76, 32), ("zinc-gatedgcn", 4, 16, 8),
                                          ("pcqm4m-small", 16, 24, 16), ("code2", 4, 64, 6)])
def test_attention_forward_backward(shape, H, hd, B):
    lib = _lib.load()
    D = H * hd
    b = make_batch(shape, seed=4, dim=8, num_graphs=B).to(DEV)
    gs = graph_of(b)
    N = b.num_nodes
    QKV = torch.randn(N, 3 * D, device=DEV)
    O = torch.empty(N, D, device=DEV)
    lse = torch.empty(N, H, device=DEV)
    base = QKV.data_ptr()
    rc = lib.gps_attention_forward(C.byref(gs.desc), H, hd, base, base + 4 * D, base + 8 * D, 3 * D, O.data_ptr(), D,
                                   lse.data_ptr(), 0.0, 0, 0, _stream())
    _lib.check(rc, "attention_forward")
    q = QKV[:, :D].double().requires_grad_(True)
    k = QKV[:, D:2 * D].double().requires_grad_(True)
    v = QKV[:, 2 * D:].double().requires_grad_(True)
    ref = _dense_attention_ref(q, k, v, b.ptr, H)
    assert rel_err(O.cpu(), ref.detach().cpu()) < 2e-5
    dO = torch.randn(N, D, device=DEV)
    ref.backward(dO.double())
    dQKV = torch.empty(N, 3 * D, device=DEV)
    delta = torch.empty(N, H, device=DEV)
    gb = dQKV.data_ptr()
    rc = lib.gps_attention_backward(C.byref(gs.desc), H, hd, base, base + 4 * D, base + 8 * D, 3 * D, O.data_ptr(),
                                    dO.data_ptr(), D, lse.data_ptr(), delta.data_ptr(), gb, gb + 4 * D, gb + 8 * D,
                                    3 * D, 0.0, 0, 0, _stream())
    _lib.check(rc, "attention_backward")
    assert rel_err(dQKV[:, :D].cpu(), q.grad.cpu()) < 5e-5
    assert rel_err(dQKV[:, D:2 * D].cpu(), k.grad.cpu()) < 5e-5
    assert rel_err(dQKV[:, 2 * D:].cpu(), v.grad.cpu()) < 5e-5


# ------------------------------------------------------------------------------- whole layer
def _build(cfg, precision="fp32", **kw):
    layer = graphgps_b200.GPSLayer(cfg["d"], cfg["local"], cfg["glob"], cfg["heads"], act=cfg["act"],
                                   precision=precision, **kw)
    return layer


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
@pytest.mark.parametrize("name", golden_names())
def test_layer_matches_golden(name, precision):
    fix = load_golden(name)
    cfg = fix["config"]
    layer = _build(cfg, precision)
    layer.load_state_dict(fix["state"], strict=True)
    layer = layer.to(DEV).train(cfg["training"])
    res = run_layer(layer, golden_batch(fix, DEV), fix, backward=cfg["training"])
    errs = compare(res, fix, TOL[precision], f"CUDA {precision} vs golden {name}", grad_l2_tol=GRAD_L2[precision])
    print(name, precision, "max err", max(errs.values()))


@pytest.mark.parametrize("shape,local,glob,heads", [("pcqm4m-small", "CustomGatedGCN", "Transformer", 4),
                                                    ("zinc-gine", "GINE", "Transformer", 4),
                                                    ("code2", "CustomGatedGCN", "Transformer", 4),
                                                    ("pcqm4m-medium-performer", "CustomGatedGCN", "Performer", 16),
                                                    ("zinc-gatedgcn", "None", "Performer", 4),
                                                    ("code2", "CustomGatedGCN", "Performer", 4),
                                                    ("pcqm4m-small", "GCN", "Transformer", 4),
                                                    ("zinc-gine", "GCN", "Performer", 4)])
def test_layer_matches_oracle_full_size(shape, local, glob, heads):
    _full_size(shape, local, glob, heads, "fp32")


@pytest.mark.parametrize("shape,local,glob,heads", [("pcqm4m-medium-performer", "CustomGatedGCN", "Performer", 16),
                                                    ("pcqm4m-small", "CustomGatedGCN", "Transformer", 4),
                                                    ("code2", "CustomGatedGCN", "Transformer", 4)])
def test_layer_matches_oracle_full_size_bf16(shape, local, glob, heads):
    """BASELINE's stated C4 mode (Performer d=384 H=16, bf16) and the C3 / C5 shapes in bf16: 1e-2 forward."""
    _full_size(shape, local, glob, heads, "bf16")


def _full_size(shape, local, glob, heads, precision):
    """BASELINE-size batch: CUDA layer vs the oracle on the same seeded inputs and weights.

    Forward outputs: 1e-3 max-abs against the fp64 and the fp32 oracle.  Gradients: 1e-3 max-abs or,
    failing that, 5e-3 relative L2 (util.compare) — at ~2M hidden units a single ReLU-kink flip
    between two correct arithmetics moves a weight-gradient entry by more than 1e-3; the reference's
    own fp32 run differs from its fp64 run by 1.8e-2 on ff_linear1.weight at the code2 shape."""
    import copy
    spec = graphgps_b200.SHAPES[shape]
    torch.manual_seed(0)
    ora = OracleGPSLayer(spec.dim, local, glob, heads)
    ours = graphgps_b200.GPSLayer(spec.dim, local, glob, heads, precision=precision)
    ours.load_state_dict(ora.state_dict())
    ours = ours.to(DEV)
    b = make_batch(shape, seed=7)
    g = torch.Generator().manual_seed(9)
    fix = {"config": dict(local=local), "ct_x": torch.randn(b.x.shape, generator=g),
           "ct_e": torch.randn(b.edge_attr.shape, generator=g)}
    ref64 = run_layer(copy.deepcopy(ora).double(), _to(b.clone(), "cpu", torch.float64), fix)
    res = run_layer(ours, b.clone().to(DEV), fix)
    if precision == "bf16":
        t = {k: ref64[k] for k in ("out_x", "out_e", "grad_x", "grad_e") if k in ref64}
        t["grad_params"], t["state_after"] = ref64["grad_params"], ref64["state_after"]
        errs = compare(res, t, TOL["bf16"], f"CUDA bf16 vs oracle fp64 @ {shape}", grad_l2_tol=GRAD_L2_FULL["bf16"])
        print(shape, "bf16", {k: f"{v:.2e}" for k, v in errs.items() if k.startswith(("out", "raw:out"))})
        return
    ref32 = run_layer(ora, b.clone(), fix)

    def target(ref):
        t = {k: ref[k] for k in ("out_x", "out_e", "grad_x", "grad_e") if k in ref}
        t["grad_params"], t["state_after"] = ref["grad_params"], ref["state_after"]
        return t
    # forward vs fp64 oracle at 1e-3; gradients: 1e-3 max-abs or 5e-3 relative-L2 (ReLU-kink flips)
    compare(res, target(ref64), 1e-3, f"CUDA fp32 vs oracle fp64 @ {shape}", grad_l2_tol=5e-3)
    compare(res, target(ref32), 1e-3, f"CUDA fp32 vs oracle fp32 @ {shape}", grad_l2_tol=5e-3)


def _to(b, dev, dt):
    b.x, b.edge_attr = b.x.to(dev, dt), b.edge_attr.to(dev, dt)
    return b


def test_edge_order_invariance_full_size():
    """Property: permuting the edge list permutes edge outputs and leaves node outputs unchanged."""
    torch.manual_seed(1)
    layer = graphgps_b200.GPSLayer(304, "CustomGatedGCN", "Transformer", 4).to(DEV).eval()
    b = make_batch("pcqm4m-small", seed=3).to(DEV)
    perm = torch.randperm(b.num_edges, device=DEV)
    b2 = graphgps_b200.GraphBatch(x=b.x.clone(), edge_index=b.edge_index[:, perm].contiguous(),
                                  edge_attr=b.edge_attr[perm].contiguous(), batch=b.batch, num_graphs=b.num_graphs)
    with torch.no_grad():
        o1 = layer(b.clone())
        o2 = layer(b2)
    assert rel_err(o2.x.cpu(), o1.x.cpu()) < 1e-5
    assert rel_err(o2.edge_attr.cpu(), o1.edge_attr[perm].cpu()) < 1e-5


def test_graphs_are_independent_in_eval_mode():
    """Property: with running statistics (eval) a graph's output does not depend on its batch mates —
    i.e. the per-graph mask of the attention is applied (no leakage across graphs), at BASELINE size."""
    torch.manual_seed(2)
    layer = graphgps_b200.GPSLayer(304, "CustomGatedGCN", "Transformer", 4).to(DEV).eval()
    big = make_batch("pcqm4m-small", seed=5)
    n0, n1 = int(big.ptr[10]), int(big.ptr[11])
    emask = (big.edge_index[0] >= n0) & (big.edge_index[0] < n1)
    single = graphgps_b200.GraphBatch(x=big.x[n0:n1].clone(), edge_index=big.edge_index[:, emask] - n0,
                                      edge_attr=big.edge_attr[emask].clone(),
                                      batch=torch.zeros(n1 - n0, dtype=torch.int64), num_graphs=1)
    with torch.no_grad():
        ob = layer(big.clone().to(DEV))
        os_ = layer(single.to(DEV))
    assert rel_err(os_.x.cpu(), ob.x[n0:n1].cpu()) < 1e-4
    assert rel_err(os_.edge_attr.cpu(), ob.edge_attr[emask.to(DEV)].cpu()) < 1e-4


def test_empty_graphs_isolated_nodes_and_no_edges():
    torch.manual_seed(3)
    d = 32
    b = batch_from_lists([4, 0, 1, 3], [[(0, 1), (1, 0), (2, 1)], [], [], []], d=d)
    ora = OracleGPSLayer(d, "CustomGatedGCN", "Transformer", 4)
    ours = graphgps_b200.GPSLayer(d, "CustomGatedGCN", "Transformer", 4)
    ours.load_state_dict(ora.state_dict())
    ours = ours.to(DEV)
    g = torch.Generator().manual_seed(1)
    fix = {"config": dict(local="CustomGatedGCN"), "ct_x": torch.randn(b.x.shape, generator=g),
           "ct_e": torch.randn(b.edge_attr.shape, generator=g)}
    ref = run_layer(ora.double(), _to(b.clone(), "cpu", torch.float64), fix)
    res = run_layer(ours, b.clone().to(DEV), fix)
    tgt = {k: ref[k] for k in ("out_x", "out_e", "grad_x", "grad_e")}
    tgt["grad_params"], tgt["state_after"] = ref["grad_params"], ref["state_after"]
    compare(res, tgt, 1e-3, "edge cases", grad_l2_tol=5e-3)


def test_gcn_self_loops_duplicates_isolated_nodes_and_dropout_consistency():
    """GCN local model (gps_layer.py:49-51): explicit self-loop edges are replaced by the single unit loop
    (add_remaining_self_loops), duplicate edges count twice, isolated nodes and an empty graph are handled; then,
    with dropout on and the Philox offset pinned, backward equals a finite difference of forward (GELU)."""
    torch.manual_seed(4)
    d = 32
    b = batch_from_lists([5, 0, 1, 4], [[(0, 1), (1, 0), (1, 1), (2, 2), (2, 3), (3, 2), (0, 1)], [], [], [(0, 1), (3, 3)]], d=d)
    ora = OracleGPSLayer(d, "GCN", "Transformer", 4)
    with torch.no_grad():
        ora.local_model.bias.uniform_(-0.5, 0.5)
    ours = graphgps_b200.GPSLayer(d, "GCN", "Transformer", 4)
    ours.load_state_dict(ora.state_dict(), strict=True)
    ours = ours.to(DEV)
    g = torch.Generator().manual_seed(1)
    fix = {"config": dict(local="GCN"), "ct_x": torch.randn(b.x.shape, generator=g)}
    ref = run_layer(ora.double(), _to(b.clone(), "cpu", torch.float64), fix)
    res = run_layer(ours, b.clone().to(DEV), fix)
    tgt = {k: ref[k] for k in ("out_x", "grad_x")}
    tgt["grad_params"], tgt["state_after"] = ref["grad_params"], ref["state_after"]
    compare(res, tgt, 1e-3, "GCN edge cases", grad_l2_tol=5e-3)

    layer = graphgps_b200.GPSLayer(64, "GCN", "Transformer", 4, act="gelu", dropout=0.2, attn_dropout=0.0).to(DEV).train()
    bb = make_batch("zinc-gine", seed=3, dim=64, num_graphs=12).to(DEV)
    ct = torch.randn(bb.x.shape, generator=g).to(DEV)
    vx = torch.randn(bb.x.shape, generator=g).to(DEV)

    def f(x):
        _set_dropout_counter(11 * 4096)
        out = layer(graphgps_b200.GraphBatch(x=x, edge_index=bb.edge_index, edge_attr=bb.edge_attr, batch=bb.batch,
                                             num_graphs=bb.num_graphs))
        return (out.x * ct).sum()

    x0 = bb.x.clone().requires_grad_(True)
    f(x0).backward()
    analytic = float((x0.grad * vx).sum())
    with torch.no_grad():
        numeric = float((f(bb.x + 1e-2 * vx) - f(bb.x - 1e-2 * vx)) / 2e-2)
    assert abs(numeric - analytic) <= 3e-2 * max(1.0, abs(analytic)), (numeric, analytic)


def test_running_stats_and_eval_after_train():
    fix = load_golden("gatedgcn_transformer_relu")
    cfg = fix["config"]
    ours = _build(cfg).to(DEV)
    ours.load_state_dict(fix["state"])
    ora = OracleGPSLayer(cfg["d"], cfg["local"], cfg["glob"], cfg["heads"])
    ora.load_state_dict(fix["state"])
    for _ in range(2):
        ours(golden_batch(fix, DEV))
        ora(golden_batch(fix))
    ours.eval(), ora.eval()
    with torch.no_grad():
        a = ours(golden_batch(fix, DEV))
        r = ora(golden_batch(fix))
    assert rel_err(a.x.cpu(), r.x) < 1e-3 and rel_err(a.edge_attr.cpu(), r.edge_attr) < 1e-3
    assert int(ours.norm2.num_batches_tracked) == int(ora.norm2.num_batches_tracked) == 2


@pytest.mark.parametrize("precision,tol", [("fp32", 1e-3), ("bf16", 3e-2)])
def test_layer_gelu_strict_gradients_full_size(precision, tol):
    """Smooth activation (GELU, 8 shipped configs) => no kink flips: every output AND gradient must meet
    the max-abs tolerance with no L2 fallback, at the PCQM4M BASELINE size, against the fp64 oracle.
    (bf16: 1e-2 on the forward outputs as BASELINE states; 3e-2 on gradients.)"""
    import copy
    spec = graphgps_b200.SHAPES["pcqm4m-small"]
    torch.manual_seed(0)
    ora = OracleGPSLayer(spec.dim, "CustomGatedGCN", "Transformer", 4, act="gelu")
    ours = graphgps_b200.GPSLayer(spec.dim, "CustomGatedGCN", "Transformer", 4, act="gelu", precision=precision)
    ours.load_state_dict(ora.state_dict())
    ours = ours.to(DEV)
    b = make_batch("pcqm4m-small", seed=21)
    g = torch.Generator().manual_seed(9)
    fix = {"config": dict(local="CustomGatedGCN"), "ct_x": torch.randn(b.x.shape, generator=g),
           "ct_e": torch.randn(b.edge_attr.shape, generator=g)}
    ref = run_layer(copy.deepcopy(ora).double(), _to(b.clone(), "cpu", torch.float64), fix)
    res = run_layer(ours, b.clone().to(DEV), fix)
    fwd_tol = 1e-3 if precision == "fp32" else 1e-2
    for k in ("out_x", "out_e"):
        assert rel_err(res[k], ref[k]) < fwd_tol, (k, rel_err(res[k], ref[k]))
    tgt = {k: ref[k] for k in ("grad_x", "grad_e")}
    tgt["grad_params"], tgt["state_after"] = ref["grad_params"], ref["state_after"]
    errs = compare(res, tgt, tol, f"CUDA {precision} GELU strict")
    print("gelu strict", precision, "max err", max(errs.values()))


# ------------------------------------------------------------------------------- dropout
def test_dropout_mask_keep_rate_and_determinism():
    lib = _lib.load()
    m1 = torch.empty(512, 304, device=DEV)
    m2 = torch.empty(512, 304, device=DEV)
    for p in (0.1, 0.5):
        _lib.check(lib.gps_dropout_mask(m1.data_ptr(), 512, 304, p, 1234, 4096, 5, _stream()), "mask")
        _lib.check(lib.gps_dropout_mask(m2.data_ptr(), 512, 304, p, 1234, 4096, 5, _stream()), "mask")
        assert torch.equal(m1, m2)
        assert abs(float(m1.mean()) - (1 - p)) < 0.01
        _lib.check(lib.gps_dropout_mask(m2.data_ptr(), 512, 304, p, 1234, 8192, 5, _stream()), "mask")
        assert not torch.equal(m1, m2)


def _set_dropout_counter(value):
    from graphgps_b200 import gps_layer
    dev = torch.device(DEV)
    ctr = gps_layer._drop_counters.get(dev)
    if ctr is None:
        ctr = torch.zeros(1, dtype=torch.int64, device=dev)
        gps_layer._drop_counters[dev] = ctr
    ctr.fill_(value)


def test_dropout_forward_backward_consistent():
    """With the Philox offset pinned, the dropout layer is a deterministic smooth (GELU) function: its
    backward must equal a central finite difference of its forward along a random direction, i.e. the
    forward and backward passes regenerate the same masks at every dropout site (GatedGCN, attention
    probabilities, attention output, both FFN sites)."""
    torch.manual_seed(5)
    d = 64
    layer = graphgps_b200.GPSLayer(d, "CustomGatedGCN", "Transformer", 4, act="gelu", dropout=0.2,
                                   attn_dropout=0.3).to(DEV).train()
    b = make_batch("zinc-gatedgcn", seed=3, dim=d, num_graphs=12).to(DEV)
    g = torch.Generator().manual_seed(2)
    ct_x = torch.randn(b.x.shape, generator=g).to(DEV)
    ct_e = torch.randn(b.edge_attr.shape, generator=g).to(DEV)
    vx = torch.randn(b.x.shape, generator=g).to(DEV)

    def f(x):
        _set_dropout_counter(7 * 4096)
        bb = graphgps_b200.GraphBatch(x=x, edge_index=b.edge_index, edge_attr=b.edge_attr.clone(), batch=b.batch,
                                      num_graphs=b.num_graphs)
        out = layer(bb)
        return (out.x * ct_x).sum() + (out.edge_attr * ct_e).sum(), out

    x0 = b.x.clone().requires_grad_(True)
    loss, out0 = f(x0)
    loss.backward()
    analytic = float((x0.grad * vx).sum())
    eps = 1e-2
    with torch.no_grad():
        lp, outp = f(b.x + eps * vx)
        lm, _ = f(b.x - eps * vx)
        _, out_again = f(b.x.clone())
    numeric = float((lp - lm) / (2 * eps))
    assert torch.equal(out_again.x, out0.x.detach())          # pinned offset => identical masks
    assert abs(numeric - analytic) <= 3e-2 * max(1.0, abs(analytic)), (numeric, analytic)
    # different offsets => different masks; eval mode => no dropout
    with torch.no_grad():
        _set_dropout_counter(9 * 4096)
        other = layer(graphgps_b200.GraphBatch(x=b.x.clone(), edge_index=b.edge_index, edge_attr=b.edge_attr.clone(),
                                               batch=b.batch, num_graphs=b.num_graphs))
    assert not torch.equal(other.x, out0.x.detach())


def test_cuda_graph_replay_matches_eager_and_redraws_dropout():
    torch.manual_seed(1)
    d = 64
    layer = graphgps_b200.GPSLayer(d, "CustomGatedGCN", "Transformer", 4, dropout=0.0, attn_dropout=0.0).to(DEV).train()
    b = make_batch("zinc-gatedgcn", seed=4, dim=d, num_graphs=10).to(DEV)
    x = b.x.clone().requires_grad_(True)
    ct = torch.randn_like(b.x)

    def body():
        bb = graphgps_b200.GraphBatch(x=x, edge_index=b.edge_index, edge_attr=b.edge_attr, batch=b.batch,
                                      num_graphs=b.num_graphs)
        if "_gps_b200_graph" in b.__dict__:
            bb.__dict__["_gps_b200_graph"] = b.__dict__["_gps_b200_graph"]
        x.grad = None
        out = layer(bb)
        torch.autograd.backward([out.x], [ct])
        return out.x

    graph_of(b)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(2):
            body()
    torch.cuda.current_stream().wait_stream(side)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        y = body()
    gx_static = x.grad
    g.replay()
    torch.cuda.synchronize()
    y1, gx1 = y.clone(), gx_static.clone()
    y_eager = body().detach()
    assert rel_err(y1.cpu(), y_eager.cpu()) < 1e-6 and rel_err(gx1.cpu(), x.grad.cpu()) < 1e-6


# ------------------------------------------------------------------------------- round-2 additions
def test_performer_attn_dropout_matches_oracle_with_injected_masks():
    """SelfAttention ends with dropout(p=attn_dropout) on to_out(out) (performer_layer.py:501-503; built with
    dropout=self.attn_dropout at gps_layer.py:112-114) before GPSLayer.dropout_attn.  The library's Philox masks for
    that site (GPS_SITE_PERF_OUT = 7) and for dropout_attn (site 4) are replayed through gps_dropout_mask and
    injected into the oracle, so the comparison is exact - forward, gradients and running statistics."""
    import copy
    from oracle.gps_oracle import to_dense_batch
    lib = _lib.load()
    d, heads, pa, pd = 64, 4, 0.5, 0.2
    torch.manual_seed(3)
    ora = OracleGPSLayer(d, "CustomGatedGCN", "Performer", heads, dropout=0.0, attn_dropout=0.0)
    ours = graphgps_b200.GPSLayer(d, "CustomGatedGCN", "Performer", heads, dropout=pd, attn_dropout=pa)
    ours.load_state_dict(ora.state_dict())
    ours = ours.to(DEV).train()
    b = make_batch("zinc-gatedgcn", seed=8, dim=d, num_graphs=9)
    N = b.num_nodes
    base = 21 * 4096
    _set_dropout_counter(base)
    seed = int(torch.initial_seed()) & 0xFFFFFFFFFFFFFFFF
    masks = {}
    for site, p in ((7, pa), (4, pd), (1, pd), (2, pd), (5, pd), (6, pd)):
        rows, cols = (b.num_edges, d) if site == 2 else ((N, 2 * d) if site == 5 else (N, d))
        m = torch.empty(rows, cols, device=DEV)
        _lib.check(lib.gps_dropout_mask(m.data_ptr(), rows, cols, p, seed, base + 4096, site, _stream()), "mask")
        masks[site] = (m.cpu().double() / (1.0 - p))

    class Fixed(torch.nn.Module):
        def __init__(self, m, dense=None):
            super().__init__()
            self.m, self.dense = m, dense

        def forward(self, t):
            if self.dense is not None:          # the Performer's dropout sees the padded dense batch
                md, _ = to_dense_batch(self.m, self.dense, None)
                return t * md
            return t * self.m

    o64 = copy.deepcopy(ora).double()
    o64.self_attn.dropout = Fixed(masks[7], dense=b.batch)
    o64.dropout_attn = Fixed(masks[4])
    _inject_gatedgcn_dropout(o64.local_model, masks[1], masks[2])
    o64.ff_dropout1, o64.ff_dropout2 = Fixed(masks[5]), Fixed(masks[6])
    g = torch.Generator().manual_seed(4)
    fix = {"config": dict(local="CustomGatedGCN"), "ct_x": torch.randn(b.x.shape, generator=g),
           "ct_e": torch.randn(b.edge_attr.shape, generator=g)}
    ref = run_layer(o64, _to(b.clone(), "cpu", torch.float64), fix)
    res = run_layer(ours, b.clone().to(DEV), fix)
    tgt = {k: ref[k] for k in ("out_x", "out_e", "grad_x", "grad_e")}
    tgt["grad_params"], tgt["state_after"] = ref["grad_params"], ref["state_after"]
    compare(res, tgt, 1e-3, "Performer with attn_dropout / dropout masks injected", grad_l2_tol=5e-3)
    # and the masks matter: without the attn_dropout site the outputs differ visibly
    o_plain = copy.deepcopy(ora).double()
    with torch.no_grad():
        plain = o_plain(_to(b.clone(), "cpu", torch.float64)).x
    assert rel_err(res["out_x"], plain.float()) > 1e-2


def _inject_gatedgcn_dropout(local, mx, me):
    """The oracle's GatedGCN applies F.dropout(x, p, training) inline (gatedgcn_layer.py:79-80): patch its p to 0 and
    multiply through a forward hook instead is not possible without touching the oracle, so wrap its forward."""
    import torch.nn.functional as F
    orig = local.forward

    def fwd(x, e, edge_index):
        calls = []
        real = F.dropout

        def fake(t, p=0.5, training=True, inplace=False):
            calls.append(1)
            return t * (mx if len(calls) == 1 else me)
        F.dropout = fake
        try:
            return orig(x, e, edge_index)
        finally:
            F.dropout = real
    local.forward = fwd


def test_three_layer_stack_matches_reference_stack():
    """GPSModel chains L GPSLayers, each consuming the previous layer's batch.x AND batch.edge_attr
    (graphgps/network/gps_model.py:100,105-108).  Three CUDA layers chained vs three oracle layers in fp64, whose
    results are pinned to those of three chained reference-verbatim layers (tests/golden/reference/stack3.pt, from
    make_golden.py): outputs, input gradients and every layer's parameter gradients."""
    d, heads, L = 64, 4, 3
    torch.manual_seed(11)
    refs = [OracleGPSLayer(d, "CustomGatedGCN", "Transformer", heads) for _ in range(L)]
    ours = []
    for r in refs:
        m = graphgps_b200.GPSLayer(d, "CustomGatedGCN", "Transformer", heads)
        m.load_state_dict(r.state_dict(), strict=True)
        ours.append(m.to(DEV).train())
    b = make_batch("zinc-gatedgcn", seed=13, dim=d, num_graphs=24)
    g = torch.Generator().manual_seed(6)
    ct_x, ct_e = torch.randn(b.x.shape, generator=g), torch.randn(b.edge_attr.shape, generator=g)
    fix = load_reference_golden("stack3")
    check_summary({f"{li}.{k}": v for li, r in enumerate(refs) for k, v in r.state_dict().items()}, fix["state"], 1e-12,
                  "seeded weights differ from make_golden.py's", scaled=True)
    check_summary({"x": b.x, "edge_attr": b.edge_attr, "edge_index": b.edge_index, "batch": b.batch, "ct_x": ct_x,
                   "ct_e": ct_e}, fix["inputs"], 1e-12, "seeded batch differs from make_golden.py's", scaled=True)

    def run(layers, bb, dev, dt):
        bb.x.requires_grad_(True)
        bb.edge_attr.requires_grad_(True)
        x_in, e_in = bb.x, bb.edge_attr
        for layer in layers:
            bb = layer(bb)
        ((bb.x * ct_x.to(dev, dt)).sum() + (bb.edge_attr * ct_e.to(dev, dt)).sum()).backward()
        return (bb.x.detach().cpu(), bb.edge_attr.detach().cpu(), x_in.grad.cpu(), e_in.grad.cpu(),
                [{n: p.grad.detach().cpu() for n, p in layer.named_parameters() if p.grad is not None} for layer in layers])

    rb = _to(b.clone(), "cpu", torch.float64)
    r = run([m.double() for m in refs], rb, "cpu", torch.float64)
    check_summary({"x": r[0], "e": r[1], "gx": r[2], "ge": r[3]}, fix["outputs"], 1e-9, "fp64 target vs reference",
                  scaled=True)
    check_summary({f"{li}.{n}": t for li in range(L) for n, t in r[4][li].items()}, fix["grads"], 1e-9,
                  "fp64 target vs reference parameter gradients", scaled=True)
    o = run(ours, b.clone().to(DEV), DEV, torch.float32)
    for name, a, t in (("x", o[0], r[0]), ("e", o[1], r[1])):
        assert rel_err(a, t) < 1e-3, (name, rel_err(a, t))
    for name, a, t in (("gx", o[2], r[2]), ("ge", o[3], r[3])):
        assert rel_err(a, t) < 1e-3 or rel_l2(a, t) < 5e-3, (name, rel_err(a, t), rel_l2(a, t))
    for li in range(L):
        for n, t in r[4][li].items():
            a = o[4][li][n]   # three layers deep: ReLU-kink flips of the later layers add up (measured 6.2e-3 on layer 0)
            assert rel_err(a, t) < 1e-3 or rel_l2(a, t) < 1e-2, (li, n, rel_err(a, t), rel_l2(a, t))


def test_eval_then_train_same_batch_and_retain_graph():
    """ADVICE r1: the plan cache must not hand an eval-sized saved buffer to a training call on the same (N, E);
    VERDICT r1: backward(retain_graph=True) followed by a second backward works as on the reference module."""
    torch.manual_seed(2)
    layer = graphgps_b200.GPSLayer(64, "CustomGatedGCN", "Transformer", 4).to(DEV)
    b = make_batch("zinc-gatedgcn", seed=2, dim=64, num_graphs=6).to(DEV)
    layer.eval()
    with torch.no_grad():
        layer(b.clone())
    layer.train()
    bb = b.clone()
    bb.x.requires_grad_(True)
    x_in = bb.x
    out = layer(bb)
    loss = out.x.square().sum()
    loss.backward(retain_graph=True)
    g1 = x_in.grad.clone()
    x_in.grad = None
    loss.backward()
    assert rel_err(x_in.grad.cpu(), g1.cpu()) < 1e-6


def test_eval_mode_backward_matches_oracle():
    """Input saliency in eval mode (running statistics, no dropout) works on the reference module; here the BatchNorm
    backward degenerates to a per-column affine map (VERDICT r1 weak #4)."""
    fix = load_golden("gatedgcn_transformer_gelu")
    cfg = fix["config"]
    ora = OracleGPSLayer(cfg["d"], cfg["local"], cfg["glob"], cfg["heads"], act=cfg["act"], dropout=0.3, attn_dropout=0.3)
    ora.load_state_dict(fix["state"])
    ours = graphgps_b200.GPSLayer(cfg["d"], cfg["local"], cfg["glob"], cfg["heads"], act=cfg["act"], dropout=0.3,
                                  attn_dropout=0.3)
    ours.load_state_dict(fix["state"])
    ours = ours.to(DEV).eval()
    ora = ora.double().eval()
    ref = run_layer(ora, golden_batch(fix, dtype=torch.float64), fix)
    res = run_layer(ours, golden_batch(fix, DEV), fix)
    tgt = {k: ref[k] for k in ("out_x", "out_e", "grad_x", "grad_e")}
    tgt["grad_params"], tgt["state_after"] = ref["grad_params"], ref["state_after"]
    compare(res, tgt, 1e-3, "eval-mode forward + backward", grad_l2_tol=5e-3)
