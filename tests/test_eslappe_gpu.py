"""GPU: EquivStableLapPE edge gate of the GatedGCN local model (GPSLayer(..., equivstable_pe=True)).

Stages (gate forward, gated aggregation, gate backward + PE gradient) against fp64 torch; the whole layer against the
reference-made ES fixtures (tests/golden/eslappe/) and, at the C3 shape, against the oracle; properties: a gate of
exactly 1 reproduces the plain layer, runs are bitwise reproducible, no PE gradient when none is asked for, and the
stack paths (captured replay, gradient bucket, overlapped events) agree with eager.

The gate's gradient is a difference (g scales numerator and denominator of the aggregation), so the PE and mlp_r_ij
gradients are small next to the rest; besides util.compare's max-abs bound they are held to a relative L2 bound."""
import copy
import ctypes as C

import pytest
import torch

import graphgps_b200
from graphgps_b200 import _lib
from graphgps_b200.batch import add_equivstable_pe, batch_from_lists, make_batch
from graphgps_b200.graph import graph_of
from es_oracle import OracleGPSLayerES
from es_util import es_batch, es_golden_names, es_l2_errors, load_es_golden, run_es_layer
from util import compare, rel_err, rel_l2

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
TOL = {"fp32": 1e-3, "bf16": 1e-2}
GRAD_L2 = {"fp32": 5e-3, "bf16": 1e-1}   # as tests/test_layer_gpu.py
ES_L2 = {"fp32": 1e-3, "bf16": GRAD_L2["bf16"]}


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _mlp(d, act, seed):
    g = torch.Generator().manual_seed(seed)
    m = torch.nn.Sequential(torch.nn.Linear(1, d), torch.nn.ReLU() if act == "relu" else torch.nn.GELU(),
                            torch.nn.Linear(d, 1), torch.nn.Sigmoid())
    with torch.no_grad():
        for p in m.parameters():
            p.copy_(torch.randn(p.shape, generator=g) * (0.5 if p.dim() == 2 and p.shape[0] == 1 else 1.0))
    return m


def _small_batch(d):
    """Isolated nodes (2, 7), self loops (1->1, 5->5), a duplicate edge (3->4 twice), an empty graph."""
    return batch_from_lists([5, 0, 4], [[(0, 1), (1, 1), (3, 4), (3, 4), (4, 0), (1, 0)],
                                        [], [(0, 1), (1, 1), (1, 0), (3, 1)]], d=d, seed=3)


STAGE_CASES = [("pcqm4m-small", 304, 304, "relu"), ("small", 52, 20, "gelu"), ("small", 52, 52, "relu"),
               ("zinc-gatedgcn", 64, 8, "gelu")]


def _stage_batch(shape, d, k):
    b = _small_batch(d) if shape == "small" else make_batch(shape, seed=2, dim=d)
    add_equivstable_pe(b, k, seed=4, scale=1.0 if k <= 52 else 0.3)
    return b.to(DEV)


@pytest.mark.parametrize("shape,d,k,act", STAGE_CASES)
def test_es_gate_and_gated_aggregation_forward(shape, d, k, act):
    lib = _lib.load()
    b = _stage_batch(shape, d, k)
    gs = graph_of(b)
    N, E = b.num_nodes, b.num_edges
    m = _mlp(d, act, 1).to(DEV)
    pe = b.pe_EquivStableLapPE
    src, dst = b.edge_index
    r64 = ((pe[dst].double() - pe[src].double()) ** 2).sum(-1, keepdim=True)
    g64 = copy.deepcopy(m).double()(r64).squeeze(1)
    r, gate = torch.empty(E, device=DEV), torch.empty(E, device=DEV)
    _lib.check(lib.gps_es_gate_forward(C.byref(gs.desc), pe.data_ptr(), k, d, _lib.ACT[act], m[0].weight.data_ptr(),
                                       m[0].bias.data_ptr(), m[2].weight.data_ptr(), m[2].bias.data_ptr(), r.data_ptr(),
                                       gate.data_ptr(), _stream()), "es_gate_forward")
    assert rel_err(r.cpu(), r64.squeeze(1).cpu()) < 2e-5
    assert rel_err(gate.cpu(), g64.cpu()) < 2e-5
    # gated aggregation, gate from the kernel above
    Y = torch.randn(N, 4 * d, device=DEV)
    Ce = torch.randn(E, d, device=DEV)
    Ax, Bx, Dx, Ex = (Y[:, i * d:(i + 1) * d].double() for i in range(4))
    e_ij = Dx[dst] + Ex[src] + Ce.double()
    sig = torch.sigmoid(e_ij) * gate.double()[:, None]
    num = torch.zeros(N, d, device=DEV, dtype=torch.float64).index_add_(0, dst, sig * Bx[src])
    den = torch.zeros(N, d, device=DEV, dtype=torch.float64).index_add_(0, dst, sig)
    xt_ref = Ax + num / (den + 1e-6)
    xt = torch.empty(N, d, device=DEV)
    sx = torch.zeros(2, d, device=DEV, dtype=torch.float64)
    se = torch.zeros(2, d, device=DEV, dtype=torch.float64)
    base = Y.data_ptr()
    _lib.check(lib.gps_gatedgcn_es_aggregate_forward(C.byref(gs.desc), d, base, base + 4 * d, base + 8 * d,
                                                     base + 12 * d, 4 * d, Ce.data_ptr(), xt.data_ptr(), sx.data_ptr(),
                                                     se.data_ptr(), gate.data_ptr(), _stream()), "es_aggregate")
    assert rel_err(xt.cpu(), xt_ref.cpu()) < 2e-5
    assert rel_err(Ce.cpu(), e_ij.cpu()) < 1e-5                 # the edge output stays ungated
    assert rel_err(sx[0].cpu(), xt_ref.sum(0).cpu()) < 1e-4


@pytest.mark.parametrize("shape,d,k,act", STAGE_CASES)
def test_es_gate_backward_and_pe_gradient(shape, d, k, act):
    lib = _lib.load()
    b = _stage_batch(shape, d, k)
    gs = graph_of(b)
    E = b.num_edges
    m = _mlp(d, act, 2).to(DEV)
    pe = b.pe_EquivStableLapPE
    src, dst = b.edge_index
    m64 = copy.deepcopy(m).double()
    pe64 = pe.double().requires_grad_(True)
    r64 = ((pe64[dst] - pe64[src]) ** 2).sum(-1, keepdim=True)
    r64.retain_grad()
    g64 = m64(r64).squeeze(1)
    g_gate = torch.randn(E, generator=torch.Generator().manual_seed(3)).to(DEV)
    g64.backward(g_gate.double())
    gz_abs = float((g_gate.double() * g64 * (1 - g64)).abs().sum())   # scale of the scalar sum d loss / d b2
    r, gate = r64.detach().squeeze(1).float().contiguous(), g64.detach().float().contiguous()
    g_r = torch.empty(E, device=DEV)
    grads = [torch.full_like(p, float("nan")) for p in (m[0].weight, m[0].bias, m[2].weight, m[2].bias)]
    nbytes = lib.gps_es_gate_backward_workspace_bytes(E, d)
    ws = torch.empty(max(nbytes, 256), dtype=torch.uint8, device=DEV)
    _lib.check(lib.gps_es_gate_backward(E, d, _lib.ACT[act], m[0].weight.data_ptr(), m[0].bias.data_ptr(),
                                        m[2].weight.data_ptr(), m[2].bias.data_ptr(), r.data_ptr(), gate.data_ptr(),
                                        g_gate.data_ptr(), g_r.data_ptr(), *(t.data_ptr() for t in grads),
                                        ws.data_ptr(), ws.numel(), _stream()), "es_gate_backward")
    grad_pe = torch.empty_like(pe)
    _lib.check(lib.gps_es_pe_backward(C.byref(gs.desc), pe.data_ptr(), k, g_r.data_ptr(), grad_pe.data_ptr(), _stream()),
               "es_pe_backward")
    torch.cuda.synchronize()
    assert rel_l2(g_r.cpu(), r64.grad.squeeze(1).cpu()) < 1e-4
    for got, p in zip(grads[:3], (m64[0].weight, m64[0].bias, m64[2].weight)):
        assert rel_l2(got.cpu(), p.grad.cpu()) < 1e-4
    # mlp_r_ij.2.bias: one scalar sum over E signed terms, which may cancel: bounded against the sum of magnitudes
    assert abs(float(grads[3]) - float(m64[2].bias.grad)) <= 1e-5 * gz_abs
    assert rel_l2(grad_pe.cpu(), pe64.grad.cpu()) < 1e-4


# ------------------------------------------------------------------------------- whole layer
def _layer(cfg, precision="fp32"):
    return graphgps_b200.GPSLayer(cfg["d"], cfg["local"], cfg["glob"], cfg["heads"], act=cfg["act"],
                                  precision=precision, equivstable_pe=True)


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
@pytest.mark.parametrize("name", es_golden_names())
def test_es_layer_matches_golden(name, precision):
    fix = load_es_golden(name)
    cfg = fix["config"]
    layer = _layer(cfg, precision)
    layer.load_state_dict(fix["state"], strict=True)
    layer = layer.to(DEV).train(cfg["training"])
    res = run_es_layer(layer, es_batch(fix, DEV), fix, backward=cfg["training"])
    ref = fix
    if precision == "bf16" and cfg["training"]:
        # BatchNorm bias gradients are near-cancelling column sums of ~100 bf16-rounded rows on these small batches:
        # measured on B200 up to 0.11 relative L2 (local_model.bn_node_x.bias) on batches of this size, while the same
        # sums are at rounding level in fp32.  Held to 0.15 here, every other gradient to GRAD_L2["bf16"].
        ref = dict(fix, grad_params={n: g for n, g in fix["grad_params"].items() if not _bn_bias(n)})
        for n, g in fix["grad_params"].items():
            if _bn_bias(n):
                assert rel_l2(res["grad_params"][n], g) <= 0.15, n
    compare(res, ref, TOL[precision], f"CUDA {precision} vs ES golden {name}", grad_l2_tol=GRAD_L2[precision])
    if cfg["training"]:
        errs = es_l2_errors(res, fix)
        print(name, precision, {k: f"{v:.2e}" for k, v in errs.items()})
        assert max(errs.values()) <= ES_L2[precision], errs


def _bn_bias(name):
    return name.endswith(".bias") and ("norm" in name or "bn_" in name)


def _c3(glob, heads, seed=0, scale=0.3):
    torch.manual_seed(seed)
    ora = OracleGPSLayerES(304, "CustomGatedGCN", glob, heads)
    b = make_batch("pcqm4m-small", seed=7)
    add_equivstable_pe(b, seed=8, scale=scale)
    g = torch.Generator().manual_seed(9)
    fix = {"config": dict(local="CustomGatedGCN"), "ct_x": torch.randn(b.x.shape, generator=g),
           "ct_e": torch.randn(b.edge_attr.shape, generator=g)}
    return ora, b, fix


def _pe_grad_batch(b, dev, dt):
    b = b.clone()
    b.x, b.edge_attr = b.x.to(dev, dt), b.edge_attr.to(dev, dt)
    b.batch, b.edge_index = b.batch.to(dev), b.edge_index.to(dev)
    b.pe_EquivStableLapPE = b.pe_EquivStableLapPE.to(dev, dt).requires_grad_(True)
    return b


@pytest.mark.parametrize("glob,heads", [("Transformer", 4), ("Performer", 4)])
def test_es_layer_matches_oracle_full_size(glob, heads):
    """C3 (pcqm4m-GPS-ESLapPE: d=304, 256 graphs) with PE at scale 0.3 (default-init gates spread, none saturated).

    Every output and every gradient outside the gate is held to the plain layer's full-size bounds (1e-3 max-abs or
    5e-3 relative L2).  The gate's own gradients (PE, mlp_r_ij) are a cancelling reduction: d loss / d g_ij is
    proportional to (Bx_j - agg_i), summed over 304 channels, then over ~7.5k edges of mixed sign.  It amplifies the
    relative error of the gradient it reads (g_x~, produced by the fp32-grade split-bf16 products) by two to three
    orders of magnitude: measured on B200, relative L2 up to 1.1e-3 (Transformer) and 2.6e-2 (Performer) against fp64,
    where the oracle's own true-fp32 run already reaches 5.4e-4 on the Transformer weights.  They are held to 5e-2 here;
    a missing or wrong term is O(1).  Their arithmetic is pinned exactly by the stage tests (1e-4 against fp64) and by
    the ES fixtures (1e-3)."""
    ora, b, fix = _c3(glob, heads)
    src, dst = b.edge_index
    with torch.no_grad():
        pe = b.pe_EquivStableLapPE
        gate = ora.local_model.mlp_r_ij(((pe[dst] - pe[src]) ** 2).sum(-1, keepdim=True))
    assert float(gate.std()) > 0.03 and float((gate > 0.999).float().mean()) <= 0.01
    ours = graphgps_b200.GPSLayer(304, "CustomGatedGCN", glob, heads, equivstable_pe=True)
    ours.load_state_dict(ora.state_dict())
    ours = ours.to(DEV)
    ref64 = run_es_layer(copy.deepcopy(ora).double(), _pe_grad_batch(b, "cpu", torch.float64), fix)
    res = run_es_layer(ours, _pe_grad_batch(b, DEV, torch.float32), fix)
    t = {k: ref64[k] for k in ("out_x", "out_e", "grad_x", "grad_e")}
    t["grad_params"] = {n: g for n, g in ref64["grad_params"].items() if "mlp_r_ij" not in n}
    t["state_after"] = ref64["state_after"]
    compare(res, t, 1e-3, f"CUDA fp32 ES vs oracle fp64 @ C3 {glob}", grad_l2_tol=5e-3)
    t["grad_params"], t["grad_pe"] = ref64["grad_params"], ref64["grad_pe"]
    errs = es_l2_errors(res, t)
    print(glob, {k: f"{v:.2e}" for k, v in errs.items()})
    assert max(errs.values()) <= 5e-2, errs


def test_gate_of_one_reproduces_the_plain_layer():
    """mlp_r_ij.2.weight = 0, .2.bias = 40: sigmoid(40) is exactly 1.0f, so the ES layer computes the plain GatedGCN
    layer (outputs to 1e-6, gradients to 2e-5: the weight and bias gradients are split-K sums with float atomics, whose
    order-dependent rounding alone moves them by ~1e-5 between two runs, as in tests/test_stack_gpu.py) and its PE
    gradient vanishes."""
    torch.manual_seed(5)
    es = graphgps_b200.GPSLayer(304, "CustomGatedGCN", "Transformer", 4, equivstable_pe=True)
    with torch.no_grad():
        es.local_model.mlp_r_ij[2].weight.zero_()
        es.local_model.mlp_r_ij[2].bias.fill_(40.0)
    plain = graphgps_b200.GPSLayer(304, "CustomGatedGCN", "Transformer", 4)
    plain.load_state_dict({k: v for k, v in es.state_dict().items() if "mlp_r_ij" not in k}, strict=True)
    es, plain = es.to(DEV), plain.to(DEV)
    b = make_batch("pcqm4m-small", seed=3)
    add_equivstable_pe(b, seed=2)
    g = torch.Generator().manual_seed(1)
    fix = {"config": dict(local="CustomGatedGCN"), "ct_x": torch.randn(b.x.shape, generator=g),
           "ct_e": torch.randn(b.edge_attr.shape, generator=g)}
    r_es = run_es_layer(es, _pe_grad_batch(b, DEV, torch.float32), fix)
    r_pl = run_es_layer(plain, _pe_grad_batch(b, DEV, torch.float32), fix)
    for k in ("out_x", "out_e"):
        assert rel_err(r_es[k], r_pl[k]) < 1e-6, k
    for k in ("grad_x", "grad_e"):
        assert rel_err(r_es[k], r_pl[k]) < 2e-5, k
    for n, gp in r_pl["grad_params"].items():
        assert rel_err(r_es["grad_params"][n], gp) < 2e-5, n
    assert r_pl["grad_pe"] is None and float(r_es["grad_pe"].abs().max()) == 0.0


def _es_step(layer, b, fix):
    res = run_es_layer(layer, _pe_grad_batch(b, DEV, torch.float32), fix)
    torch.cuda.synchronize()
    return res


def test_es_layer_is_deterministic_and_pe_gradient_is_optional():
    ora, b, fix = _c3("Transformer", 4, seed=2)
    layer = graphgps_b200.GPSLayer(304, "CustomGatedGCN", "Transformer", 4, equivstable_pe=True)
    layer.load_state_dict(ora.state_dict())
    layer = layer.to(DEV)
    a1 = _es_step(layer, b, fix)
    layer.zero_grad(set_to_none=True)
    a2 = _es_step(layer, b, fix)
    assert torch.equal(a1["out_x"], a2["out_x"]) and torch.equal(a1["grad_pe"], a2["grad_pe"])
    for n in a1["grad_params"]:
        if "mlp_r_ij" in n:
            assert torch.equal(a1["grad_params"][n], a2["grad_params"][n]), n
    # pe.requires_grad = False: no PE gradient, every other gradient as before
    layer.zero_grad(set_to_none=True)
    bb = _pe_grad_batch(b, DEV, torch.float32)
    bb.pe_EquivStableLapPE.requires_grad_(False)
    a3 = run_es_layer(layer, bb, fix)
    assert a3["grad_pe"] is None and bb.pe_EquivStableLapPE.grad is None
    assert torch.equal(a3["out_x"], a1["out_x"])
    assert rel_err(a3["grad_x"], a1["grad_x"]) < 1e-6
    for n, g in a1["grad_params"].items():
        assert rel_err(a3["grad_params"][n], g) < 1e-5, n


def test_es_layer_requires_the_batch_pe():
    layer = graphgps_b200.GPSLayer(64, "CustomGatedGCN", "Transformer", 4, equivstable_pe=True).to(DEV)
    b = make_batch("zinc-gatedgcn", seed=1, dim=64, num_graphs=4).to(DEV)
    with pytest.raises(AttributeError):
        layer(b.clone())
    b.pe_EquivStableLapPE = torch.zeros(b.num_nodes, 64, dtype=torch.float64, device=DEV)
    with pytest.raises(TypeError):
        layer(b.clone())
    b.pe_EquivStableLapPE = torch.zeros(b.num_nodes + 1, 64, device=DEV)
    with pytest.raises(ValueError):
        layer(b.clone())


# ------------------------------------------------------------------------------- stack
def _stack_eager(stack, b, ct_x, ct_e):
    bb = b.clone()
    for t in (bb.x, bb.edge_attr, bb.pe_EquivStableLapPE):
        t.requires_grad_(True)
    x_in, pe_in = bb.x, bb.pe_EquivStableLapPE
    out = stack(bb)
    torch.autograd.backward([out.x, out.edge_attr], [ct_x, ct_e])
    return out.x.detach().clone(), x_in.grad.clone(), pe_in.grad.clone()


def test_es_stack_capture_bucket_and_overlap_events():
    torch.manual_seed(4)
    stack = graphgps_b200.GPSStack(3, 64, "CustomGatedGCN", "Transformer", 4, equivstable_pe=True).to(DEV).train()
    b = make_batch("zinc-gatedgcn", seed=5, dim=64, num_graphs=12)
    add_equivstable_pe(b, seed=6, scale=2.0)
    b = b.to(DEV)
    graph_of(b)
    ct_x, ct_e = torch.randn_like(b.x), torch.randn_like(b.edge_attr)
    # plain path (fresh .grad tensors), plane hand-off on
    for p in stack.parameters():
        p.grad = None
    eager = _stack_eager(stack, b, ct_x, ct_e)
    plain_grads = [p.grad.clone() for p in stack.parameters()]
    # GradBucket path: gradients added into the static bucket views
    bucket = stack.make_grad_bucket(overlap=True)
    bucket.zero_()
    ev_mid = bucket.events[1][1]       # layer 1, MID group (local model incl. mlp_r_ij)
    snap_stream = torch.cuda.Stream(device=DEV)
    mlp = [p for n, p in stack.layers[1].named_parameters() if "mlp_r_ij" in n]
    viaB = _stack_eager(stack, b, ct_x, ct_e)
    with torch.cuda.stream(snap_stream):
        snap_stream.wait_event(ev_mid)
        snap = [p.grad.clone() for p in mlp]
    torch.cuda.current_stream().wait_stream(snap_stream)
    torch.cuda.synchronize()
    for s, p in zip(snap, mlp):
        assert torch.equal(s, p.grad)                 # final when ev_grads_mid fires
    assert rel_err(viaB[0].cpu(), eager[0].cpu()) < 1e-6 and rel_err(viaB[2].cpu(), eager[2].cpu()) < 1e-5
    for p, g in zip(stack.parameters(), plain_grads):
        assert rel_err(p.grad.cpu(), g.cpu()) < 1e-5
    # captured replay of the whole step equals eager
    step = stack.capture(b, ct_x, ct_e, bucket=bucket)
    for _ in range(2):
        step.replay()
    torch.cuda.synchronize()
    assert rel_err(step.x_out.cpu(), eager[0].cpu()) < 1e-6 and rel_err(step.grad_x.cpu(), eager[1].cpu()) < 1e-6
    assert rel_l2(step.grad_pe.cpu(), eager[2].cpu()) < 1e-5
    for p, g in zip(stack.parameters(), plain_grads):
        assert rel_err(p.grad.cpu(), g.cpu()) < 1e-5
