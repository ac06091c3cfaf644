"""B200-native drop-in for `graphgps.layer.gps_layer.GPSLayer`.

Same constructor signature, `forward(batch) -> batch` contract and `state_dict` layout as the
reference module (graphgps/layer/gps_layer.py:16-264; parameter names per SURVEY.md section 8b), so
`graphgps/network/gps_model.py:85-99` can instantiate it unchanged and reference checkpoints load
with `load_state_dict`.  All arithmetic of the layer — the five GatedGCN projections, the
CSR/CSC segmented gather-reduce, softmax attention over each graph's node set, residual/BatchNorm/FFN
and the whole backward pass — runs in hand-written CUDA (libgps_b200.so, sm_100a) reached through
one C-ABI call per direction; PyTorch only owns memory, streams and the autograd graph edge.
There is NO fallback: CPU tensors or a missing library raise.
"""
from __future__ import annotations

import ctypes as C
import math

import torch
import torch.nn as nn

from . import _lib
from .graph import graph_of

_SUPPORTED_LOCAL = ("None", "CustomGatedGCN", "GINE", "GCN")
_EDGE_LOCAL = ("CustomGatedGCN", "GINE")   # local models that read batch.edge_attr (gps_layer.py:44-53)
_KNOWN_LOCAL = _SUPPORTED_LOCAL + ("GIN", "GENConv", "GAT", "PNA")
_SUPPORTED_GLOBAL = ("None", "Transformer", "Performer")
_KNOWN_GLOBAL = _SUPPORTED_GLOBAL + ("BiasedTransformer", "BigBird")
_ACT_MODULES = {"relu": nn.ReLU, "gelu": nn.GELU}

_workspaces = {}
_dropout_calls = [0]
_drop_counters = {}


def _next_dropout_offset(device):
    """Device-resident Philox offset for this call: counter += 4096; snapshot = counter.

    Kept on the device (two tiny stream-ordered ops) so that a captured CUDA graph draws fresh dropout
    masks on every replay; the snapshot tensor is what forward and backward of this call both read."""
    ctr = _drop_counters.get(device)
    if ctr is None:
        ctr = torch.zeros(1, dtype=torch.int64, device=device)
        _drop_counters[device] = ctr
    ctr.add_(4096)
    return ctr.clone()


def _workspace(device, nbytes):
    """Transient scratch for one C call, one buffer per (device, stream): layers running on different streams never
    share it, and a buffer is never freed while the process lives (a captured CUDA graph may hold its address) -
    growth keeps the old ones.  Under stream capture the buffer is allocated from the graph's own pool instead."""
    if torch.cuda.is_current_stream_capturing():
        return torch.empty(int(nbytes) + 256, dtype=torch.uint8, device=device)
    key = (device, torch.cuda.current_stream(device).cuda_stream)
    held = _workspaces.setdefault(key, [])
    if not held or held[-1].numel() < nbytes:
        held.append(torch.empty(int(nbytes * 1.25) + 256, dtype=torch.uint8, device=device))
    return held[-1]


_PLANES_ATTR = "_gps_b200_planes"


def _batch_planes_get(batch):
    try:
        v = getattr(batch, _PLANES_ATTR, None)
    except Exception:
        v = None
    return v if isinstance(v, dict) else None


def _batch_planes_put(batch, produced, lo):
    """Remember, on the batch object, the operand planes this layer wrote next to its outputs, keyed by the identity
    (address, version, shape) of the tensors they mirror: the next GPSLayer uses them only if batch.x / batch.edge_attr
    are still exactly those tensors."""
    rec = {}
    for name, (t, buf) in (produced or {}).items():
        rec[name] = ((t.data_ptr(), t._version, tuple(t.shape), lo), buf)
    try:
        setattr(batch, _PLANES_ATTR, rec)
    except Exception:
        pass


class _GatedGCNParams(nn.Module):
    """Parameter container with the names of graphgps/layer/gatedgcn_layer.py:21-38; with equivstable_pe the
    EquivStableLapPE gate MLP `mlp_r_ij` (Linear(1,d), act, Linear(d,1), Sigmoid) sits between E and bn_node_x."""

    def __init__(self, dim, act="relu", equivstable_pe=False):
        super().__init__()
        self.A = nn.Linear(dim, dim, bias=True)
        self.B = nn.Linear(dim, dim, bias=True)
        self.C = nn.Linear(dim, dim, bias=True)
        self.D = nn.Linear(dim, dim, bias=True)
        self.E = nn.Linear(dim, dim, bias=True)
        if equivstable_pe:
            self.mlp_r_ij = nn.Sequential(nn.Linear(1, dim), _ACT_MODULES[act](), nn.Linear(dim, 1), nn.Sigmoid())
        self.bn_node_x = nn.BatchNorm1d(dim)
        self.bn_edge_e = nn.BatchNorm1d(dim)


class _GINEParams(nn.Module):
    """Names of PyG GINEConv(gin_nn) as built at gps_layer.py:62-69: nn.0, nn.2, eps buffer."""

    def __init__(self, dim, act):
        super().__init__()
        self.nn = nn.Sequential(nn.Linear(dim, dim), _ACT_MODULES[act](), nn.Linear(dim, dim))
        self.register_buffer("eps", torch.Tensor([0.0]))


class _GCNConvParams(nn.Module):
    """Names of PyG 2.2 GCNConv(dim_h, dim_h) as built at gps_layer.py:49-51: lin.weight (no bias, glorot), bias (zeros)."""

    def __init__(self, dim):
        super().__init__()
        self.lin = nn.Linear(dim, dim, bias=False)
        nn.init.xavier_uniform_(self.lin.weight)       # PyG Linear(weight_initializer='glorot')
        self.bias = nn.Parameter(torch.zeros(dim))


def _orthogonal_gaussian_matrix(nb_rows, nb_cols):
    """Random-feature projection drawn once at construction (performer_layer.py:163-195, scaling=0)."""
    blocks = []
    full = nb_rows // nb_cols
    for _ in range(full):
        q, _r = torch.linalg.qr(torch.randn(nb_cols, nb_cols), mode="reduced")
        blocks.append(q.t())
    rem = nb_rows - full * nb_cols
    if rem > 0:
        q, _r = torch.linalg.qr(torch.randn(nb_cols, nb_cols), mode="reduced")
        blocks.append(q.t()[:rem])
    final = torch.cat(blocks)
    mult = torch.randn(nb_rows, nb_cols).norm(dim=1)
    return torch.diag(mult) @ final


class _FastAttentionParams(nn.Module):
    def __init__(self, dim_head):
        super().__init__()
        nb = int(dim_head * math.log(dim_head))  # performer_layer.py:261
        self.register_buffer("projection_matrix", _orthogonal_gaussian_matrix(nb, dim_head))


class _PerformerParams(nn.Module):
    """Names of performer_pytorch.SelfAttention as built at gps_layer.py:111-114
    (dim_head=64, qkv_bias=False, attn_out_bias=True; performer_layer.py:421-474)."""

    def __init__(self, dim, heads, dim_head=64):
        super().__init__()
        inner = dim_head * heads
        self.heads, self.dim_head = heads, dim_head
        self.fast_attention = _FastAttentionParams(dim_head)
        self.to_q = nn.Linear(dim, inner, bias=False)
        self.to_k = nn.Linear(dim, inner, bias=False)
        self.to_v = nn.Linear(dim, inner, bias=False)
        self.to_out = nn.Linear(inner, dim, bias=True)


def _lin(weight, bias, gw=None, gb=None):
    return _lib.GpsLinear(_lib.ptr(weight), _lib.ptr(bias), _lib.ptr(gw), _lib.ptr(gb))


def _bn(mod, gw=None, gb=None):
    return _lib.GpsBatchNorm(_lib.ptr(mod.weight), _lib.ptr(mod.bias), _lib.ptr(mod.running_mean),
                             _lib.ptr(mod.running_var), _lib.ptr(mod.num_batches_tracked),
                             _lib.ptr(gw), _lib.ptr(gb))


class _GPSLayerFn(torch.autograd.Function):
    """One autograd node for the whole layer: forward = gps_layer_forward, backward = gps_layer_backward."""

    @staticmethod
    def forward(ctx, layer, gs, x, e, pe, *params):
        lib = _lib.load()
        dev = x.device
        named = dict(zip(layer._param_names, params))
        args = layer._base_args(gs, named)
        N, E, d = gs.N, gs.E, layer.dim_h
        x_out = torch.empty_like(x)
        e_out = torch.empty_like(e) if layer.local_gnn_type == "CustomGatedGCN" else None
        plan = layer._plan(args, gs)
        saved = torch.empty(max(plan[0], 256), dtype=torch.uint8, device=dev)
        ws = _workspace(dev, plan[1])
        args.x, args.edge_attr = x.data_ptr(), _lib.ptr(e)
        args.x_out, args.edge_out = x_out.data_ptr(), _lib.ptr(e_out)
        args.saved, args.saved_bytes = saved.data_ptr(), saved.numel()
        args.workspace, args.workspace_bytes = ws.data_ptr(), ws.numel()
        if layer._es:
            args.pe, args.pe_dim = pe.data_ptr(), pe.shape[1]
        hand = layer._handoff_args(args, plan, params, x, e, x_out, e_out)
        snap = None
        if layer.training and (layer.dropout > 0 or layer.attn_dropout > 0):
            snap = _next_dropout_offset(dev)
            args.offset, args.offset_dev = 0, snap.data_ptr()
        stream = torch.cuda.current_stream(dev).cuda_stream
        _lib.check(lib.gps_layer_forward(C.byref(args), stream), "gps_layer_forward")
        ctx.layer, ctx.gs, ctx.saved_buf, ctx.snap = layer, gs, saved, snap
        ctx.hand = hand
        ctx.seed, ctx.offset, ctx.training = args.seed, args.offset, bool(args.training)
        ctx.save_for_backward(x, e, pe, *params)
        if e_out is not None:
            return x_out, e_out
        return x_out

    @staticmethod
    def backward(ctx, g_x_out, g_e_out=None):
        lib = _lib.load()
        layer, gs = ctx.layer, ctx.gs
        x, e, pe, *params = ctx.saved_tensors
        dev = x.device
        named = dict(zip(layer._param_names, params))
        bucket = layer._bucket_grads(named)
        if bucket is not None:
            # static gradient bucket (graphgps_b200.dp.GradBucket): the library ADDS this call's gradients to the
            # parameters' .grad views in place (torch's accumulation semantics), so CUDA-graph replays and the
            # gradient all-reduce see the same memory
            grads = bucket
            args = layer._base_args(gs, named, grads)
            args.reserved0 = 3
        else:
            grads = {n: torch.empty_like(p) for n, p in named.items()}
            torch._foreach_zero_(list(grads.values()))   # one multi-tensor fill; the library then skips its memsets
            args = layer._base_args(gs, named, grads)
            args.reserved0 = 1
        args.seed, args.offset, args.training = ctx.seed, ctx.offset, 1 if ctx.training else 0
        if ctx.snap is not None:
            args.offset_dev = ctx.snap.data_ptr()
        g_x_out = g_x_out.contiguous()
        gated = layer.local_gnn_type == "CustomGatedGCN"
        if g_e_out is not None:
            g_e_out = g_e_out.contiguous()
        g_x = torch.empty_like(x)
        g_e = torch.empty_like(e) if layer.local_gnn_type in _EDGE_LOCAL else None
        plan = layer._plan(args, gs)
        ws = _workspace(dev, plan[1])
        args.x, args.edge_attr = x.data_ptr(), _lib.ptr(e)
        args.grad_x_out = g_x_out.data_ptr()
        args.grad_edge_out = _lib.ptr(g_e_out) if gated else 0
        args.grad_x, args.grad_edge_attr = g_x.data_ptr(), _lib.ptr(g_e)
        args.saved, args.saved_bytes = ctx.saved_buf.data_ptr(), ctx.saved_buf.numel()
        args.workspace, args.workspace_bytes = ws.data_ptr(), ws.numel()
        g_pe = None
        if layer._es:
            args.pe, args.pe_dim = pe.data_ptr(), pe.shape[1]
            if ctx.needs_input_grad[4]:
                g_pe = torch.empty_like(pe)
                args.grad_pe = g_pe.data_ptr()
        if ctx.hand is not None:
            args.x_planes_in, args.e_planes_in, args.wplanes, args.wplanes_bytes = ctx.hand[:4]
            args.wplanes_valid = 1
        evs = layer.__dict__.get("grad_events")
        if evs is not None:
            args.ev_grads_early, args.ev_grads_mid, args.ev_grads_done = (e.cuda_event for e in evs)
        stream = torch.cuda.current_stream(dev).cuda_stream
        _lib.check(lib.gps_layer_backward(C.byref(args), stream), "gps_layer_backward")
        # (ctx.saved_buf stays alive with the autograd node: backward(retain_graph=True) may run again)
        if bucket is not None:
            return (None, None, g_x, g_e, g_pe) + (None,) * len(layer._param_names)
        # parameters the configuration never reads get no gradient (as under autograd in the reference)
        unused = []
        if layer.local_gnn_type == "None":
            unused.append("norm1_local.")
        if layer.global_model_type == "None":
            unused.append("norm1_attn.")
        pg = tuple(None if any(n.startswith(u) for u in unused) else grads[n] for n in layer._param_names)
        return (None, None, g_x, g_e, g_pe) + pg


class GPSLayer(nn.Module):
    """Local MPNN + full graph attention x-former layer (reference: gps_layer.py:16-264)."""

    def __init__(self, dim_h, local_gnn_type, global_model_type, num_heads, act="relu",
                 pna_degrees=None, equivstable_pe=False, dropout=0.0, attn_dropout=0.0,
                 layer_norm=False, batch_norm=True, bigbird_cfg=None, log_attn_weights=False,
                 precision="fp32"):
        super().__init__()
        self.dim_h = dim_h
        self.num_heads = num_heads
        self.attn_dropout = attn_dropout
        self.dropout = dropout
        self.layer_norm = layer_norm
        self.batch_norm = batch_norm
        self.equivstable_pe = equivstable_pe
        self.act = act
        self.precision = precision
        if act not in _ACT_MODULES:
            raise NotImplementedError(f"activation '{act}' is not built in graphgps_b200 (relu, gelu)")
        self.activation = _ACT_MODULES[act]
        self.log_attn_weights = log_attn_weights
        if log_attn_weights and global_model_type not in ["Transformer", "BiasedTransformer"]:
            raise NotImplementedError(                                    # gps_layer.py:36-41
                f"Logging of attention weights is not supported "
                f"for '{global_model_type}' global attention model.")
        if log_attn_weights:
            raise NotImplementedError("log_attn_weights is not built in graphgps_b200")

        # ---- local message-passing model (gps_layer.py:44-99)
        self.local_gnn_with_edge_attr = True
        if local_gnn_type not in _KNOWN_LOCAL:
            raise ValueError(f"Unsupported local GNN model: {local_gnn_type}")
        if local_gnn_type not in _SUPPORTED_LOCAL:
            raise NotImplementedError(f"local GNN '{local_gnn_type}' is not built in graphgps_b200 "
                                      f"(available: {_SUPPORTED_LOCAL}); there is no fallback path")
        # EquivStableLapPE (gps_layer.py:66-69, 92-96, 163-171): GatedGCN gates its messages with it; GCN and None never
        # read it (as in the reference).  The reference's GINEConvESLapPE cannot be constructed (its reset_parameters()
        # reads mlp_r_ij before assigning it, gine_conv_layer.py:35,44,54), so there is no behaviour to reproduce.
        if equivstable_pe and local_gnn_type == "GINE":
            raise NotImplementedError("equivstable_pe with GINE is not built in graphgps_b200: the reference's "
                                      "GINEConvESLapPE raises AttributeError in its own constructor")
        self._es = bool(equivstable_pe) and local_gnn_type == "CustomGatedGCN"
        if local_gnn_type == "None":
            self.local_model = None
        elif local_gnn_type == "GINE":
            self.local_model = _GINEParams(dim_h, act)
        elif local_gnn_type == "GCN":
            self.local_gnn_with_edge_attr = False
            self.local_model = _GCNConvParams(dim_h)
        else:
            self.local_model = _GatedGCNParams(dim_h, act, self._es)
        self.local_gnn_type = local_gnn_type

        # ---- global attention model (gps_layer.py:101-122)
        if global_model_type not in _KNOWN_GLOBAL:
            raise ValueError(f"Unsupported global x-former model: {global_model_type}")
        if global_model_type not in _SUPPORTED_GLOBAL:
            raise NotImplementedError(f"global model '{global_model_type}' is not built in graphgps_b200")
        if global_model_type == "None":
            self.self_attn = None
        elif global_model_type == "Transformer":
            if dim_h % num_heads != 0:
                raise ValueError("embed_dim must be divisible by num_heads")
            # torch's own module is the parameter container (same init, same state_dict keys);
            # its forward is never called.
            self.self_attn = nn.MultiheadAttention(dim_h, num_heads, dropout=attn_dropout, batch_first=True)
        else:
            self.self_attn = _PerformerParams(dim_h, num_heads)
        self.global_model_type = global_model_type

        if self.layer_norm and self.batch_norm:
            raise ValueError("Cannot apply two types of normalization together")   # gps_layer.py:125-126
        if self.layer_norm or not self.batch_norm:
            raise NotImplementedError("graphgps_b200 builds the BatchNorm configuration "
                                      "(layer_norm=False, batch_norm=True) used by every shipped config")
        if self.local_model is None and self.self_attn is None:
            raise ValueError("GPSLayer needs a local model or a global model")
        self.norm1_local = nn.BatchNorm1d(dim_h)
        self.norm1_attn = nn.BatchNorm1d(dim_h)
        self.ff_linear1 = nn.Linear(dim_h, dim_h * 2)
        self.ff_linear2 = nn.Linear(dim_h * 2, dim_h)
        self.norm2 = nn.BatchNorm1d(dim_h)
        self._param_names = [n for n, _ in self.named_parameters()]
        self._grad_shapes = [tuple(p.shape) for _, p in self.named_parameters()]
        self._grad_sizes = [p.numel() for _, p in self.named_parameters()]
        self._grad_numel = sum(self._grad_sizes)
        self._plan_cache = {}

    # ------------------------------------------------------------------ operand planes across layers / steps
    def _handoff_args(self, args, plan, params, x, e, x_out, e_out):
        """Fills the ABI-3 plane fields: (i) the bf16 hi/lo planes of x / edge_attr that the previous GPSLayer of the
        model wrote next to its outputs (gps_model.py:100,105-108 chains the layers on one batch object), so this layer
        skips converting its inputs; (ii) plane buffers for this layer's own outputs; (iii) the persistent weight-plane
        buffer, re-packed only when a parameter changed (once per optimiser step, not once per forward call).
        Returns what backward needs to see again, and keeps the buffers alive through the autograd node."""
        if plan[2] <= 0 or not self.__dict__.get("plane_handoff", True):
            return None
        dev = x.device
        lo = self.precision == "fp32"

        def planes_of(t):
            buf = torch.empty((2 if lo else 1, t.shape[0], (t.shape[1] + 7) // 8 * 8), dtype=torch.bfloat16, device=dev)
            return buf, _lib.GpsPlanes(buf[0].data_ptr(), buf[1].data_ptr() if lo else 0, buf.shape[2])

        keep = []
        zero = _lib.GpsPlanes(0, 0, 0)
        xin, ein = zero, zero
        src = self.__dict__.pop("_planes_in", None) or {}
        for name, t in (("x", x), ("e", e)):
            h = src.get(name)
            if h is not None and h[0] == (t.data_ptr(), t._version, tuple(t.shape), lo):
                keep.append(h[1])
                pl = _lib.GpsPlanes(h[1][0].data_ptr(), h[1][1].data_ptr() if lo else 0, h[1].shape[2])
                if name == "x":
                    xin = pl
                else:
                    ein = pl
        args.x_planes_in, args.e_planes_in = xin, ein
        out = {}
        xb, args.x_planes_out = planes_of(x_out)
        out["x"] = (x_out, xb)
        if e_out is not None:
            eb, args.e_planes_out = planes_of(e_out)
            out["e"] = (e_out, eb)
        self.__dict__["_planes_out"] = out
        # persistent weight planes
        key = (tuple((p.data_ptr(), p._version) for p in params), self.precision, plan[2])
        wp = self.__dict__.get("_wplanes")
        if wp is None or wp[0].numel() < plan[2] or wp[0].device != dev:
            wp = [torch.empty(plan[2] + 256, dtype=torch.uint8, device=dev), None]
            self.__dict__["_wplanes"] = wp
        args.wplanes, args.wplanes_bytes = wp[0].data_ptr(), wp[0].numel()
        capturing = torch.cuda.is_current_stream_capturing()
        args.wplanes_valid = 1 if (wp[1] == key and not capturing) else 0   # a captured graph always re-packs
        wp[1] = key
        keep.append(wp[0])
        return (xin, ein, args.wplanes, args.wplanes_bytes, keep)

    def _bucket_grads(self, named):
        """{name: .grad view} when every parameter's .grad is a view of this layer's static bucket, else None."""
        b = self.__dict__.get("_grad_bucket")
        if b is None:
            return None
        lo, hi = b
        out = {}
        for n, p in self.named_parameters():
            g = p.grad
            if g is None or not (lo <= g.data_ptr() < hi) or not g.is_contiguous():
                return None
            out[n] = g
        return out

    def _plan(self, args, gs):
        """(saved_bytes, workspace_bytes); gps_layer_plan is pure in (config, N, E, B, training, precision)."""
        key = (gs.N, gs.E, gs.B, bool(self.training), self.precision, float(self.dropout), float(self.attn_dropout))
        hit = self._plan_cache.get(key)
        if hit is None:
            plan = _lib.GpsLayerPlan()
            _lib.check(_lib.load().gps_layer_plan(C.byref(args), C.byref(plan)), "gps_layer_plan")
            hit = (int(plan.saved_bytes), int(max(plan.fwd_workspace_bytes, plan.bwd_workspace_bytes)),
                   int(plan.wplanes_bytes))
            if len(self._plan_cache) > 64:
                self._plan_cache.clear()
            self._plan_cache[key] = hit
        return hit

    # ------------------------------------------------------------------------------------
    def _base_args(self, gs, named, grads=None):
        """GpsLayerArgs with configuration, graph and parameter (+gradient) pointers filled in.

        The forward-direction struct (no gradient pointers) only depends on the parameter addresses and the
        module flags, so it is cached and copied; building ~30 nested ctypes structs per call costs more host
        time than the GPU needs for the whole layer at the ZINC shape."""
        if grads is None:
            key = (tuple(t.data_ptr() for t in named.values()), self.training, self.precision,
                   float(self.dropout), float(self.attn_dropout))
            cached = self.__dict__.get("_args_cache")
            if cached is None or cached[0] != key:
                self._check_params(named)
                cached = (key, self._build_args(named, None))
                self.__dict__["_args_cache"] = cached
            a = _lib.GpsLayerArgs.from_buffer_copy(cached[1])
        else:
            a = self._build_args(named, grads)
        a.seed = int(torch.initial_seed()) & 0xFFFFFFFFFFFFFFFF
        _dropout_calls[0] += 1
        a.offset = _dropout_calls[0] * 4096
        a.graph = gs.desc
        return a

    def _check_params(self, named):
        """The library reads raw fp32 device pointers: refuse anything else (the reference would cast or raise)."""
        bufs = {n: b for n, b in self.named_buffers() if b.is_floating_point()}
        for n, t in list(named.items()) + list(bufs.items()):
            if t.dtype != torch.float32 or not t.is_cuda or not t.is_contiguous():
                raise TypeError(f"graphgps_b200.GPSLayer: parameter/buffer '{n}' must be a contiguous float32 CUDA "
                                f"tensor (got {t.dtype} on {t.device})")

    def _build_args(self, named, grads):
        g = grads or {}
        a = _lib.GpsLayerArgs()
        a.d, a.heads = self.dim_h, self.num_heads
        a.local_type = _lib.LOCAL[self.local_gnn_type]
        a.global_type = _lib.GLOBAL[self.global_model_type]
        a.act = _lib.ACT[self.act]
        a.training = 1 if self.training else 0
        a.precision = _lib.PRECISION[self.precision]
        a.dropout, a.attn_dropout = float(self.dropout), float(self.attn_dropout)

        def lin(prefix, bias=True):
            return _lin(named[prefix + ".weight"], named.get(prefix + ".bias") if bias else None,
                        g.get(prefix + ".weight"), g.get(prefix + ".bias") if bias else None)

        def bn(prefix, mod):
            return _lib.GpsBatchNorm(_lib.ptr(named[prefix + ".weight"]), _lib.ptr(named[prefix + ".bias"]),
                                     _lib.ptr(mod.running_mean), _lib.ptr(mod.running_var),
                                     _lib.ptr(mod.num_batches_tracked),
                                     _lib.ptr(g.get(prefix + ".weight")), _lib.ptr(g.get(prefix + ".bias")))

        if self.local_gnn_type == "CustomGatedGCN":
            a.gcn_A, a.gcn_B, a.gcn_C = lin("local_model.A"), lin("local_model.B"), lin("local_model.C")
            a.gcn_D, a.gcn_E = lin("local_model.D"), lin("local_model.E")
            a.bn_node_x = bn("local_model.bn_node_x", self.local_model.bn_node_x)
            a.bn_edge_e = bn("local_model.bn_edge_e", self.local_model.bn_edge_e)
            if self._es:
                a.reserved1 |= _lib.ES_FLAG
                a.es_r0, a.es_r1 = lin("local_model.mlp_r_ij.0"), lin("local_model.mlp_r_ij.2")
        elif self.local_gnn_type == "GINE":
            a.gine_lin0, a.gine_lin1 = lin("local_model.nn.0"), lin("local_model.nn.2")
            a.gine_eps = float(self._gine_eps_host)
        elif self.local_gnn_type == "GCN":
            a.gcn_conv = _lin(named["local_model.lin.weight"], named["local_model.bias"],
                              g.get("local_model.lin.weight"), g.get("local_model.bias"))
        if self.global_model_type == "Transformer":
            a.attn_in = _lin(named["self_attn.in_proj_weight"], named["self_attn.in_proj_bias"],
                             g.get("self_attn.in_proj_weight"), g.get("self_attn.in_proj_bias"))
            a.attn_out = lin("self_attn.out_proj")
        elif self.global_model_type == "Performer":
            a.perf_q, a.perf_k, a.perf_v = (lin("self_attn.to_q", False), lin("self_attn.to_k", False),
                                            lin("self_attn.to_v", False))
            a.attn_out = lin("self_attn.to_out")
            pm = self.self_attn.fast_attention.projection_matrix
            a.perf_proj, a.perf_features, a.perf_dim_head = pm.data_ptr(), pm.shape[0], pm.shape[1]
        a.norm1_local = bn("norm1_local", self.norm1_local)
        a.norm1_attn = bn("norm1_attn", self.norm1_attn)
        a.norm2 = bn("norm2", self.norm2)
        a.ff1, a.ff2 = lin("ff_linear1"), lin("ff_linear2")
        return a

    @property
    def _gine_eps_host(self):
        # eps is a constant buffer (train_eps=False); read once, no per-step sync
        v = self.__dict__.get("_gine_eps_cache")
        if v is None:
            v = float(self.local_model.eps.item())
            self.__dict__["_gine_eps_cache"] = v
        return v

    def forward(self, batch):
        x = batch.x
        if not x.is_cuda:
            raise RuntimeError("graphgps_b200.GPSLayer runs on CUDA tensors only; there is no CPU fallback "
                               "(use the oracle under oracle/ for CPU checks)")
        if x.dtype != torch.float32:
            raise TypeError("batch.x must be float32")
        x = x.contiguous()
        e = getattr(batch, "edge_attr", None)
        if self.local_gnn_type in _EDGE_LOCAL:
            if e is None or e.shape[-1] != self.dim_h:
                raise ValueError("Node and edge feature dimensionalities do not match")
            if e.dtype != torch.float32 or e.device != x.device:
                raise TypeError("batch.edge_attr must be float32 on the device of batch.x")
            e = e.contiguous()
        else:
            e = None
        pe = self._pe_of(batch, x) if self._es else x.new_empty(0)
        gs = graph_of(batch)
        params = [p for _, p in self.named_parameters()]
        e_arg = e if e is not None else x.new_empty(0)
        self.__dict__["_planes_in"] = _batch_planes_get(batch)
        out = _GPSLayerFn.apply(self, gs, x, e_arg, pe, *params)
        produced = self.__dict__.pop("_planes_out", None)
        if self.local_gnn_type == "CustomGatedGCN":
            batch.x, batch.edge_attr = out           # gps_layer.py:173-174, :231
        else:
            batch.x = out
        _batch_planes_put(batch, produced, self.precision == "fp32")
        return batch

    @staticmethod
    def _pe_of(batch, x):
        """batch.pe_EquivStableLapPE (a missing attribute raises, as in the reference: gps_layer.py:166): [N, k] float32,
        contiguous, on the device of batch.x.  Its gradient flows back to the PE encoder."""
        pe = batch.pe_EquivStableLapPE
        if not torch.is_tensor(pe) or pe.dtype != torch.float32 or pe.device != x.device:
            raise TypeError("batch.pe_EquivStableLapPE must be a float32 tensor on the device of batch.x")
        if pe.dim() != 2 or pe.shape[0] != x.shape[0] or pe.shape[1] == 0:
            raise ValueError(f"batch.pe_EquivStableLapPE must be [N={x.shape[0]}, k>0] (got {tuple(pe.shape)})")
        if not pe.is_contiguous():
            raise ValueError("batch.pe_EquivStableLapPE must be contiguous")
        return pe

    def extra_repr(self):
        return (f"summary: dim_h={self.dim_h}, local_gnn_type={self.local_gnn_type}, "
                f"global_model_type={self.global_model_type}, heads={self.num_heads}, "
                f"{'equivstable_pe=True, ' if self._es else ''}"
                f"backend=libgps_b200(sm_100a), precision={self.precision}")
