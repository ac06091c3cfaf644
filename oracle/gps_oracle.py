"""TEST INFRASTRUCTURE — CPU restatement (pure torch) of the reference GPSLayer hot path.

Only tests/, bench.py's ``cpu_baseline`` / ``--impl reference`` legs and
``__graft_entry__.smoke()`` may import this file.  The product package (graphgps_b200/) never
does; it fails loudly when its CUDA library is missing.

PARITY PINNING.  The reference's own tests hold *no* golden vectors for this path (SURVEY.md
section 4 / 8c: "parity unpinned" by the reference).  This restatement is therefore pinned against
outputs of the reference itself: ``tests/test_oracle.py::test_oracle_equals_reference_live`` asserts
equality of this file in fp64 with the reference's own layer files run verbatim (oracle/ref_shim.py) by
tests/golden/make_golden.py, kept in tests/golden/reference/ as seeded samples and full-tensor sums
(<=1e-10 outputs, <=1e-9 gradients), forward and backward, for seven variants;
``test_oracle_matches_golden_fp64`` / ``test_oracle_fp32_close_to_golden`` pin it to the fixtures (2e-6 / 5e-4); and
``tests/golden/*.pt`` (made by tests/golden/make_golden.py from the reference-verbatim layer in
fp64) travel to the GPU box.  The published parameter totals (README.md:77-79 of the reference)
are checked as shape KATs.

What is restated, each following the cited reference lines (paths relative to /root/reference):
  * GPSLayer.forward composition ............ graphgps/layer/gps_layer.py:155-232, 234-257
  * GatedGCNLayer forward/message/aggregate . graphgps/layer/gatedgcn_layer.py:45-136
  * GINEConv (PyG 2.2, third party) ......... maths evidenced by graphgps/layer/gine_conv_layer.py:56-84
  * GCNConv (PyG 2.2, third party, source not under /root/reference; call site gps_layer.py:49-51,186):
                                              published algorithm (Kipf & Welling; PyG gcn_norm with
                                              add_remaining_self_loops) -- pinned only to oracle/ref_shim.py's
                                              message-passing restatement of the same algorithm, not to PyG itself
  * to_dense_batch (PyG 2.2, third party) ... SURVEY.md Appendix A; call site gps_layer.py:199
  * Performer SelfAttention / FAVOR+ ........ graphgps/layer/performer_layer.py:119-144 (softmax_kernel),
                                              :163-195 (projection), :200-205 (linear_attention),
                                              :421-508 (Attention.forward)
torch's own nn.Linear / nn.BatchNorm1d / nn.MultiheadAttention are used as-is: they ARE the
reference's arithmetic for those ops (gps_layer.py:104-106,136-151).
"""
from __future__ import annotations

import math

import torch
import torch.nn as nn
import torch.nn.functional as F

_ACTS = {"relu": nn.ReLU, "gelu": nn.GELU}


def to_dense_batch(x, batch, num_graphs=None):
    """PyG to_dense_batch (SURVEY Appendix A). Returns ([B,Nmax,d], mask [B,Nmax])."""
    B = int(batch.max()) + 1 if num_graphs is None else num_graphs
    n = torch.bincount(batch, minlength=B)
    ptr = torch.zeros(B + 1, dtype=torch.int64, device=x.device)
    ptr[1:] = torch.cumsum(n, 0)
    nmax = int(n.max())
    idx = torch.arange(x.shape[0], device=x.device) - ptr[batch] + batch * nmax
    out = x.new_zeros((B * nmax,) + tuple(x.shape[1:]))
    out[idx] = x
    mask = torch.zeros(B * nmax, dtype=torch.bool, device=x.device)
    mask[idx] = True
    return out.view(B, nmax, *x.shape[1:]), mask.view(B, nmax)


class OracleGatedGCN(nn.Module):
    """gatedgcn_layer.py:11-136 with residual=True (as built at gps_layer.py:92-96)."""

    def __init__(self, dim, dropout, act="relu"):
        super().__init__()
        self.A = nn.Linear(dim, dim)
        self.B = nn.Linear(dim, dim)
        self.C = nn.Linear(dim, dim)
        self.D = nn.Linear(dim, dim)
        self.E = nn.Linear(dim, dim)
        self.bn_node_x = nn.BatchNorm1d(dim)
        self.bn_edge_e = nn.BatchNorm1d(dim)
        self.act_fn_x = _ACTS[act]()
        self.act_fn_e = _ACTS[act]()
        self.dropout = dropout

    def forward(self, x, e, edge_index):
        src, dst = edge_index[0], edge_index[1]          # j = source, i = target (Appendix A)
        x_in, e_in = x, e                                  # :52-54
        Ax, Bx, Ce, Dx, Ex = self.A(x), self.B(x), self.C(e), self.D(x), self.E(x)   # :57-61
        e_ij = Dx[dst] + Ex[src] + Ce                      # :96
        sigma = torch.sigmoid(e_ij)                        # :97
        N = x.shape[0]
        num = torch.zeros_like(Bx).index_add_(0, dst, sigma * Bx[src])   # :117-119
        den = torch.zeros_like(Bx).index_add_(0, dst, sigma)             # :121-123
        x = Ax + num / (den + 1e-6)                        # :125, :133
        e = e_ij                                           # :106, :134 (pre-activation edge output)
        x = self.bn_node_x(x)                              # :72
        e = self.bn_edge_e(e)                              # :73
        x = self.act_fn_x(x)                               # :75
        e = self.act_fn_e(e)                               # :76
        x = F.dropout(x, self.dropout, training=self.training)   # :78
        e = F.dropout(e, self.dropout, training=self.training)   # :79
        return x_in + x, e_in + e                          # :81-83


class OracleGINE(nn.Module):
    """PyG GINEConv(gin_nn) as built at gps_layer.py:62-69; maths per gine_conv_layer.py:56-84."""

    def __init__(self, dim, act="relu"):
        super().__init__()
        self.nn = nn.Sequential(nn.Linear(dim, dim), _ACTS[act](), nn.Linear(dim, dim))
        self.register_buffer("eps", torch.Tensor([0.0]))

    def forward(self, x, edge_index, edge_attr):
        src, dst = edge_index[0], edge_index[1]
        msg = (x[src] + edge_attr).relu()
        out = torch.zeros_like(x).index_add_(0, dst, msg)
        out = out + (1 + self.eps) * x
        return self.nn(out)


class OracleGCN(nn.Module):
    """PyG 2.2 GCNConv(dim, dim) with default arguments as built at gps_layer.py:49-51:
    h = D^-1/2 (A' + I) D^-1/2 (x W^T) + b, A' = adjacency without self loops, D = 1 + in-degree under A'."""

    def __init__(self, dim):
        super().__init__()
        self.lin = nn.Linear(dim, dim, bias=False)
        nn.init.xavier_uniform_(self.lin.weight)
        self.bias = nn.Parameter(torch.zeros(dim))

    def forward(self, x, edge_index, edge_attr=None):
        N = x.shape[0]
        src, dst = edge_index[0], edge_index[1]
        keep = src != dst
        src, dst = src[keep], dst[keep]
        deg = torch.ones(N, dtype=x.dtype).index_add_(0, dst, torch.ones(dst.shape[0], dtype=x.dtype))
        dinv = deg.rsqrt()
        y = self.lin(x)
        agg = (dinv * dinv).unsqueeze(1) * y                                        # the self loop
        agg = agg.index_add(0, dst, (dinv[src] * dinv[dst]).unsqueeze(1) * y[src])
        return agg + self.bias


def gaussian_orthogonal_random_matrix(nb_rows, nb_columns, generator=None):
    """performer_layer.py:163-195 (scaling=0)."""
    blocks = []
    full = nb_rows // nb_columns
    for _ in range(full):
        q, _ = torch.linalg.qr(torch.randn(nb_columns, nb_columns, generator=generator), mode="reduced")
        blocks.append(q.t())
    rem = nb_rows - full * nb_columns
    if rem > 0:
        q, _ = torch.linalg.qr(torch.randn(nb_columns, nb_columns, generator=generator), mode="reduced")
        blocks.append(q.t()[:rem])
    final = torch.cat(blocks)
    mult = torch.randn(nb_rows, nb_columns, generator=generator).norm(dim=1)
    return torch.diag(mult) @ final


def softmax_kernel(data, projection_matrix, is_query, eps=1e-4):
    """performer_layer.py:119-144. data [b,h,n,dh], projection [m,dh]."""
    dn = data.shape[-1] ** -0.25
    ratio = projection_matrix.shape[0] ** -0.5
    proj = projection_matrix.to(data.dtype)
    dd = torch.einsum("bhid,jd->bhij", dn * data, proj)
    diag = ((data ** 2).sum(-1) / 2.0) * dn ** 2
    diag = diag.unsqueeze(-1)
    if is_query:
        return ratio * (torch.exp(dd - diag - torch.amax(dd, dim=-1, keepdim=True)) + eps)
    return ratio * (torch.exp(dd - diag - torch.amax(dd, dim=(-1, -2), keepdim=True)) + eps)


def linear_attention(q, k, v):
    """performer_layer.py:200-205."""
    k_cumsum = k.sum(dim=-2)
    d_inv = 1.0 / torch.einsum("bhnd,bhd->bhn", q, k_cumsum)
    context = torch.einsum("bhnd,bhne->bhde", k, v)
    return torch.einsum("bhde,bhnd,bhn->bhne", context, q, d_inv)


class _FastAttention(nn.Module):
    def __init__(self, dim_heads):
        super().__init__()
        nb = int(dim_heads * math.log(dim_heads))          # performer_layer.py:261
        self.register_buffer("projection_matrix", gaussian_orthogonal_random_matrix(nb, dim_heads))


class OraclePerformerSelfAttention(nn.Module):
    """performer_layer.py:421-508 with the ctor arguments of gps_layer.py:111-114
    (dim_head=64 default, qkv_bias=False, attn_out_bias=True, causal=False)."""

    def __init__(self, dim, heads, dropout=0.0, dim_head=64):
        super().__init__()
        inner = dim_head * heads
        self.heads = heads
        self.fast_attention = _FastAttention(dim_head)
        self.to_q = nn.Linear(dim, inner, bias=False)
        self.to_k = nn.Linear(dim, inner, bias=False)
        self.to_v = nn.Linear(dim, inner, bias=False)
        self.to_out = nn.Linear(inner, dim, bias=True)
        self.dropout = nn.Dropout(dropout)

    def forward(self, x, mask):
        b, n, _ = x.shape
        h = self.heads
        q, k, v = self.to_q(x), self.to_k(x), self.to_v(x)                    # :476
        q, k, v = (t.view(b, n, h, -1).transpose(1, 2) for t in (q, k, v))    # :478
        v = v.masked_fill(~mask[:, None, :, None], 0.0)                       # :485-487
        P = self.fast_attention.projection_matrix
        q = softmax_kernel(q, P, True)                                        # :313-315
        k = softmax_kernel(k, P, False)
        out = linear_attention(q, k, v)                                       # :318
        out = out.transpose(1, 2).reshape(b, n, -1)                           # :500
        return self.dropout(self.to_out(out))                                 # :501-502


class OracleGPSLayer(nn.Module):
    """Restatement of graphgps/layer/gps_layer.py:16-257 for
    local in {None, GINE, GCN, CustomGatedGCN} x global in {None, Transformer, Performer}, BatchNorm."""

    def __init__(self, dim_h, local_gnn_type, global_model_type, num_heads, act="relu",
                 pna_degrees=None, equivstable_pe=False, dropout=0.0, attn_dropout=0.0,
                 layer_norm=False, batch_norm=True, bigbird_cfg=None, log_attn_weights=False):
        super().__init__()
        assert not equivstable_pe and not layer_norm
        self.dim_h, self.num_heads = dim_h, num_heads
        self.local_gnn_type, self.global_model_type = local_gnn_type, global_model_type
        self.batch_norm = batch_norm
        if local_gnn_type == "None":
            self.local_model = None
        elif local_gnn_type == "GINE":
            self.local_model = OracleGINE(dim_h, act)
        elif local_gnn_type == "GCN":
            self.local_model = OracleGCN(dim_h)
        elif local_gnn_type == "CustomGatedGCN":
            self.local_model = OracleGatedGCN(dim_h, dropout, act)
        else:
            raise ValueError(f"Unsupported local GNN model: {local_gnn_type}")
        if global_model_type == "None":
            self.self_attn = None
        elif global_model_type == "Transformer":
            self.self_attn = nn.MultiheadAttention(dim_h, num_heads, dropout=attn_dropout,
                                                   batch_first=True)
        elif global_model_type == "Performer":
            self.self_attn = OraclePerformerSelfAttention(dim_h, num_heads, dropout=attn_dropout)
        else:
            raise ValueError(f"Unsupported global x-former model: {global_model_type}")
        if batch_norm:
            self.norm1_local = nn.BatchNorm1d(dim_h)
            self.norm1_attn = nn.BatchNorm1d(dim_h)
            self.norm2 = nn.BatchNorm1d(dim_h)
        self.dropout_local = nn.Dropout(dropout)
        self.dropout_attn = nn.Dropout(dropout)
        self.ff_linear1 = nn.Linear(dim_h, dim_h * 2)
        self.ff_linear2 = nn.Linear(dim_h * 2, dim_h)
        self.act_fn_ff = _ACTS[act]()
        self.ff_dropout1 = nn.Dropout(dropout)
        self.ff_dropout2 = nn.Dropout(dropout)

    def forward(self, batch):
        h = batch.x
        h_in1 = h                                                            # :156-157
        outs = []
        if self.local_model is not None:
            if self.local_gnn_type == "CustomGatedGCN":
                h_local, e_out = self.local_model(h, batch.edge_attr, batch.edge_index)   # :163-174
                batch.edge_attr = e_out
            else:
                h_local = self.local_model(h, batch.edge_index, batch.edge_attr)    # :182-184
                h_local = self.dropout_local(h_local)                               # :188
                h_local = h_in1 + h_local                                           # :189
            if self.batch_norm:
                h_local = self.norm1_local(h_local)                                 # :194
            outs.append(h_local)
        if self.self_attn is not None:
            h_dense, mask = to_dense_batch(h, batch.batch, getattr(batch, "num_graphs", None))  # :199
            if self.global_model_type == "Transformer":
                h_attn = self.self_attn(h_dense, h_dense, h_dense, attn_mask=None,
                                        key_padding_mask=~mask, need_weights=False)[0][mask]   # :201,:238
            else:
                h_attn = self.self_attn(h_dense, mask=mask)[mask]                              # :206
            h_attn = self.dropout_attn(h_attn)                                      # :212
            h_attn = h_in1 + h_attn                                                 # :213
            if self.batch_norm:
                h_attn = self.norm1_attn(h_attn)                                    # :217
            outs.append(h_attn)
        h = sum(outs)                                                               # :222
        h = h + self.ff_dropout2(self.ff_linear2(self.ff_dropout1(self.act_fn_ff(self.ff_linear1(h)))))  # :225,:253-257
        if self.batch_norm:
            h = self.norm2(h)                                                       # :229
        batch.x = h
        return batch


def param_count(module):
    return sum(p.numel() for p in module.parameters())
