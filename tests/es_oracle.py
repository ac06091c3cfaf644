"""TEST INFRASTRUCTURE: the CPU oracle (oracle/gps_oracle.py) extended by the EquivStableLapPE edge gate of the
GatedGCN local model, graphgps/layer/gatedgcn_layer.py:29-35 (mlp_r_ij), :63-70 (PE = batch.pe_EquivStableLapPE) and
:99-103 (r_ij = ||PE_i - PE_j||^2, sigma_ij = sigmoid(e_ij) * mlp_r_ij(r_ij)).

The plain oracle stays as it is; this module subclasses it.  Pinned against the reference's own layer files by
tests/test_eslappe.py::test_oracle_equals_reference_live_es (tests/golden/reference/eslappe_live.pt, written by
tests/golden/make_golden_eslappe.py)."""
import torch
import torch.nn as nn
import torch.nn.functional as F

from oracle.gps_oracle import _ACTS, OracleGatedGCN, OracleGPSLayer


class OracleGatedGCNES(OracleGatedGCN):
    """OracleGatedGCN with mlp_r_ij = Linear(1,d), act, Linear(d,1), Sigmoid.  The layer hands it the batch's PE in
    `self.pe` before each call (the plain oracle's call signature has no PE argument)."""

    def __init__(self, dim, dropout, act="relu"):
        super().__init__(dim, dropout, act)
        self.mlp_r_ij = nn.Sequential(nn.Linear(1, dim), _ACTS[act](), nn.Linear(dim, 1), nn.Sigmoid())
        self.pe = None

    def forward(self, x, e, edge_index):
        src, dst = edge_index[0], edge_index[1]
        x_in, e_in = x, e
        Ax, Bx, Ce, Dx, Ex = self.A(x), self.B(x), self.C(e), self.D(x), self.E(x)
        e_ij = Dx[dst] + Ex[src] + Ce
        r_ij = ((self.pe[dst] - self.pe[src]) ** 2).sum(dim=-1, keepdim=True)      # :101
        sigma = torch.sigmoid(e_ij) * self.mlp_r_ij(r_ij)                        # :97, :102-103
        num = torch.zeros_like(Bx).index_add_(0, dst, sigma * Bx[src])
        den = torch.zeros_like(Bx).index_add_(0, dst, sigma)
        x = Ax + num / (den + 1e-6)
        x = self.act_fn_x(self.bn_node_x(x))
        e = self.act_fn_e(self.bn_edge_e(e_ij))
        x = F.dropout(x, self.dropout, training=self.training)
        e = F.dropout(e, self.dropout, training=self.training)
        return x_in + x, e_in + e


class OracleGPSLayerES(OracleGPSLayer):
    """OracleGPSLayer(..., equivstable_pe=True): GatedGCN gates its messages with the batch's PE; GCN and None never
    read it (gps_layer.py:163-184), so for them this is the plain oracle."""

    def __init__(self, dim_h, local_gnn_type, global_model_type, num_heads, act="relu", dropout=0.0,
                 attn_dropout=0.0):
        super().__init__(dim_h, local_gnn_type, global_model_type, num_heads, act=act, dropout=dropout,
                         attn_dropout=attn_dropout)
        if local_gnn_type == "CustomGatedGCN":
            self.local_model = OracleGatedGCNES(dim_h, dropout, act)

    def forward(self, batch):
        if isinstance(self.local_model, OracleGatedGCNES):
            self.local_model.pe = batch.pe_EquivStableLapPE      # a missing attribute raises, as at gps_layer.py:166
        try:
            return super().forward(batch)
        finally:
            if isinstance(self.local_model, OracleGatedGCNES):
                self.local_model.pe = None
