"""Duck-typed graph mini-batch + seeded synthetic generators for the BASELINE shapes.

PyG is not installed in this image, so the layer takes any object that exposes the
attributes the reference layer reads (graphgps/layer/gps_layer.py:155-232):
``x [N,d] f32``, ``edge_index [2,E] i64`` (row 0 = source j, row 1 = target i),
``edge_attr [E,d] f32`` and ``batch [N] i64`` (sorted, as PyG collation produces).
``GraphBatch`` additionally carries the host-side ints a PyG ``Batch`` also has
(``num_graphs``, ``ptr``) so the layer never needs a device->host sync.

Shapes follow SURVEY.md section 8(d): the per-dataset means come from the reference's
own run logs (final-results.zip, logging.log:7-9 of the pcqm4mv2 / zinc / ogbg-code2
runs); ranges are generator parameters.
"""
from __future__ import annotations

import dataclasses
from typing import Optional

import torch


class GraphBatch:
    """Attribute bag with the fields of a collated PyG ``Batch`` that GPSLayer touches."""

    def __init__(self, x, edge_index, edge_attr, batch, num_graphs=None, ptr=None, **extra):
        self.x = x
        self.edge_index = edge_index
        self.edge_attr = edge_attr
        self.batch = batch
        self.num_graphs = num_graphs
        self.ptr = ptr
        for k, v in extra.items():
            setattr(self, k, v)

    # -- helpers mirroring torch_geometric.data.Batch ---------------------------------
    def _tensor_items(self):
        for k, v in list(self.__dict__.items()):
            if torch.is_tensor(v):
                yield k, v

    def to(self, device, non_blocking: bool = False):
        for k, v in self._tensor_items():
            setattr(self, k, v.to(device, non_blocking=non_blocking))
        # cached device-side graph structure (graphgps_b200.graph) is device specific
        self.__dict__.pop("_gps_b200_graph", None)
        return self

    def pin_memory(self):
        for k, v in self._tensor_items():
            setattr(self, k, v.pin_memory())
        return self

    def clone(self):
        out = GraphBatch.__new__(GraphBatch)
        for k, v in self.__dict__.items():
            if k == "_gps_b200_graph":
                continue
            out.__dict__[k] = v.clone() if torch.is_tensor(v) else v
        return out

    @property
    def num_nodes(self):
        return int(self.x.shape[0])

    @property
    def num_edges(self):
        return int(self.edge_index.shape[1])

    def __repr__(self):
        return (f"GraphBatch(N={self.num_nodes}, E={self.num_edges}, B={self.num_graphs}, "
                f"d={self.x.shape[1]})")


@dataclasses.dataclass(frozen=True)
class ShapeSpec:
    """Generator parameters of one BASELINE.json config (SURVEY.md section 8d)."""
    name: str
    num_graphs: int
    dim: int
    heads: int
    n_mean: float
    n_std: float
    n_min: int
    n_max: int
    # undirected extra (ring-closing) edges per node on top of a spanning tree
    extra_edges_per_node: float
    symmetric: bool          # store (i,j),(j,i) pairs (molecules) or a directed tree (code2 AST)
    lognormal: bool = False  # heavy-tailed node counts (code2)
    local_gnn: str = "CustomGatedGCN"
    global_model: str = "Transformer"
    layers: int = 1


# C1..C5 of SURVEY.md 8(d) / BASELINE.json "configs".
SHAPES = {
    # C1: "ZINC GPS(GINE+Transformer) d=64 batch=32 on CPU"
    "zinc-gine": ShapeSpec("zinc-gine", 32, 64, 4, 23.16, 4.5, 9, 37, 0.118, True,
                           local_gnn="GINE", layers=10),
    # C2: zinc-GPS+RWSE.yaml, BASELINE labels it GatedGCN+Transformer
    "zinc-gatedgcn": ShapeSpec("zinc-gatedgcn", 32, 64, 4, 23.16, 4.5, 9, 37, 0.118, True,
                               layers=10),
    # C3: pcqm4m-GPS+RWSE.yaml (GPS-small): the headline workload
    "pcqm4m-small": ShapeSpec("pcqm4m-small", 256, 304, 4, 14.14, 2.6, 1, 51, 0.101, True,
                              layers=5),
    # C4: pcqm4m-GPSmedium+RWSE.yaml shape with Performer (BASELINE)
    "pcqm4m-medium-performer": ShapeSpec("pcqm4m-medium-performer", 256, 384, 16, 14.14, 2.6,
                                         1, 51, 0.101, True, global_model="Performer",
                                         layers=10),
    # C5: ogbg-code2 shaped
    "code2": ShapeSpec("code2", 32, 256, 4, 125.0, 0.0, 11, 1000, 0.0, False, lognormal=True,
                       layers=4),
}


def _draw_sizes(spec: ShapeSpec, gen: torch.Generator) -> torch.Tensor:
    B = spec.num_graphs
    if spec.lognormal:
        # log-normal with the requested mean; sigma chosen for a heavy tail
        sigma = 0.8
        mu = torch.log(torch.tensor(spec.n_mean)) - sigma * sigma / 2
        n = torch.exp(mu + sigma * torch.randn(B, generator=gen))
    else:
        n = spec.n_mean + spec.n_std * torch.randn(B, generator=gen)
    return n.round().clamp(spec.n_min, spec.n_max).to(torch.int64)


def _graph_edges(n: int, spec: ShapeSpec, gen: torch.Generator) -> torch.Tensor:
    """Directed edge list [2, e] of one graph with local node ids."""
    if n <= 1:
        return torch.zeros(2, 0, dtype=torch.int64)
    # random spanning tree: node k attaches to a uniformly drawn earlier node
    child = torch.arange(1, n, dtype=torch.int64)
    parent = (torch.rand(n - 1, generator=gen) * child.to(torch.float32)).floor().to(torch.int64)
    und = {(int(min(a, b)), int(max(a, b))) for a, b in zip(parent.tolist(), child.tolist())}
    n_extra = int(round(spec.extra_edges_per_node * n))
    tries = 0
    while n_extra > 0 and tries < 20 * n and n > 2:
        tries += 1
        a, b = torch.randint(0, n, (2,), generator=gen).tolist()
        if a == b:
            continue
        key = (min(a, b), max(a, b))
        if key in und:
            continue
        und.add(key)
        n_extra -= 1
    pairs = sorted(und)
    if spec.symmetric:
        # (i,j),(j,i) interleaved, NOT sorted by destination (OGB/PyG molecule collation)
        src = [v for a, b in pairs for v in (a, b)]
        dst = [v for a, b in pairs for v in (b, a)]
    else:
        # directed tree: parent -> child (AST edges)
        src = [a for a, b in pairs]
        dst = [b for a, b in pairs]
    return torch.tensor([src, dst], dtype=torch.int64)


def make_batch(shape, seed: int = 0, dim: Optional[int] = None,
               num_graphs: Optional[int] = None, dtype=torch.float32) -> GraphBatch:
    """Seeded synthetic batch of the named BASELINE shape (CPU tensors)."""
    spec = SHAPES[shape] if isinstance(shape, str) else shape
    if num_graphs is not None:
        spec = dataclasses.replace(spec, num_graphs=num_graphs)
    d = spec.dim if dim is None else dim
    gen = torch.Generator().manual_seed(seed)
    sizes = _draw_sizes(spec, gen)
    ptr = torch.zeros(spec.num_graphs + 1, dtype=torch.int64)
    ptr[1:] = torch.cumsum(sizes, 0)
    edges = []
    for g in range(spec.num_graphs):
        ei = _graph_edges(int(sizes[g]), spec, gen)
        edges.append(ei + ptr[g])
    edge_index = torch.cat(edges, dim=1) if edges else torch.zeros(2, 0, dtype=torch.int64)
    N = int(ptr[-1])
    E = int(edge_index.shape[1])
    x = torch.randn(N, d, generator=gen, dtype=torch.float32).to(dtype)
    edge_attr = torch.randn(E, d, generator=gen, dtype=torch.float32).to(dtype)
    batch = torch.repeat_interleave(torch.arange(spec.num_graphs, dtype=torch.int64), sizes)
    return GraphBatch(x=x, edge_index=edge_index, edge_attr=edge_attr, batch=batch,
                      num_graphs=spec.num_graphs, ptr=ptr)


def batch_from_lists(sizes, edge_lists, d, seed=0) -> GraphBatch:
    """Hand-built batch for edge-case tests: ``edge_lists[g]`` = list of (src, dst) local ids."""
    gen = torch.Generator().manual_seed(seed)
    sizes_t = torch.tensor(list(sizes), dtype=torch.int64)
    B = len(sizes)
    ptr = torch.zeros(B + 1, dtype=torch.int64)
    ptr[1:] = torch.cumsum(sizes_t, 0)
    src, dst = [], []
    for g, el in enumerate(edge_lists):
        for a, b in el:
            src.append(a + int(ptr[g]))
            dst.append(b + int(ptr[g]))
    edge_index = torch.tensor([src, dst], dtype=torch.int64).reshape(2, -1)
    N, E = int(ptr[-1]), edge_index.shape[1]
    x = torch.randn(N, d, generator=gen)
    edge_attr = torch.randn(E, d, generator=gen)
    batch = torch.repeat_interleave(torch.arange(B, dtype=torch.int64), sizes_t)
    return GraphBatch(x=x, edge_index=edge_index, edge_attr=edge_attr, batch=batch,
                      num_graphs=B, ptr=ptr)


def add_equivstable_pe(batch: GraphBatch, dim: Optional[int] = None, seed: int = 0, max_freqs: int = 8,
                       scale: float = 1.0) -> GraphBatch:
    """Attaches an encoder-like ``pe_EquivStableLapPE`` [N, dim] (default dim = batch.x's width) to ``batch``.

    Stands in for the EquivStableLapPE encoder's output (graphgps/encoder/equivstable_laplace_pos_encoder.py:46-49:
    Linear(max_freqs -> dim) over the Laplacian eigenvectors): per-graph L2-normalised random "eigenvector" columns
    [N, max_freqs] through a seeded Linear(max_freqs, dim) with torch's default init, times ``scale``.  Full scale with
    default mlp_r_ij weights saturates most edge gates near 1; scale 0.3 keeps them spread.  Uses its own generator, so
    the batch's other tensors (and ``make_batch``'s stream) are untouched."""
    d = int(batch.x.shape[1]) if dim is None else dim
    gen = torch.Generator().manual_seed(seed)
    N = batch.num_nodes
    ev = torch.randn(N, max_freqs, generator=gen)
    gid = batch.batch.cpu()
    B = int(batch.num_graphs) if batch.num_graphs is not None else (int(gid.max()) + 1 if N else 0)
    norm = torch.zeros(B, max_freqs).index_add_(0, gid, ev * ev).sqrt().clamp_min(1e-12)
    ev = ev / norm[gid]
    bound = 1.0 / max_freqs ** 0.5                       # nn.Linear's default init range
    w = (torch.rand(d, max_freqs, generator=gen) * 2 - 1) * bound
    b = (torch.rand(d, generator=gen) * 2 - 1) * bound
    pe = (ev @ w.t() + b) * scale
    batch.pe_EquivStableLapPE = pe.to(device=batch.x.device, dtype=batch.x.dtype)
    return batch
