"""GraphGym-side glue for the drop-in (SURVEY.md section 8b, INTEGRATION.md section 1).

The reference instantiates ``GPSLayer`` directly in ``GPSModel.__init__`` (graphgps/network/gps_model.py:85-99,
imported at :9), so the drop-in is a rebinding of that module attribute (`install`).  GraphGym's own plugin
convention -- modules self-register with ``@register_layer(name)`` (graphgps/layer/gatedgcn_layer.py:139) -- is
served by `register`.  Neither function imports torch_geometric at module import time: this package must load
(and fail loudly on its own terms) on machines without PyG.
"""
from __future__ import annotations

import importlib

from .gps_layer import GPSLayer


def install(gps_model_module=None):
    """Rebind ``GPSLayer`` inside ``graphgps.network.gps_model`` so ``create_model()`` builds the B200 layer.

    Call after ``import graphgps`` and before ``create_model()`` (main.py:144).  Returns the class it replaced so a
    caller can restore it."""
    if gps_model_module is None:
        gps_model_module = importlib.import_module("graphgps.network.gps_model")
    previous = getattr(gps_model_module, "GPSLayer", None)
    gps_model_module.GPSLayer = GPSLayer
    return previous


def register(name="gpslayer_b200"):
    """Register a LayerConfig-style wrapper under ``name`` in GraphGym's layer registry.

    Raises ``RuntimeError`` when torch_geometric.graphgym is not importable, and (from GraphGym itself) ``KeyError``
    when the name is already taken."""
    try:
        register_mod = importlib.import_module("torch_geometric.graphgym.register")
        cfg = importlib.import_module("torch_geometric.graphgym.config").cfg
    except ImportError as e:  # pragma: no cover - depends on the host environment
        raise RuntimeError("torch_geometric.graphgym is not importable; use graphgps_b200.graphgym.install() or "
                           "construct graphgps_b200.GPSLayer directly") from e

    class GPSLayerB200GraphGym(GPSLayer):
        """dim_in == dim_out == cfg.gt.dim_hidden; layer types split as in gps_model.py:80."""

        def __init__(self, layer_config, **kwargs):
            local, glob = cfg.gt.layer_type.split("+")
            # gps_model.py:92: equivstable_pe=cfg.posenc_EquivStableLapPE.enable (absent section: off)
            es = getattr(getattr(cfg, "posenc_EquivStableLapPE", None), "enable", False)
            kwargs.setdefault("equivstable_pe", bool(es))
            super().__init__(dim_h=layer_config.dim_out, local_gnn_type=local, global_model_type=glob,
                             num_heads=cfg.gt.n_heads, act=cfg.gnn.act, dropout=cfg.gt.dropout,
                             attn_dropout=cfg.gt.attn_dropout, layer_norm=cfg.gt.layer_norm,
                             batch_norm=cfg.gt.batch_norm, **kwargs)

    register_mod.register_layer(name, GPSLayerB200GraphGym)
    return GPSLayerB200GraphGym
