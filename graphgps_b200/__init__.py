"""graphgps_b200 — B200 (sm_100a) implementation of the GraphGPS `GPSLayer` hot path.

Public surface (mirrors the reference's module boundary, SURVEY.md section 8b):
    GPSLayer      drop-in for graphgps.layer.gps_layer.GPSLayer
    GraphBatch    duck-typed stand-in for a collated PyG Batch (PyG is optional)
    make_batch    seeded synthetic batches of the BASELINE shapes
    add_equivstable_pe   attaches an encoder-like batch.pe_EquivStableLapPE (for equivstable_pe=True layers)
    GPSStack      the L-layer stack of a GPSModel (shared graph structure, plane hand-off, one gradient bucket, capture)
    GradBucket    static flat gradient storage + in-place / overlapped all-reduce (data parallel)
    BatchPrefetcher, collate   pinned pre-collated host batches, copy + graph-structure build ahead of the compute stream
"""
from .batch import GraphBatch, SHAPES, add_equivstable_pe, make_batch, batch_from_lists  # noqa: F401
from .gps_layer import GPSLayer  # noqa: F401
from .dp import GradBucket  # noqa: F401
from .stack import GPSStack  # noqa: F401
from .loader import BatchPrefetcher, collate  # noqa: F401

__all__ = ["GPSLayer", "GPSStack", "GradBucket", "GraphBatch", "BatchPrefetcher", "collate", "SHAPES", "make_batch",
           "batch_from_lists", "add_equivstable_pe"]
