"""gnn_tableextraction_b200 -- B200-native (sm_100a) graph-convolution hot path of
AILab-UniFI/GNN-TableExtraction.

Public surface (mirrors /root/reference/src/components/graphs/models.py):
    GcnSAGELayer, GcnSAGE, WeightedMeanSAGELayer, MeanSAGE   -- drop-in nn.Modules
    PageGraphBatch, as_page_graph_batch                      -- the graph argument
    SageTrainer                                              -- fused train / inference step
    BatchCapacity                                            -- largest batch a capacity-captured step accepts
    PagePool                                                 -- a dataset's pages resident on the device; captured
                                                                passes gather their batches from it (plan_epoch)
    features.bbox_features                                   -- the 13 BBOX node features on the device
    CrossEntropyLoss, cross_entropy                          -- loss on the CUDA kernels
    metrics.precision_recall_f1                              -- per-class scores of an evaluation's confusion matrix
    ops                                                      -- tensor-level wrappers of include/gte.h

Everything computes through ``libgte_b200.so`` (hand-written CUDA, C ABI in
``include/gte.h``).  There is no CPU fallback: importing works anywhere, but the
first compute call raises if the library or a CUDA device is missing.
"""
from ._lib import GteError, LIB_PATH, lib  # noqa: F401
from .graph import PageGraphBatch, as_page_graph_batch, batch_pages_host  # noqa: F401
from .nn import CrossEntropyLoss, GcnSAGE, GcnSAGELayer, MeanSAGE, WeightedMeanSAGELayer  # noqa: F401
from .layers import cross_entropy  # noqa: F401
from .engine import BatchCapacity, EvalCapture, SageTrainer  # noqa: F401
from .pool import PagePool  # noqa: F401
from . import features, metrics, ops, synth  # noqa: F401
from .metrics import precision_recall_f1  # noqa: F401

__all__ = [
    "GcnSAGELayer", "GcnSAGE", "WeightedMeanSAGELayer", "MeanSAGE", "CrossEntropyLoss", "cross_entropy",
    "PageGraphBatch", "as_page_graph_batch", "batch_pages_host", "SageTrainer", "BatchCapacity", "EvalCapture",
    "PagePool", "ops", "synth", "metrics", "precision_recall_f1", "GteError", "lib",
]
