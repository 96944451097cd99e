"""B200-native gated-GCN hot path (see DESIGN.md)."""

from ._lib import EdgError                               # noqa: F401
from .gcn import GraphConvolution, gcn_layer            # noqa: F401
from .gated import GatedGCNStack, StackOutput, GATE_ARCHS  # noqa: F401
from .graph import DepGraph, TriggerPairs, build_graph, graph_from_dense, pairs_from_ptr, tree_distance  # noqa: F401
from .segment import wordpiece_mean, transform_bmm, segments_from_transform, lr_pool, span_max  # noqa: F401
from .wire import PackedBatch, collate_packed, heads_from_adjacency, split_adjacency  # noqa: F401
from .optim import FusedAdam                             # noqa: F401
from .head import DenseHead, CrossEntropyLoss, cross_entropy, total_loss  # noqa: F401

__all__ = ["EdgError", "GraphConvolution", "gcn_layer", "GatedGCNStack", "StackOutput", "GATE_ARCHS", "DepGraph",
           "build_graph", "graph_from_dense", "tree_distance", "TriggerPairs", "pairs_from_ptr", "wordpiece_mean", "transform_bmm",
           "segments_from_transform", "lr_pool", "span_max", "PackedBatch", "collate_packed", "heads_from_adjacency",
           "split_adjacency", "FusedAdam",
           "DenseHead", "CrossEntropyLoss", "cross_entropy", "total_loss"]
