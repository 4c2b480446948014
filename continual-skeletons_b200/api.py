"""Public surface of the package."""
from .graph import Graph, kinetics_graph, ntu_graph
from .lib import CoskError, build_library, library_path, load_library
from .model import CoAGcn, CoModelBase, CoStack, CoSTr, CoStGcn, CoStGcnMod, BlockSpec, StreamMeta, StreamState
from .dist import LogitGather, all_gather_logits, any_rank, shard_range
from .ensemble import MultiStream, aggregate_preds

__all__ = [
    "Graph", "ntu_graph", "kinetics_graph",
    "CoskError", "build_library", "library_path", "load_library",
    "CoModelBase", "CoStack", "CoStGcn", "CoStGcnMod", "CoAGcn", "CoSTr", "BlockSpec", "StreamMeta", "StreamState",
    "all_gather_logits", "shard_range", "LogitGather", "any_rank",
    "MultiStream", "aggregate_preds",
]
