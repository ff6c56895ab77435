"""windgnn_b200 — B200-native (sm_100a) forward hot path of WindGNN.

Public surface (mirrors the reference's step5/step6 modules and step2 graph build):

    GCN_GRU, GraphConvLayer      drop-in nn.Modules (windgnn_b200.model)
    build_graph, knn_graph, ...  bit-exact graph build on the GPU (windgnn_b200.graph)
    ops.gcn_gru_forward, ...     torch custom ops over the C-ABI (windgnn_b200.ops)
    window_starts, forecast_targets  rolling-forecast windows for GCN_GRU.forecast (windgnn_b200.sequences)

CUDA only.  ``import windgnn_b200`` works without a GPU (so that the package can be built and
its host logic tested), but every compute call raises unless the in-tree library is built and a
CUDA device is present.
"""

from . import _lib, ops  # noqa: F401
from .model import GCN_GRU, GraphConvLayer  # noqa: F401
from .graph import (  # noqa: F401
    CsrGraph,
    build_graph,
    build_graph_from_latlon,
    knn_graph_csr,
    knn_graph_csr_from_latlon,
    knn_graph_from_latlon,
    mercator,
    synthetic_coordinates,
)

from .sequences import (  # noqa: F401
    create_sequences,
    denormalise_last_step,
    forecast_targets,
    num_windows,
    pivot_long_table,
    window_starts,
)

__all__ = [
    "pivot_long_table",
    "CsrGraph",
    "knn_graph_csr",
    "knn_graph_csr_from_latlon",
    "create_sequences",
    "denormalise_last_step",
    "num_windows",
    "window_starts",
    "forecast_targets",
    "GCN_GRU",
    "GraphConvLayer",
    "build_graph",
    "build_graph_from_latlon",
    "knn_graph_from_latlon",
    "mercator",
    "synthetic_coordinates",
    "ops",
]
