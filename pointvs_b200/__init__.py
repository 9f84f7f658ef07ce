"""B200-native EGNN scoring path for PointVS (see DESIGN.md)."""
from .egnn import (EGNNLayer, PygLinearPass, SartorrasEGNN,  # noqa: F401
                   MultitaskSatorrasEGNN, PNNGeometricBase)
from .graph import (CSRGraph, PackedBatch, generate_edges,  # noqa: F401
                    radius_graph_batch, csr_from_edge_index)
from .base import PointNeuralNetworkBase, DEVICE  # noqa: F401
from .screening import Pocket, score_poses  # noqa: F401

__all__ = ['EGNNLayer', 'PygLinearPass', 'SartorrasEGNN',
           'MultitaskSatorrasEGNN', 'PNNGeometricBase', 'CSRGraph',
           'PackedBatch', 'generate_edges', 'radius_graph_batch',
           'csr_from_edge_index', 'PointNeuralNetworkBase', 'DEVICE',
           'Pocket', 'score_poses']
