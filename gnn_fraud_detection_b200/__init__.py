"""gnn_fraud_detection_b200 -- B200-native GAT message passing for aum2606/GNN-Fraud-Detection.

Only the hot path lives here: the drop-in ``GATConv`` layer (``nn``), the model classes that host it
(``models``), the CUDA-built graph structures (``graph``), the autograd glue over the C ABI
(``functional``), the fused operators around the layers -- train-mode BatchNorm tail, GRU head, masked BCE -- (``fused``),
the device-resident training step (``train_step``), multi-GPU partitioning (``partition``), the snapshot builder that
feeds the temporal configuration (``snapshot``), the neighbour sampler and its ``NeighborLoader`` drop-in for mini-batch
training and seed-set inference (``sampler``) and synthetic data generators (``synth``).
Importing the package does not load the CUDA library; the first layer call does, and raises if it is
missing (there is no CPU or PyTorch fallback).
"""
from . import _abi  # noqa: F401
from .graph import GLOBAL_CSR_CACHE, CSRCache, GraphCSR, build_csr  # noqa: F401
from .models import GAT, TemporalGNN  # noqa: F401
from .nn import GATConv  # noqa: F401
from .sampler import NeighborLoader, NeighborSampler  # noqa: F401
from .snapshot import create_temporal_subgraph, select_steps  # noqa: F401

__all__ = ["GATConv", "GAT", "TemporalGNN", "GraphCSR", "build_csr", "CSRCache", "GLOBAL_CSR_CACHE",
           "create_temporal_subgraph", "select_steps", "NeighborSampler", "NeighborLoader"]
__version__ = "0.1.0"
