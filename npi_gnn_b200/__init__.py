"""npi_gnn_b200 -- B200-native (sm_100a) hot path of NPI-GNN.

Drop-in surface (same names as the reference's imports, SURVEY.md 8b):
    from npi_gnn_b200 import Net_1, SAGEConv, TopKPooling, global_mean_pool, global_max_pool
    from npi_gnn_b200 import Data, DataLoader, LncRNA_Protein_Interaction_dataset_1hop_1220_InMemory
Native surface: BipartiteGraph, PairSet, Engine, Trainer, Scorer, Explainer.
All compute goes through the C ABI of libnpi.so (include/npi.h); nothing falls back to the CPU.
"""
from ._lib import NPIError  # noqa: F401
from .graph import BipartiteGraph, PairSet  # noqa: F401
from .engine import Engine, FlatParams  # noqa: F401
from .trainer import Trainer, Scorer, Explainer, group_rank_metrics, metrics, rank_metrics, top_k_by_group  # noqa: F401
from .nn import Net_1, SAGEConv, TopKPooling, global_max_pool, global_mean_pool  # noqa: F401
from .data import (Data, Batch, DataLoader, EnclosingSubgraphDataset,  # noqa: F401
                   LncRNA_Protein_Interaction_dataset_1hop_1220_InMemory)

__version__ = "0.1.0"
