"""pcompanion_b200 - B200-native implementation of the P-Companion data-parallel hot path.

Public surface mirrors the reference (emreatilgan/P-Companion): ``Product2Vec``,
``ComplementaryTypeTransition``, ``ComplementaryItemPrediction``, ``PCompanion``,
``BehaviorProductGraph``, ``Metrics``.  Importing the package loads the C-ABI CUDA library
(pcompanion_b200/csrc/libpcompanion_b200.so) and fails loudly if it is missing.
"""
from . import _lib  # noqa: F401  (loads the shared library, raises NativeLibraryError if absent)
from . import ops
from .bpg import BehaviorProductGraph
from .p_companion import ComplementaryItemPrediction, ComplementaryTypeTransition, PCompanion
from .product2vec import Product2Vec
from .retrieval import CatalogIndex, Exclusions, Metrics, ShardedCatalog
from .data import ComplementaryDataset, GraphTripletSampler, SimilarityDataset, TripletBatch, collate_fn
from .inference import PCompanionInference
from .graphs import GraphedTrainStep

__all__ = ["ops", "BehaviorProductGraph", "Product2Vec", "ComplementaryTypeTransition",
           "ComplementaryItemPrediction", "PCompanion", "Metrics", "CatalogIndex", "Exclusions", "ShardedCatalog",
           "SimilarityDataset", "ComplementaryDataset", "collate_fn", "GraphTripletSampler", "TripletBatch", "PCompanionInference", "GraphedTrainStep"]
