"""hypergraphembedding_b200 -- B200-native HOBE (HG2V_ALG_DIST) hot path.

Drop-in replacements for the reference's ``algebraic_distance``, ``hg2v_weighting`` and
``hg2v_sample`` entry points, backed by hand-written sm_100a CUDA kernels behind a C ABI
(include/hge_b200.h, libhge_b200.so).  Importing the package does not need a GPU; calling
any compute entry point does, and fails loudly otherwise.
"""
from .hypergraph_pb2 import (EvaluationMetrics, ExperimentalResult, Hypergraph,
                             HypergraphEmbedding)
from .hypergraph_util import (AddNodeToEdge, CompressRange, IsEmpty, Relabel, ToCsrMatrix,
                              ToEdgeCsrMatrix)
from .algebraic_distance import EmbedAlgebraicDistance
from .hg2v_sample import (AlgebraicDistanceSamples, AlgebraicDistanceSamplesCsr,
                          AlgebraicDistanceSamplesDevice, BooleanSamples, BooleanSamplesCsr,
                          BooleanSamplesDevice, DeviceSampleColumns,
                          SampleColumns, SamplesToModelInput, SimilarityRecord,
                          SparseWeightedJaccard, WeightedJaccardSamples,
                          WeightedJaccardSamplesDevice)
from .hg2v_model import BooleanModel, KerasModelToEmbedding, UnweightedFloatModel
from .embedding import (EMBEDDING_OPTIONS, EmbedHg2vAdjJaccard, EmbedHg2vAdjJaccardDevice,
                        EmbedHg2vAlgDist, EmbedHg2vAlgDistDevice, EmbedHg2vBoolean,
                        EmbedHg2vBooleanDevice, EmbedHg2vNeighborhoodWeightedJaccard,
                        EmbedHg2vNeighborhoodWeightedJaccardDevice, EmbedNMFDevice, EmbedNode2VecCliqueDevice,
                        EmbedNode2VecDevice, EmbedSVDDevice)
from .nmf import NonNegativeFactorizationDevice
from .node2vec import Node2VecCliqueDevice, Node2VecDevice
from .svd import TruncatedSVDDevice
from .hg2v_weighting import (AlphaScaleValues, ComputeSpans, DictToSparseRow, OneMinusValues,
                             UniformWeight, WeightByAlgebraicSpan, WeightByDistance,
                             WeightByDistanceCluster, WeightByNeighborhood,
                             WeightBySameTypeDistance, ZeroOneScaleValues)

__all__ = [
    "Hypergraph", "HypergraphEmbedding", "EvaluationMetrics", "ExperimentalResult",
    "AddNodeToEdge", "CompressRange", "IsEmpty", "Relabel", "ToCsrMatrix", "ToEdgeCsrMatrix",
    "EmbedAlgebraicDistance",
    "AlgebraicDistanceSamples", "AlgebraicDistanceSamplesCsr", "AlgebraicDistanceSamplesDevice",
    "BooleanSamples", "BooleanSamplesCsr", "BooleanSamplesDevice",
    "DeviceSampleColumns", "SampleColumns",
    "SamplesToModelInput", "SimilarityRecord", "SparseWeightedJaccard", "WeightedJaccardSamples",
    "WeightedJaccardSamplesDevice",
    "BooleanModel", "UnweightedFloatModel", "KerasModelToEmbedding", "EMBEDDING_OPTIONS",
    "EmbedHg2vBoolean", "EmbedHg2vAdjJaccard", "EmbedHg2vNeighborhoodWeightedJaccard",
    "EmbedHg2vAlgDist", "EmbedHg2vBooleanDevice", "EmbedHg2vAlgDistDevice",
    "EmbedHg2vAdjJaccardDevice", "EmbedHg2vNeighborhoodWeightedJaccardDevice",
    "EmbedNMFDevice", "NonNegativeFactorizationDevice", "EmbedSVDDevice", "TruncatedSVDDevice",
    "EmbedNode2VecDevice", "Node2VecDevice", "EmbedNode2VecCliqueDevice", "Node2VecCliqueDevice",
    "AlphaScaleValues", "ComputeSpans", "DictToSparseRow", "OneMinusValues", "UniformWeight",
    "WeightByAlgebraicSpan", "WeightByDistance", "WeightByDistanceCluster", "WeightByNeighborhood",
    "WeightBySameTypeDistance", "ZeroOneScaleValues",
]
