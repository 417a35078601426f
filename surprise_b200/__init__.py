"""surprise_b200 -- B200-native fit-time hot path of Surprise behind Surprise's own Python API.

    from surprise_b200 import Dataset, Reader, KNNBasic, KNNBaseline, SVD, SVDpp, NMF, CoClustering, accuracy

Host code is Python; all numerics run in hand-written sm_100a CUDA kernels reached through the C-ABI
of libsurprise_b200.so (include/surprise_b200.h).  There is no CPU fallback.
"""
from . import accuracy, dump, similarities
from .dataset import Dataset
from .prediction_algorithms import (AlgoBase, BaselineOnly, KNNBaseline, KNNBasic, KNNWithMeans, KNNWithZScore, NMF,
                                    SVD, SVDpp, SlopeOne, CoClustering, Prediction,
                                    PredictionImpossible)
from .reader import Reader
from .trainset import Trainset

__all__ = ["AlgoBase", "BaselineOnly", "KNNBasic", "KNNBaseline", "KNNWithMeans", "KNNWithZScore", "SVD", "SVDpp", "NMF", "SlopeOne", "CoClustering", "Prediction",
           "PredictionImpossible", "Dataset", "Reader", "Trainset", "accuracy", "dump", "similarities"]
__version__ = "0.1.0"
