"""Prediction algorithms of surprise_b200 (the hot-path subset of the reference's package)."""
from .algo_base import AlgoBase
from .baseline_only import BaselineOnly
from .knns import KNNBasic, KNNBaseline, KNNWithMeans, KNNWithZScore
from .matrix_factorization import SVD, SVDpp, NMF
from .slope_one import SlopeOne
from .co_clustering import CoClustering
from .predictions import Prediction, PredictionImpossible

__all__ = ["AlgoBase", "BaselineOnly", "KNNBasic", "KNNBaseline", "KNNWithMeans", "KNNWithZScore", "SVD", "SVDpp", "NMF", "SlopeOne", "CoClustering", "Prediction",
           "PredictionImpossible"]
