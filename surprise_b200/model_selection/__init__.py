from .search import GridSearchCV, RandomizedSearchCV
from .split import KFold, LeaveOneOut, PredefinedKFold, RepeatedKFold, ShuffleSplit, train_test_split
from .validation import cross_validate, fit_and_score

__all__ = ["KFold", "LeaveOneOut", "PredefinedKFold", "RepeatedKFold", "ShuffleSplit", "train_test_split",
           "cross_validate", "fit_and_score", "GridSearchCV", "RandomizedSearchCV"]
