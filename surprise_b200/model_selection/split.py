"""Cross-validation iterators (reference: model_selection/split.py): KFold (:57-122), RepeatedKFold (:365-415),
ShuffleSplit (:418-540), train_test_split (:543-583), PredefinedKFold (:654-685), and upstream Surprise 1.1's
LeaveOneOut.  Same index arithmetic and the same RNG calls as the reference, so a given random_state yields the same
trainset / testset rows.

All of them work on index arrays and hand them to ``Dataset._take``: a list-backed dataset yields the reference's
raw-rating lists, an array-backed one (Dataset.load_from_arrays) slices its three arrays, so that 10^7..10^8
ratings are split without ever becoming Python tuples.
"""
from math import ceil, floor

import numpy as np

from ..dataset import first_appearance
from ..utils import get_rng


class PredefinedKFold(object):
    """Folds come from Dataset.load_from_folds()."""

    def split(self, data):
        self.n_splits = len(data.folds_files)
        for raw_train, raw_test in data.raw_folds():
            yield data.construct_trainset(raw_train), data.construct_testset(raw_test)

    def get_n_folds(self):
        return self.n_splits


class KFold(object):
    def __init__(self, n_splits=5, random_state=None, shuffle=True):
        self.n_splits, self.random_state, self.shuffle = n_splits, random_state, shuffle

    def split(self, data):
        n = data.n_raw_ratings()
        if self.n_splits > n or self.n_splits < 2:
            raise ValueError("Incorrect value for n_splits={0}. Must be >=2 and less than the number of ratings"
                             .format(n))
        idx = np.arange(n)
        if self.shuffle:
            get_rng(self.random_state).shuffle(idx)
        start = stop = 0
        for fold in range(self.n_splits):
            start = stop
            stop += n // self.n_splits + (1 if fold < n % self.n_splits else 0)
            train = data._take(np.concatenate((idx[:start], idx[stop:])))
            test = data._take(idx[start:stop])
            yield data.construct_trainset(train), data.construct_testset(test)

    def get_n_folds(self):
        return self.n_splits


class RepeatedKFold(object):
    def __init__(self, n_splits=5, n_repeats=10, random_state=None):
        self.n_splits, self.n_repeats, self.random_state = n_splits, n_repeats, random_state

    def split(self, data):
        rng = get_rng(self.random_state)
        for _ in range(self.n_repeats):
            for pair in KFold(n_splits=self.n_splits, random_state=rng, shuffle=True).split(data):
                yield pair

    def get_n_folds(self):
        return self.n_repeats * self.n_splits


class ShuffleSplit(object):
    """Random train / test splits.  As in the reference (:506-536) the trainset is the HEAD of the permutation
    (permutation[:n_train]) and the testset the n_test entries that follow; with shuffle=False the testset is
    therefore the tail of the file, the usual chronological hold-out."""

    def __init__(self, n_splits=5, test_size=.2, train_size=None, random_state=None, shuffle=True):
        if n_splits <= 0:
            raise ValueError("n_splits = {0} should be strictly greater than 0.".format(n_splits))
        if test_size is not None and test_size <= 0:
            raise ValueError("test_size={0} should be strictly greater than 0".format(test_size))
        if train_size is not None and train_size <= 0:
            raise ValueError("train_size={0} should be strictly greater than 0".format(train_size))
        self.n_splits, self.test_size, self.train_size = n_splits, test_size, train_size
        self.random_state, self.shuffle = random_state, shuffle

    def validate_train_test_sizes(self, test_size, train_size, n_ratings):
        if test_size is not None and test_size >= n_ratings:
            raise ValueError("test_size={0} should be less than the number of ratings {1}".format(test_size, n_ratings))
        if train_size is not None and train_size >= n_ratings:
            raise ValueError("train_size={0} should be less than the number of ratings {1}".format(train_size, n_ratings))
        if np.asarray(test_size).dtype.kind == "f":
            test_size = ceil(test_size * n_ratings)
        if train_size is None:
            train_size = n_ratings - test_size
        elif np.asarray(train_size).dtype.kind == "f":
            train_size = floor(train_size * n_ratings)
        if test_size is None:
            test_size = n_ratings - train_size
        if train_size + test_size > n_ratings:
            raise ValueError("The sum of train_size and test_size ({0}) should be smaller than the number of "
                             "ratings {1}.".format(train_size + test_size, n_ratings))
        return int(train_size), int(test_size)

    def split(self, data):
        n = data.n_raw_ratings()
        n_train, n_test = self.validate_train_test_sizes(self.test_size, self.train_size, n)
        rng = get_rng(self.random_state)
        for _ in range(self.n_splits):
            perm = rng.permutation(n) if self.shuffle else np.arange(n)
            train = data._take(perm[:n_train])
            test = data._take(perm[n_train:n_train + n_test])
            yield data.construct_trainset(train), data.construct_testset(test)

    def get_n_folds(self):
        return self.n_splits


class LeaveOneOut(object):
    """Each split holds out one rating per user: upstream Surprise 1.1's LeaveOneOut, restated here.

    The reference groups ``data.raw_ratings`` by uid into a ``defaultdict(list)`` (users in first-appearance order,
    equal uids merged, each user's ratings in file order) and draws ``rng = get_rng(random_state)`` once for the whole
    iterator.  Then, for each of the ``n_splits`` splits and each user with ``len(ratings) > min_n_ratings``, in group
    order, it draws ``k = rng.randint(0, len(ratings))``, appends ``ratings[k]`` to the testset and the user's other
    ratings, in order, to the trainset.  Users at or below ``min_n_ratings`` are in neither set.  An empty trainset
    raises ``ValueError('Could not build any trainset. Maybe min_n_ratings is too high?')``.

    The trainset is therefore in user-grouped order, not file order, and its inner item ids differ from the ones KFold
    assigns.  Here the groups are index arrays (a stable sort of the first-appearance user codes), and the per-user
    draws of one split are one ``rng.randint(0, lengths)`` call, which consumes the RandomState's stream exactly as
    the scalar draws in user order do.  An array-backed dataset is split without creating tuples."""

    def __init__(self, n_splits=5, random_state=None, min_n_ratings=0):
        self.n_splits, self.random_state, self.min_n_ratings = n_splits, random_state, min_n_ratings

    def split(self, data):
        if data._arrays is not None:
            code, uniq = first_appearance(data._arrays[0])
            n_users = len(uniq)
        else:
            users = {}
            setd = users.setdefault
            code = np.array([setd(row[0], len(users)) for row in data.raw_ratings], dtype=np.int64)
            n_users = len(users)
        order = np.argsort(code, kind="stable")         # row indices grouped by user, file order within a user
        length = np.bincount(code, minlength=n_users)
        start = np.cumsum(length) - length
        kept = np.flatnonzero(length > self.min_n_ratings)
        in_kept = np.repeat(length > self.min_n_ratings, length)     # per entry of order
        rng = get_rng(self.random_state)
        for _ in range(self.n_splits):
            test = start[kept] + rng.randint(0, length[kept]) if len(kept) else kept
            train = in_kept.copy()
            train[test] = False
            if not train.any():
                raise ValueError("Could not build any trainset. Maybe min_n_ratings is too high?")
            yield data.construct_trainset(data._take(order[train])), data.construct_testset(data._take(order[test]))

    def get_n_folds(self):
        return self.n_splits


def get_cv(cv):
    """The splitter cross_validate and the searches use: 5-fold KFold for None, KFold(n_splits=cv) for an int, cv
    itself otherwise."""
    return KFold(n_splits=5) if cv is None else (KFold(n_splits=cv) if isinstance(cv, int) else cv)


def train_test_split(data, test_size=.2, train_size=None, random_state=None, shuffle=True):
    """split.py:543-583: one ShuffleSplit draw."""
    ss = ShuffleSplit(n_splits=1, test_size=test_size, train_size=train_size, random_state=random_state,
                      shuffle=shuffle)
    return next(ss.split(data))
