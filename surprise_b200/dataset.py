"""Dataset: raw ratings -> Trainset / testset (reference: surprise/dataset.py:44-375).

Inner ids are assigned in first-appearance order (dataset.py:219-234); that order defines the
iteration order the kernels must reproduce.
"""
import itertools
import os

import numpy as np

from .reader import Reader
from .trainset import Trainset


def first_appearance(a):
    """(code, uniq): each entry's rank among the distinct values of a in first-appearance order (int32), and those
    values in that order."""
    n = len(a)
    if n and np.issubdtype(a.dtype, np.integer) and int(a.max()) - int(a.min()) <= max(4 * n, 10_000_000):
        # integer raw ids in a modest range: O(N) table instead of a sort of all the ratings
        lo = int(a.min())
        shifted = (a - lo).astype(np.int64)
        first = np.full(int(shifted.max()) + 1, n, dtype=np.int64)
        first[shifted[::-1]] = np.arange(n - 1, -1, -1, dtype=np.int64)   # repeated index: last write wins
        present = np.nonzero(first < n)[0]
        order = np.argsort(first[present], kind="stable")
        rank = np.empty(len(first), dtype=np.int32)
        rank[present[order]] = np.arange(len(present), dtype=np.int32)
        return rank[shifted], (present[order] + lo).astype(a.dtype)
    uniq, first, inv = np.unique(a, return_index=True, return_inverse=True)
    order = np.argsort(first, kind="stable")          # uniq[order] is in first-appearance order
    rank = np.empty(len(uniq), dtype=np.int64)
    rank[order] = np.arange(len(uniq))
    return rank[inv].astype(np.int32), uniq[order]


class Dataset(object):
    def __init__(self, reader):
        self.reader = reader

    # -- loaders ---------------------------------------------------------------------------------------
    @classmethod
    def load_from_file(cls, file_path, reader):
        return DatasetAutoFolds(ratings_file=file_path, reader=reader)

    @classmethod
    def load_from_folds(cls, folds_files, reader):
        return DatasetUserFolds(folds_files=folds_files, reader=reader)

    @classmethod
    def load_from_df(cls, df, reader):
        return DatasetAutoFolds(reader=reader, df=df)

    @classmethod
    def load_from_arrays(cls, uids, iids, ratings, reader=None):
        """Array fast path: three equal-length arrays (raw user ids, raw item ids, ratings)."""
        return DatasetAutoFolds(reader=reader or Reader(), arrays=(uids, iids, ratings))

    def read_ratings(self, file_name):
        with open(os.path.expanduser(file_name)) as fh:
            return [self.reader.parse_line(line) for line in itertools.islice(fh, self.reader.skip_lines, None)]

    # -- trainset / testset ----------------------------------------------------------------------------
    def construct_trainset(self, raw_trainset):
        if isinstance(raw_trainset, tuple) and len(raw_trainset) == 3 and isinstance(raw_trainset[0], np.ndarray):
            return self._trainset_from_arrays(*raw_trainset)
        u2i, i2i = {}, {}
        n = len(raw_trainset)
        u = np.empty(n, dtype=np.int32)
        i = np.empty(n, dtype=np.int32)
        r = np.empty(n, dtype=np.float64)
        for k, (ruid, riid, rating, _) in enumerate(raw_trainset):
            u[k] = u2i.setdefault(ruid, len(u2i))
            i[k] = i2i.setdefault(riid, len(i2i))
            r[k] = rating
        ts = Trainset.from_coo(u, i, r, len(u2i), len(i2i), self.reader.rating_scale, self.reader.offset)
        ts._raw2inner_id_users, ts._raw2inner_id_items = u2i, i2i
        return ts

    def _trainset_from_arrays(self, uids, iids, ratings):
        u, raw_u = first_appearance(np.asarray(uids))
        i, raw_i = first_appearance(np.asarray(iids))
        r = np.asarray(ratings, dtype=np.float64) + self.reader.offset
        return Trainset.from_coo(u, i, r, len(raw_u), len(raw_i), self.reader.rating_scale, self.reader.offset,
                                 raw_uids=raw_u.tolist(), raw_iids=raw_i.tolist())

    def construct_testset(self, raw_testset):
        if isinstance(raw_testset, tuple) and len(raw_testset) == 3 and isinstance(raw_testset[0], np.ndarray):
            uids, iids, ratings = raw_testset     # array fast path: ratings still carry no offset
            r = np.asarray(ratings, dtype=np.float64) + self.reader.offset
            return list(zip(uids.tolist(), iids.tolist(), r.tolist()))
        return [(ruid, riid, r_ui_trans) for (ruid, riid, r_ui_trans, _) in raw_testset]


class DatasetUserFolds(Dataset):
    """Predefined (train file, test file) folds."""

    def __init__(self, folds_files=None, reader=None):
        Dataset.__init__(self, reader)
        self.folds_files = folds_files
        for pair in self.folds_files:
            for f in pair:
                if not os.path.isfile(os.path.expanduser(f)):
                    raise ValueError("File " + str(f) + " does not exist.")

    def raw_folds(self):
        for train_file, test_file in self.folds_files:
            yield self.read_ratings(train_file), self.read_ratings(test_file)


class DatasetAutoFolds(Dataset):
    """A single ratings source; folds are made by the cross-validation iterators."""

    def __init__(self, ratings_file=None, reader=None, df=None, arrays=None):
        Dataset.__init__(self, reader)
        self.has_been_split = False
        self._arrays = None
        if ratings_file is not None:
            self.ratings_file = ratings_file
            self.raw_ratings = self.read_ratings(ratings_file)
        elif df is not None:
            self.raw_ratings = [(uid, iid, float(r) + self.reader.offset, None)
                                for (uid, iid, r) in df.itertuples(index=False)]
        elif arrays is not None:
            self._arrays = tuple(np.asarray(a) for a in arrays)
            self.raw_ratings = None
        else:
            raise ValueError("Must specify ratings file or dataframe.")

    def n_raw_ratings(self):
        return len(self._arrays[0]) if self._arrays is not None else len(self.raw_ratings)

    def _take(self, idx):
        """The raw ratings at positions idx: a list of the reference's raw tuples, or (array-backed dataset) the
        three arrays sliced -- both are accepted by construct_trainset / construct_testset."""
        if self._arrays is not None:
            return tuple(a[idx] for a in self._arrays)
        return [self.raw_ratings[k] for k in idx]

    def build_full_trainset(self):
        if self._arrays is not None:
            return self.construct_trainset(self._arrays)
        return self.construct_trainset(self.raw_ratings)
