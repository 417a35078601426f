"""GridSearchCV and RandomizedSearchCV (upstream Surprise 1.1: model_selection/search.py).

Same constructors, candidates, task order, ``cv_results`` keys, ranks and ``best_*`` attributes as upstream.  Two
differences: the tasks run in this process, one after another (``n_jobs``, ``pre_dispatch`` and ``joblib_verbose``
are accepted and ignored, as in cross_validate), and a randomized search over lists only draws its candidates from
``random_state`` instead of numpy's global state, so that the seed is honoured.

Every candidate is fitted and scored by ``validation._fit_and_score`` on the same folds; each fold maps its pairs to
inner ids once, and a device-batched algorithm is scored from arrays without building Prediction tuples.
"""
from itertools import product

import numpy as np

from .. import accuracy
from ..dataset import DatasetUserFolds
from ..utils import get_rng
from .split import get_cv
from .validation import Fold, _fit_and_score


class BaseSearchCV(object):
    def __init__(self, algo_class, measures=["rmse", "mae"], cv=None, refit=False, return_train_measures=False,
                 n_jobs=1, pre_dispatch="2*n_jobs", joblib_verbose=0):
        self.algo_class = algo_class
        self.measures = [measure.lower() for measure in measures]
        self.cv = cv
        if isinstance(refit, str):
            if refit.lower() not in self.measures:
                raise ValueError("It looks like the measure you want to use with refit ({}) is not in the measures "
                                 "parameter".format(refit))
            self.refit = refit.lower()
        elif refit is True:
            self.refit = self.measures[0]
        else:
            self.refit = False
        self.return_train_measures = return_train_measures
        self.n_jobs = n_jobs
        self.pre_dispatch = pre_dispatch
        self.joblib_verbose = joblib_verbose

    @staticmethod
    def _parse_options(params):
        """sim_options / bsl_options given as a dict of lists become the list of every combination of them."""
        for key in ("sim_options", "bsl_options"):
            if key in params and isinstance(params[key], dict):
                options = params[key]
                params[key] = [dict(zip(options, v)) for v in product(*options.values())]
        return params

    def fit(self, data):
        if self.refit and isinstance(data, DatasetUserFolds):
            raise ValueError("refit cannot be used when data has been loaded with load_from_folds().")
        folds = [Fold(trainset, testset) for trainset, testset in get_cv(self.cv).split(data)]
        out = [_fit_and_score(self.algo_class(**params), fold, self.measures, self.return_train_measures)
               for params, fold in product(self.param_combinations, folds)]
        test_measures_dicts, train_measures_dicts, fit_times, test_times = zip(*out)

        # (candidates, folds) arrays per measure
        n_folds = len(folds)
        new_shape = (len(self.param_combinations), n_folds)
        test_measures, train_measures = {}, {}
        for m in self.measures:
            test_measures[m] = np.asarray([d[m] for d in test_measures_dicts]).reshape(new_shape)
            if self.return_train_measures:
                train_measures[m] = np.asarray([d[m] for d in train_measures_dicts]).reshape(new_shape)

        cv_results, best_index, best_params, best_score, best_estimator = {}, {}, {}, {}, {}
        for m in self.measures:
            for split in range(n_folds):
                cv_results["split{0}_test_{1}".format(split, m)] = test_measures[m][:, split]
                if self.return_train_measures:
                    cv_results["split{0}_train_{1}".format(split, m)] = train_measures[m][:, split]
            mean_test_measures = test_measures[m].mean(axis=1)
            cv_results["mean_test_{}".format(m)] = mean_test_measures
            cv_results["std_test_{}".format(m)] = test_measures[m].std(axis=1)
            if self.return_train_measures:
                cv_results["mean_train_{}".format(m)] = train_measures[m].mean(axis=1)
                cv_results["std_train_{}".format(m)] = train_measures[m].std(axis=1)

            indices = mean_test_measures.argsort()
            rank = np.empty_like(indices)
            cv_results["rank_test_{}".format(m)] = rank
            if m in ("mae", "rmse", "mse", "mpr"):
                rank[indices] = np.arange(len(indices)) + 1
                best_index[m] = mean_test_measures.argmin()
            elif m in ("fcp", "auc", "mrr") or accuracy._top_n_measure(m) or accuracy._top_n_list_measure(m):
                rank[indices] = np.arange(len(indices), 0, -1)
                best_index[m] = mean_test_measures.argmax()
            best_params[m] = self.param_combinations[best_index[m]]
            best_score[m] = mean_test_measures[best_index[m]]
            best_estimator[m] = self.algo_class(**best_params[m])

        for s, times in (("fit", fit_times), ("test", test_times)):
            times = np.array(times).reshape(new_shape)
            cv_results["mean_{}_time".format(s)] = times.mean(axis=1)
            cv_results["std_{}_time".format(s)] = times.std(axis=1)

        cv_results["params"] = self.param_combinations
        for param in self.param_combinations[0]:
            cv_results["param_" + param] = [comb[param] for comb in self.param_combinations]

        if self.refit:
            best_estimator[self.refit].fit(data.build_full_trainset())

        self.best_index = best_index
        self.best_params = best_params
        self.best_score = best_score
        self.best_estimator = best_estimator
        self.cv_results = cv_results

    def test(self, testset, verbose=False):
        """``test()`` of the best estimator for the refit measure."""
        if not self.refit:
            raise ValueError("refit is False, cannot use test()")
        return self.best_estimator[self.refit].test(testset, verbose)

    def predict(self, *args):
        """``predict()`` of the best estimator for the refit measure."""
        if not self.refit:
            raise ValueError("refit is False, cannot use predict()")
        return self.best_estimator[self.refit].predict(*args)


class GridSearchCV(BaseSearchCV):
    """Every combination of ``param_grid`` (a dict of lists): insertion order, the last key varying fastest."""

    def __init__(self, algo_class, param_grid, measures=["rmse", "mae"], cv=None, refit=False,
                 return_train_measures=False, n_jobs=1, pre_dispatch="2*n_jobs", joblib_verbose=0):
        super(GridSearchCV, self).__init__(algo_class=algo_class, measures=measures, cv=cv, refit=refit,
                                           return_train_measures=return_train_measures, n_jobs=n_jobs,
                                           pre_dispatch=pre_dispatch, joblib_verbose=joblib_verbose)
        self.param_grid = self._parse_options(param_grid.copy())
        self.param_combinations = [dict(zip(self.param_grid, v)) for v in product(*self.param_grid.values())]


class RandomizedSearchCV(BaseSearchCV):
    """``n_iter`` candidates drawn from ``param_distributions`` (a dict of lists or of objects with ``rvs``).  When
    every value is a list, ``n_iter`` distinct combinations of the full grid are drawn without replacement (more
    than the grid holds raises ValueError); otherwise each parameter is drawn independently per candidate, ``rvs``
    or a uniform pick from the list.  All draws come from ``get_rng(random_state)``."""

    def __init__(self, algo_class, param_distributions, n_iter=10, measures=["rmse", "mae"], cv=None, refit=False,
                 return_train_measures=False, n_jobs=1, pre_dispatch="2*n_jobs", random_state=None,
                 joblib_verbose=0):
        super(RandomizedSearchCV, self).__init__(algo_class=algo_class, measures=measures, cv=cv, refit=refit,
                                                 return_train_measures=return_train_measures, n_jobs=n_jobs,
                                                 pre_dispatch=pre_dispatch, joblib_verbose=joblib_verbose)
        self.n_iter = n_iter
        self.random_state = random_state
        self.param_distributions = self._parse_options(param_distributions.copy())
        self.param_combinations = self._sample_parameters(self.param_distributions, self.n_iter, self.random_state)

    @staticmethod
    def _sample_parameters(param_distributions, n_iter, random_state=None):
        all_lists = all(not hasattr(v, "rvs") for v in param_distributions.values())
        rnd = get_rng(random_state)
        items = sorted(param_distributions.items())     # sorted for reproducibility
        if all_lists:
            param_grid = [dict(zip(param_distributions, v)) for v in product(*param_distributions.values())]
            # RandomState.choice(param_grid, ...) draws the same positions; indexing keeps a list of dicts
            return [param_grid[k] for k in rnd.choice(len(param_grid), n_iter, replace=False).tolist()]
        combos = []
        for _ in range(n_iter):
            params = dict()
            for k, v in items:
                params[k] = v.rvs(random_state=rnd) if hasattr(v, "rvs") else v[rnd.randint(len(v))]
            combos.append(params)
        return combos
