"""SVD, SVDpp, NMF (reference: prediction_algorithms/matrix_factorization.pyx:19-761).

Constructors, defaults and per-parameter lr/reg override logic are the reference's (:129-151, :389-411,
:616-637); ``sgd()`` hands the all_ratings() COO and the host-generated initial factors (numpy
RandomState, same draw order as the reference so that seeds agree: pu then qi (then yj)) to the CUDA
kernels and gets float64 factors back.  ``estimate`` for a whole testset is one device call.
"""
import ctypes as C

import numpy as np

from .. import _native as nat
from ..utils import get_rng
from .algo_base import AlgoBase
from .predictions import PredictionImpossible


def _pick(value, default):
    return default if value is None else value


def _as_inner(v):
    return int(v) if isinstance(v, (int, np.integer)) else -1


class _FactorModel(AlgoBase):
    """Shared device plumbing of the three factor models."""
    _has_yj = False

    def _coo_dev(self, trainset):
        u, i, r = trainset.coo()
        return nat.to_dev(u, np.int32), nat.to_dev(i, np.int32), nat.to_dev(r, np.float64), len(r)

    def _device_factors(self):
        dev = getattr(self, "_dev_cache", None)
        if dev is None:
            ts = self.trainset
            dev = dict(pu=nat.to_dev(self.pu, np.float64), qi=nat.to_dev(self.qi, np.float64),
                       bu=nat.to_dev(self.bu, np.float64), bi=nat.to_dev(self.bi, np.float64))
            if self._has_yj:
                ptr, idx, _ = ts.user_csr()
                dev.update(yj=nat.to_dev(self.yj, np.float64), up=nat.to_dev(ptr, np.int64),
                           ui=nat.to_dev(idx, np.int32))
            self._dev_cache = dev
        return dev

    def _predict_dev(self, d_u, d_i, biased):
        """(est, impossible) device tensors for the device pairs (d_u, d_i) (sb2_mf_predict_dev)."""
        n = len(d_u)
        dev = self._device_factors()
        est = nat.empty_dev((max(n, 1),), np.float64)
        imp = nat.empty_dev((max(n, 1),), np.uint8)
        rc = nat.lib().sb2_mf_predict_dev(n, nat.ptr(d_u), nat.ptr(d_i), self.pu.shape[1], int(bool(biased)),
                                          float(self.trainset.global_mean), nat.ptr(dev["pu"]), nat.ptr(dev["qi"]),
                                          nat.ptr(dev["bu"]), nat.ptr(dev["bi"]), nat.ptr(dev.get("yj")),
                                          nat.ptr(dev.get("up")), nat.ptr(dev.get("ui")), nat.ptr(est), nat.ptr(imp),
                                          nat.stream())
        nat.check(rc)
        return est, imp

    def _predict_batch(self, iu, ii, biased):
        n = len(iu)
        est, imp = self._predict_dev(nat.to_dev(iu, np.int32), nat.to_dev(ii, np.int32), biased)
        est, imp = est.cpu().numpy()[:n], imp.cpu().numpy()[:n]
        details = [({"was_impossible": True, "reason": "User and item are unkown."} if imp[k]
                    else {"was_impossible": False}) for k in range(n)]
        return est, details

    def _estimate_dev(self, d_u, d_i):
        return self._predict_dev(d_u, d_i, self._est_biased())

    def _top_n_scorer(self):
        return dict(self._device_factors(), f=int(self.pu.shape[1]), biased=int(bool(self._est_biased())))

    def __setattr__(self, name, value):
        # the reference's estimate() reads pu / qi / bu / bi / yj live: assigning any of them after fit (warm starts,
        # factor surgery) must not leave predict() / test() on stale device copies
        if name in ("pu", "qi", "bu", "bi", "yj", "trainset"):
            self.__dict__.pop("_dev_cache", None)
        object.__setattr__(self, name, value)

    def __getstate__(self):
        state = dict(self.__dict__)
        state.pop("_dev_cache", None)
        return state

    def _estimate_one(self, u, i):
        est, details = self._estimate_batch(np.array([_as_inner(u)], dtype=np.int32),
                                            np.array([_as_inner(i)], dtype=np.int32))
        if details[0]["was_impossible"]:
            raise PredictionImpossible(details[0]["reason"])
        return est[0]


class SVD(_FactorModel):
    """matrix_factorization.pyx:19-299."""

    def __init__(self, n_factors=100, n_epochs=20, biased=True, init_mean=0, init_std_dev=.1, lr_all=.005,
                 reg_all=.02, lr_bu=None, lr_bi=None, lr_pu=None, lr_qi=None, reg_bu=None, reg_bi=None, reg_pu=None,
                 reg_qi=None, random_state=None, verbose=False):
        self.n_factors, self.n_epochs, self.biased = n_factors, n_epochs, biased
        self.init_mean, self.init_std_dev = init_mean, init_std_dev
        self.lr_bu, self.lr_bi = _pick(lr_bu, lr_all), _pick(lr_bi, lr_all)
        self.lr_pu, self.lr_qi = _pick(lr_pu, lr_all), _pick(lr_qi, lr_all)
        self.reg_bu, self.reg_bi = _pick(reg_bu, reg_all), _pick(reg_bi, reg_all)
        self.reg_pu, self.reg_qi = _pick(reg_pu, reg_all), _pick(reg_qi, reg_all)
        self.random_state, self.verbose = random_state, verbose
        AlgoBase.__init__(self)

    def fit(self, trainset):
        AlgoBase.fit(self, trainset)
        self.sgd(trainset)
        return self

    def _params(self, trainset, lr_yj=0.0, reg_yj=0.0, biased=True):
        return nat.SgdParams(n_factors=self.n_factors, n_epochs=self.n_epochs, biased=int(bool(biased)), reserved=0,
                             global_mean=float(trainset.global_mean), lr_bu=self.lr_bu, lr_bi=self.lr_bi,
                             lr_pu=self.lr_pu, lr_qi=self.lr_qi, lr_yj=lr_yj, reg_bu=self.reg_bu, reg_bi=self.reg_bi,
                             reg_pu=self.reg_pu, reg_qi=self.reg_qi, reg_yj=reg_yj)

    def _initial_factors(self, trainset):
        """(pu, qi, None): rng.normal draws in the reference's order (matrix_factorization.pyx:233-236)."""
        rng = get_rng(self.random_state)
        pu = rng.normal(self.init_mean, self.init_std_dev, (trainset.n_users, self.n_factors))
        qi = rng.normal(self.init_mean, self.init_std_dev, (trainset.n_items, self.n_factors))
        return pu, qi, None

    def _sgd_params(self, trainset):
        return self._params(trainset, biased=self.biased)

    def sgd(self, trainset):
        """matrix_factorization.pyx:172-267.  The host draws the initial factors with numpy's RandomState (seed parity
        with the reference; ~15 ms for 10^6 normals) while a helper thread uploads the ratings and stratifies them on
        the device (sb2_svd_plan_create_dev); then reset -> epochs -> factors back as float64."""
        import threading
        if self.verbose:
            for ep in range(self.n_epochs):
                print("Processing epoch {}".format(ep))
        prm = self._sgd_params(trainset)
        lib = nat.lib()
        torch = nat.torch_cuda()
        stream, dev_index = nat.stream(), torch.cuda.current_device()
        box = {}

        def prepare():
            try:
                torch.cuda.set_device(dev_index)
                d_u, d_i, d_r, n = self._coo_dev(trainset)
                plan = C.c_void_p()
                nat.check(lib.sb2_svd_plan_create_dev(trainset.n_users, trainset.n_items, n, nat.ptr(d_u), nat.ptr(d_i),
                                                      nat.ptr(d_r), C.byref(prm), 0, None, None, stream, C.byref(plan)))
                box["plan"] = plan
            except BaseException as e:  # re-raised on the calling thread
                box["error"] = e
        helper = threading.Thread(target=prepare)
        helper.start()
        try:
            pu, qi, _ = self._initial_factors(trainset)
        finally:
            helper.join()
        if "error" in box:
            raise box["error"]
        plan = box["plan"]
        try:
            d_pu, d_qi = nat.to_dev(pu, np.float64), nat.to_dev(qi, np.float64)
            d_bu = nat.empty_dev((trainset.n_users,), np.float64)
            d_bi = nat.empty_dev((trainset.n_items,), np.float64)
            nat.check(lib.sb2_svd_plan_reset_dev(plan, nat.ptr(d_pu), nat.ptr(d_qi), None, stream))
            nat.check(lib.sb2_svd_plan_run(plan, int(self.n_epochs), stream))
            nat.check(lib.sb2_svd_plan_read_dev(plan, nat.ptr(d_pu), nat.ptr(d_qi), nat.ptr(d_bu), nat.ptr(d_bi), None,
                                                stream))
            nat.check(lib.sb2_svd_plan_status(plan, stream))
        finally:
            lib.sb2_svd_plan_destroy(plan)
        self.pu, self.qi = d_pu.cpu().numpy(), d_qi.cpu().numpy()
        self.bu, self.bi = d_bu.cpu().numpy(), d_bi.cpu().numpy()
        self._dev_cache = None

    def _est_biased(self):
        return self.biased

    def _estimate_batch(self, iu, ii):
        return self._predict_batch(iu, ii, self.biased)

    def estimate(self, u, i):
        return self._estimate_one(u, i)

    _batch_estimate_of = estimate


class SVDpp(_FactorModel):
    """matrix_factorization.pyx:302-522."""
    _has_yj = True

    def __init__(self, n_factors=20, n_epochs=20, init_mean=0, init_std_dev=.1, lr_all=.007, reg_all=.02,
                 lr_bu=None, lr_bi=None, lr_pu=None, lr_qi=None, lr_yj=None, reg_bu=None, reg_bi=None, reg_pu=None,
                 reg_qi=None, reg_yj=None, random_state=None, verbose=False):
        self.n_factors, self.n_epochs = n_factors, n_epochs
        self.init_mean, self.init_std_dev = init_mean, init_std_dev
        self.lr_bu, self.lr_bi = _pick(lr_bu, lr_all), _pick(lr_bi, lr_all)
        self.lr_pu, self.lr_qi, self.lr_yj = _pick(lr_pu, lr_all), _pick(lr_qi, lr_all), _pick(lr_yj, lr_all)
        self.reg_bu, self.reg_bi = _pick(reg_bu, reg_all), _pick(reg_bi, reg_all)
        self.reg_pu, self.reg_qi, self.reg_yj = _pick(reg_pu, reg_all), _pick(reg_qi, reg_all), _pick(reg_yj, reg_all)
        self.random_state, self.verbose = random_state, verbose
        AlgoBase.__init__(self)

    def fit(self, trainset):
        AlgoBase.fit(self, trainset)
        self.sgd(trainset)
        return self

    def _initial_factors(self, trainset):
        """(pu, qi, yj) drawn in the reference's order (matrix_factorization.pyx:455-460)."""
        rng = get_rng(self.random_state)
        shape_u, shape_i = (trainset.n_users, self.n_factors), (trainset.n_items, self.n_factors)
        pu = rng.normal(self.init_mean, self.init_std_dev, shape_u)
        qi = rng.normal(self.init_mean, self.init_std_dev, shape_i)
        yj = rng.normal(self.init_mean, self.init_std_dev, shape_i)
        return pu, qi, yj

    def _sgd_params(self, trainset):
        return SVD._params(self, trainset, lr_yj=self.lr_yj, reg_yj=self.reg_yj, biased=True)

    def sgd(self, trainset):
        pu, qi, yj = self._initial_factors(trainset)
        if self.verbose:
            for ep in range(self.n_epochs):
                print(" processing epoch {}".format(ep))
        d_u, d_i, d_r, n = self._coo_dev(trainset)
        ptr, idx, _ = trainset.user_csr()
        d_up, d_ui = nat.to_dev(ptr, np.int64), nat.to_dev(idx, np.int32)
        d_pu, d_qi, d_yj = (nat.to_dev(a, np.float64) for a in (pu, qi, yj))
        d_bu = nat.empty_dev((trainset.n_users,), np.float64)
        d_bi = nat.empty_dev((trainset.n_items,), np.float64)
        prm = self._sgd_params(trainset)
        rc = nat.lib().sb2_svdpp_fit_dev(trainset.n_users, trainset.n_items, n, nat.ptr(d_u), nat.ptr(d_i),
                                         nat.ptr(d_r), nat.ptr(d_up), nat.ptr(d_ui), C.byref(prm), nat.ptr(d_pu),
                                         nat.ptr(d_qi), nat.ptr(d_yj), nat.ptr(d_bu), nat.ptr(d_bi), nat.stream())
        nat.check(rc)
        self.pu, self.qi, self.yj = d_pu.cpu().numpy(), d_qi.cpu().numpy(), d_yj.cpu().numpy()
        self.bu, self.bi = d_bu.cpu().numpy(), d_bi.cpu().numpy()
        self._dev_cache = None

    def _est_biased(self):
        return True

    def _estimate_batch(self, iu, ii):
        return self._predict_batch(iu, ii, True)

    def estimate(self, u, i):
        return self._estimate_one(u, i)

    _batch_estimate_of = estimate


class NMF(_FactorModel):
    """matrix_factorization.pyx:525-761.  Bit-exact against the reference (fp64, reference order)."""

    def __init__(self, n_factors=15, n_epochs=50, biased=False, reg_pu=.06, reg_qi=.06, reg_bu=.02, reg_bi=.02,
                 lr_bu=.005, lr_bi=.005, init_low=0, init_high=1, random_state=None, verbose=False):
        self.n_factors, self.n_epochs, self.biased = n_factors, n_epochs, biased
        self.reg_pu, self.reg_qi, self.reg_bu, self.reg_bi = reg_pu, reg_qi, reg_bu, reg_bi
        self.lr_bu, self.lr_bi = lr_bu, lr_bi
        self.init_low, self.init_high = init_low, init_high
        self.random_state, self.verbose = random_state, verbose
        if self.init_low < 0:
            raise ValueError("init_low should be greater than zero")
        AlgoBase.__init__(self)

    def fit(self, trainset):
        AlgoBase.fit(self, trainset)
        self.sgd(trainset)
        return self

    def sgd(self, trainset):
        rng = get_rng(self.random_state)
        pu = rng.uniform(self.init_low, self.init_high, size=(trainset.n_users, self.n_factors))
        qi = rng.uniform(self.init_low, self.init_high, size=(trainset.n_items, self.n_factors))
        if self.verbose:
            for ep in range(self.n_epochs):
                print("Processing epoch {}".format(ep))
        d_u, d_i, d_r, n = self._coo_dev(trainset)
        d_pu, d_qi = nat.to_dev(pu, np.float64), nat.to_dev(qi, np.float64)
        d_bu = nat.empty_dev((trainset.n_users,), np.float64)
        d_bi = nat.empty_dev((trainset.n_items,), np.float64)
        prm = nat.NmfParams(n_factors=self.n_factors, n_epochs=self.n_epochs, biased=int(bool(self.biased)),
                            reserved=0, global_mean=float(trainset.global_mean), reg_pu=self.reg_pu,
                            reg_qi=self.reg_qi, reg_bu=self.reg_bu, reg_bi=self.reg_bi, lr_bu=self.lr_bu,
                            lr_bi=self.lr_bi)
        rc = nat.lib().sb2_nmf_fit_dev(trainset.n_users, trainset.n_items, n, nat.ptr(d_u), nat.ptr(d_i), nat.ptr(d_r),
                                       C.byref(prm), nat.ptr(d_pu), nat.ptr(d_qi), nat.ptr(d_bu), nat.ptr(d_bi),
                                       nat.stream())
        nat.check(rc)
        self.pu, self.qi = d_pu.cpu().numpy(), d_qi.cpu().numpy()
        self.bu, self.bi = d_bu.cpu().numpy(), d_bi.cpu().numpy()
        self._dev_cache = None

    def _est_biased(self):
        return self.biased

    def _estimate_batch(self, iu, ii):
        return self._predict_batch(iu, ii, self.biased)

    def estimate(self, u, i):
        return self._estimate_one(u, i)

    _batch_estimate_of = estimate
