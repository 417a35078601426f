"""Write tests/golden/coclustering_golden.json from the COMPILED, UNMODIFIED reference.

Run where the reference can be built (oracle/_ref):

    bash oracle/build_ref.sh && python tests/golden/make_coclustering_golden.py

What is pinned: CoClustering (co_clustering.pyx:68-237) on the u1 fixture with the defaults and random_state=1 (the
seed of the reference's tests/test_co_clustering.py): the RMSE / MAE reprs of AlgoBase.test + accuracy, and the
sha256 of cltr_u / cltr_i / avg_cltr_u / avg_cltr_i / avg_cocltr.
"""
import hashlib
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
import oracle  # noqa: E402

oracle.import_reference()
from surprise import CoClustering, Dataset, Reader, accuracy  # noqa: E402
from surprise.model_selection import PredefinedKFold  # noqa: E402


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


data = Dataset.load_from_folds([(os.path.join(HERE, "u1_ml100k_train"), os.path.join(HERE, "u1_ml100k_test"))],
                               Reader("ml-100k"))
trainset, testset = next(PredefinedKFold().split(data))
cc = CoClustering(random_state=1)
cc.fit(trainset)
preds = cc.test(testset)
out = {"source": "the compiled reference's CoClustering (tests/golden/make_coclustering_golden.py)",
       "u1_default_rs1": {"kwargs": {"n_cltr_u": 3, "n_cltr_i": 3, "n_epochs": 20, "random_state": 1},
                          "rmse": repr(float(accuracy.rmse(preds, verbose=False))),
                          "mae": repr(float(accuracy.mae(preds, verbose=False))),
                          "sha256": {k: sha(np.asarray(getattr(cc, k))) for k in
                                     ("cltr_u", "cltr_i", "avg_cltr_u", "avg_cltr_i", "avg_cocltr")}}}
with open(os.path.join(HERE, "coclustering_golden.json"), "w") as fh:
    json.dump(out, fh, indent=1)
    fh.write("\n")
print(json.dumps(out, indent=1))
