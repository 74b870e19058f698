"""TEST INFRASTRUCTURE - writes tests/golden/task_classifier_scaler.pkl: an sklearn ``StandardScaler`` pickled by sklearn itself,
holding the statistics of the reference's classifier scaler (``scaler_mean`` / ``scaler_scale`` of task_classifier.npz). It lets
tests/test_ensemble_host.py check that ``TaskClassifier.load`` reads sklearn's pickle format without importing sklearn.

    python tests/golden/make_scaler_pickle.py        # needs scikit-learn
"""
import os
import pickle

import numpy as np
from sklearn.preprocessing import StandardScaler

HERE = os.path.dirname(os.path.abspath(__file__))

g = np.load(os.path.join(HERE, "task_classifier.npz"))
sc = StandardScaler()
sc.mean_, sc.scale_ = g["scaler_mean"], g["scaler_scale"]
sc.var_ = sc.scale_ ** 2
sc.n_features_in_, sc.n_samples_seen_ = len(sc.mean_), np.int64(1000)       # the sample count is not recorded; the loader ignores it
with open(os.path.join(HERE, "task_classifier_scaler.pkl"), "wb") as f:
    pickle.dump(sc, f)
