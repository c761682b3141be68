"""small run of isb_gmm_predict (both paths, with and without a device row count) and of a pipeline with a DeviceClassModel, for
compute-sanitizer --tool memcheck"""
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), 'tests'))
from conftest import synth_regions  # noqa: E402
from sklearn import mixture, pipeline, preprocessing  # noqa: E402

from pyimsegm_b200 import pipelines as pl  # noqa: E402
from pyimsegm_b200.engine import get_engine  # noqa: E402
from pyimsegm_b200.graph_cuts import DeviceClassModel  # noqa: E402

rng = np.random.RandomState(0)
eng = get_engine()
for D in (5, 24):
    X = np.concatenate([c + rng.normal(0, 0.7, (70, D)) for c in rng.normal(0, 2.0, (3, D))])
    X[5, 1] = np.nan
    model = pipeline.Pipeline([('s', preprocessing.StandardScaler()), ('m', mixture.GaussianMixture(3, random_state=0))])
    model.fit(np.nan_to_num(X))
    dcm = DeviceClassModel(model)
    err = np.abs(dcm.predict_proba(X) - model.predict_proba(np.nan_to_num(X))).max()
    d_n = eng.to_device(np.array([123], dtype=np.int32), 'san_n')
    eng.gmm_predict(eng.to_device(X, 'san_feat'), dcm.device_params(eng), 3, d_n=d_n)
    eng.torch.cuda.synchronize()
    print('predict D=%d ok, max |diff| %.2e' % (D, err))
img, _ = synth_regions(96, 136, seed=1)
feats = {'color': ['mean', 'std']}
_, fts = pl.compute_color2d_superpixels_features(img, feats, sp_size=12, sp_regul=0.3)
dcm = DeviceClassModel(mixture.GaussianMixture(3, random_state=0).fit(fts))
segm, soft = pl.segment_color2d_slic_features_model_graphcut(img, dcm, feats, sp_size=12, sp_regul=0.3)
print('pipeline ok', np.bincount(segm.ravel()))
