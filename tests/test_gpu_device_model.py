"""graph_cuts.DeviceClassModel on the GPU: isb_gmm_predict against scikit-learn's predict_proba, the pipelines with a shared model
kept on the device (single image, batch, resident, CUDA-graph replays, config-3 width, banded mode)."""
import numpy as np
import pytest

from conftest import synth_disc, synth_regions
from test_device_model_host import COVARIANCES, KINDS, evaluation_set, fitted_model, make_data

pytestmark = pytest.mark.gpu


def _shared_model(fts, K, covariance='full', scaler=True, **kw):
    from sklearn import mixture, pipeline, preprocessing
    mm = mixture.GaussianMixture(K, covariance_type=covariance, random_state=0, **kw)
    return (pipeline.Pipeline([('std_scaler', preprocessing.StandardScaler()), ('model', mm)]) if scaler else mm).fit(fts)


@pytest.mark.parametrize('D', [3, 16, 17, 40, 189])
@pytest.mark.parametrize('scaler', [False, True])
@pytest.mark.parametrize('covariance', COVARIANCES)
@pytest.mark.parametrize('kind', KINDS)
def test_device_predict_matches_sklearn(kind, covariance, scaler, D):
    from pyimsegm_b200.graph_cuts import DeviceClassModel
    model = fitted_model(kind, covariance, scaler, D)
    X = evaluation_set(model, D)
    extra = make_data(D, seed=7)
    while len(X) % 96 == 0 or len(X) % 128 == 0 or len(X) % 8 == 0:     # not a multiple of any tile of the kernels
        X = np.vstack([X, extra[len(X) % len(extra)]])
    got = DeviceClassModel(model).predict_proba(X)
    np.testing.assert_allclose(got, model.predict_proba(np.nan_to_num(X)), rtol=1e-9, atol=1e-9)


@pytest.mark.parametrize('D', [5, 16, 17, 189])
def test_rows_beyond_the_device_count_are_untouched(D):
    from pyimsegm_b200.engine import get_engine
    from pyimsegm_b200.graph_cuts import DeviceClassModel
    eng = get_engine()
    model = fitted_model('gm', 'full', True, D) if D != 5 else _shared_model(make_data(5), 3)
    dcm = DeviceClassModel(model)
    X = make_data(D, seed=3)[:301]
    n = 187
    d_feat = eng.to_device(X, 'test_feat')
    d_n = eng.to_device(np.array([n], dtype=np.int32), 'test_n')
    eng.buf('proba', (len(X), 3), eng.torch.float64).fill_(-7.0)
    proba = eng.to_host(eng.gmm_predict(d_feat, dcm.device_params(eng), 3, d_n=d_n)).copy()
    np.testing.assert_allclose(proba[:n], model.predict_proba(X[:n]), rtol=1e-9, atol=1e-9)
    assert (proba[n:] == -7.0).all()


@pytest.mark.parametrize('case', ['config1', 'config2_full'])
def test_single_image_device_model_equals_host_model(case):
    from pyimsegm_b200 import pipelines as pl
    from pyimsegm_b200.graph_cuts import DeviceClassModel
    if case == 'config1':
        img, K, sp = synth_disc(512, 512, seed=0), 2, 25
    else:
        img, K, sp = synth_regions(2048, 2048, seed=2)[0], 3, 29
    feats = {'color': ['mean']}
    _, fts = pl.compute_color2d_superpixels_features(img, feats, sp_size=sp, sp_regul=0.2)
    model = _shared_model(fts, K)
    segm, soft = pl.segment_color2d_slic_features_model_graphcut(img, model, feats, sp_size=sp, sp_regul=0.2, gc_regul=1.)
    segm_d, soft_d = pl.segment_color2d_slic_features_model_graphcut(img, DeviceClassModel(model), feats, sp_size=sp, sp_regul=0.2,
                                                                     gc_regul=1.)
    assert np.array_equal(segm_d, segm)
    np.testing.assert_allclose(soft_d, soft, rtol=0, atol=1e-9)


def test_device_path_never_calls_the_host_model(monkeypatch):
    """with the wrapped object's predict_proba made to raise, the single-image call, the batch and segment_resident still run; the
    batch gives what the per-image calls give"""
    from pyimsegm_b200 import pipelines as pl
    from pyimsegm_b200.engine import get_engine
    from pyimsegm_b200.graph_cuts import DeviceClassModel
    imgs = [synth_regions(200, 264, seed=s)[0] for s in (51, 52, 53, 54)]
    feats = {'color': ['mean', 'std']}
    model, _ = pl.estim_model_classes_group(imgs, 3, feats, sp_size=16, sp_regul=0.2)
    dcm = DeviceClassModel(model)

    def refuse(*_):
        raise AssertionError('the host model was called')

    monkeypatch.setattr(model, 'predict_proba', refuse)
    single = [pl.segment_color2d_slic_features_model_graphcut(im, dcm, feats, sp_size=16, sp_regul=0.2) for im in imgs]
    batch = pl.segment_images_batch(imgs, dict_features=feats, sp_size=16, sp_regul=0.2, model_pipeline=dcm)
    for (segm, soft), (segm_b, soft_b) in zip(single, batch):
        assert np.array_equal(segm_b, segm)
        np.testing.assert_allclose(soft_b, soft, rtol=1e-6, atol=1e-9)   # the colour statistics use floating-point atomics
    eng = get_engine()
    d_segm, d_soft = pl.segment_resident(eng.to_device(imgs[0].astype(np.float64)), dcm, feats, sp_size=16, sp_regul=0.2)
    assert np.array_equal(eng.to_host(d_segm), single[0][0])


def test_cuda_graph_replay_with_device_models():
    """the same configuration three times (eager, capture, replay) gives the eager result; two different models alternating on
    the same image each keep giving their own result"""
    from pyimsegm_b200 import pipelines as pl
    from pyimsegm_b200.graph_cuts import DeviceClassModel
    img, _ = synth_regions(160, 208, seed=61)
    feats = {'color': ['mean']}
    _, fts = pl.compute_color2d_superpixels_features(img, feats, sp_size=16, sp_regul=0.2)
    a = DeviceClassModel(_shared_model(fts, 3))
    b = DeviceClassModel(_shared_model(fts, 2, covariance='diag', scaler=False))
    pl.USE_CUDA_GRAPHS = False
    try:
        eager = {m: pl.segment_color2d_slic_features_model_graphcut(img, m, feats, sp_size=16, sp_regul=0.2) for m in (a, b)}
    finally:
        pl.USE_CUDA_GRAPHS = True
    runs = [pl.segment_color2d_slic_features_model_graphcut(img, a, feats, sp_size=16, sp_regul=0.2) for _ in range(3)]
    assert any(isinstance(v, tuple) and k[0] == 'probabilities' and k[5] == ('predict', a.digest) for k, v in pl._GRAPHS.items()), \
        'no CUDA graph was captured for the device model'
    for segm, soft in runs:
        assert np.array_equal(segm, eager[a][0])
        np.testing.assert_allclose(soft, eager[a][1], rtol=1e-6, atol=1e-9)
    for m in (b, a, b, a, b, a):
        segm, soft = pl.segment_color2d_slic_features_model_graphcut(img, m, feats, sp_size=16, sp_regul=0.2)
        assert soft.shape[-1] == m.n_classes
        assert np.array_equal(segm, eager[m][0])
        np.testing.assert_allclose(soft, eager[m][1], rtol=1e-6, atol=1e-9)


def test_config3_width_device_model_equals_host_model():
    """colour + full Leung-Malik statistics (D = 189), a diagonal-covariance shared model: the device evaluation against the host
    model on the same device features"""
    import bench
    from pyimsegm_b200 import pipelines as pl
    from pyimsegm_b200.graph_cuts import DeviceClassModel
    img = bench.synth_texture_image(77, 160, 224, n_classes=4, cell=32)
    feats = {'color': ('mean', 'std', 'energy'), 'tLM': ('mean', 'std', 'energy')}
    _, fts = pl.compute_color2d_superpixels_features(img, feats, sp_size=16, sp_regul=0.2)
    assert fts.shape[1] == 189
    model = _shared_model(fts, 4, covariance='diag', reg_covar=1e-3)
    segm, soft = pl.segment_color2d_slic_features_model_graphcut(img, model, feats, sp_size=16, sp_regul=0.2, gc_regul=1.)
    segm_d, soft_d = pl.segment_color2d_slic_features_model_graphcut(img, DeviceClassModel(model), feats, sp_size=16, sp_regul=0.2,
                                                                     gc_regul=1.)
    assert np.array_equal(segm_d, segm)
    np.testing.assert_allclose(soft_d, soft, rtol=0, atol=1e-9)


@pytest.mark.parametrize('features', [{'color': ['mean', 'std']}, {'color': ['mean'], 'tLM_short': ['mean']}])
def test_banded_entry_with_a_given_model_matches_single_gpu(features):
    from pyimsegm_b200 import pipelines as pl
    from pyimsegm_b200.graph_cuts import DeviceClassModel
    from pyimsegm_b200.tiled import segment_color2d_slic_features_model_graphcut_tiled
    img, _ = synth_regions(600, 512, seed=17)
    _, fts = pl.compute_color2d_superpixels_features(img, features, sp_size=20, sp_regul=0.2)
    model = _shared_model(fts, 3, covariance='diag' if len(fts[0]) > 16 else 'full')
    dcm = DeviceClassModel(model)
    segm, soft = pl.segment_color2d_slic_features_model_graphcut(img, dcm, features, sp_size=20, sp_regul=0.2)
    for m in (dcm, model):      # a raw model is wrapped on entry
        got, got_soft, (lo, hi) = segment_color2d_slic_features_model_graphcut_tiled(img, m, features, sp_size=20, sp_regul=0.2,
                                                                                    bands_per_rank=3)
        assert (lo, hi) == (0, 600)
        if 'tLM_short' in features:
            assert (got == segm).mean() > 0.999
            np.testing.assert_allclose(got_soft, soft, rtol=1e-4, atol=1e-6)
        else:
            assert np.array_equal(got, segm)
            np.testing.assert_allclose(got_soft, soft, rtol=1e-6, atol=1e-9)
