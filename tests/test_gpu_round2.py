"""Round-2 GPU parity tests: the API holes the round-1 review listed (gray images, tLM median / meanGrad, classes_ relabel, the group
model on the device path) and the configurations that had no parity test (Leung-Malik on an image larger than the sigma-150
kernel, a config-3 shaped end-to-end run)."""
import os

import numpy as np
import pytest

from conftest import synth_regions

pytestmark = pytest.mark.gpu
GOLD_LM = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden', 'lm_large.npz')


def test_gray2d_features_reference_doctest():
    """imsegm/descriptors.py:1179-1197 (golden values of compute_selected_features_gray2d)"""
    from pyimsegm_b200 import descriptors as ds
    image = np.zeros((2, 10))
    image[0, 2:6] = 1
    image[1, 3:7] = 3
    segm = np.array([[0] * 5 + [1] * 5] * 2)
    features, names = ds.compute_selected_features_gray2d(image, segm, {'color': ('mean', 'std', 'median')})
    np.testing.assert_allclose(np.round(features, 3), [[0.9, 1.136, 0.5], [0.7, 1.187, 0.]])
    features, _ = ds.compute_selected_features_gray2d(image, segm, {'tLM_short': ('mean', 'std', 'energy')})
    assert features.shape == (2, 45)
    features, _ = ds.compute_selected_features_gray2d(image, segm)
    assert features.shape == (2, 105)
    features, _ = ds.compute_selected_features_img2d(image, segm, {'color': ('mean', )})
    assert features.shape == (2, 1)


def test_gray_image_through_the_pipeline(oracle):
    """a 2-D gray image: SLIC replicates it to three channels (superpixels.py:50-51), features go through the gray-3D statistics"""
    from pyimsegm_b200 import pipelines as pl
    img, _ = synth_regions(160, 200, seed=11)
    gray = img[..., 0]
    slic, fts = pl.compute_color2d_superpixels_features(gray, {'color': ('mean', 'std')}, sp_size=16, sp_regul=0.2)
    assert np.array_equal(slic, oracle.segment_slic_img2d(gray, 16, 0.2))
    nb = slic.max() + 1
    want = np.array([gray[slic == k].mean() for k in range(nb)])
    np.testing.assert_allclose(fts[:, 0], want, rtol=1e-6)
    segm, soft = pl.pipe_color2d_slic_features_model_graphcut(gray, 2, {'color': ('mean', )}, sp_size=16)
    assert segm.shape == gray.shape and soft.shape == gray.shape + (2, )


def test_default_feature_set_runs_and_lm_median_matches_oracle(oracle):
    """FEATURES_SET_ALL is the default of compute_selected_features_color2d (descriptors.py:1207): tLM with median / meanGrad goes
    through the materialised responses; against the SciPy oracle (responses float64 on both sides)"""
    from oracle import texture as otex
    from pyimsegm_b200 import descriptors as ds
    h, w, step = 30, 20, 5
    rng = np.random.RandomState(0)
    seg = (np.arange(h)[:, None] // step) * (w // step) + np.arange(w)[None, :] // step
    img = rng.random_sample((h, w, 3))
    fts, names = ds.compute_selected_features_color2d(img, seg)
    assert fts.shape == (24, 15 + 300) and len(names) == 315          # reference doctest :1235-1239: (2, 315) columns
    flags = ('mean', 'std', 'median', 'meanGrad')
    got, gnames = ds.compute_texture_desc_lm_img2d_clr(img, seg, flags, 'short')
    want, wnames = otex.texture_desc_lm(img, seg, flags, 'short')
    assert gnames == wnames and got.shape == want.shape == (24, 15 * 12)
    np.testing.assert_allclose(got, want, rtol=1e-5, atol=1e-7)


def test_classes_relabel_of_a_supplied_classifier(oracle):
    """imsegm/pipelines.py:238-239: a model with `classes_` maps the graph-cut indices through it (single image and batch API)"""
    from sklearn import mixture, pipeline, preprocessing
    from pyimsegm_b200 import pipelines as pl

    class WithClasses(object):
        def __init__(self, inner, classes):
            self.inner, self.classes_ = inner, np.asarray(classes)

        def predict_proba(self, x):
            return self.inner.predict_proba(x)

    img, _ = synth_regions(192, 256, seed=5)
    feats = {'color': ['mean']}
    _, fts_o = oracle.compute_color2d_superpixels_features(img, ('mean',), 16, 0.2)
    model = pipeline.Pipeline([('std_scaler', preprocessing.StandardScaler()),
                               ('model', mixture.GaussianMixture(3, covariance_type='full', random_state=0))]).fit(fts_o)
    plain, _ = pl.segment_color2d_slic_features_model_graphcut(img, model, feats, sp_size=16, sp_regul=0.2)
    classes = np.array([7, 3, 11])
    wrapped = WithClasses(model, classes)
    relab, _ = pl.segment_color2d_slic_features_model_graphcut(img, wrapped, feats, sp_size=16, sp_regul=0.2)
    assert np.array_equal(relab, classes[plain])
    batch = pl.segment_images_batch([img, img], dict_features=feats, sp_size=16, sp_regul=0.2, model_pipeline=wrapped)
    assert all(np.array_equal(b[0], classes[plain]) for b in batch)


def test_group_model_features_equal_the_oracle_concatenation(oracle):
    """estim_model_classes_group (imsegm/pipelines.py:113-157): per-image features = the oracle's, the model is fitted on their
    concatenation (order of the images) and classifies every superpixel"""
    from pyimsegm_b200 import pipelines as pl
    imgs = [synth_regions(128, 160, seed=s)[0] for s in (21, 22, 23)]
    feats = {'color': ('mean', 'std')}
    model, list_fts = pl.estim_model_classes_group(imgs, 3, feats, sp_size=16, sp_regul=0.2)
    assert len(list_fts) == 3
    for im, f in zip(imgs, list_fts):
        _, want = oracle.compute_color2d_superpixels_features(im, ('mean', 'std'), 16, 0.2)
        assert f.shape == want.shape
        np.testing.assert_allclose(f, want, rtol=1e-6, atol=1e-9)
    proba = model.predict_proba(np.concatenate(list_fts))
    assert proba.shape == (sum(len(f) for f in list_fts), 3)
    np.testing.assert_allclose(proba.sum(1), 1.0, rtol=1e-9)
    segm, _ = pl.segment_color2d_slic_features_model_graphcut(imgs[0], model, feats, sp_size=16, sp_regul=0.2)
    assert segm.shape == imgs[0].shape[:2] and len(np.unique(segm)) >= 2


@pytest.mark.skipif(not os.path.isfile(GOLD_LM), reason='tests/golden/lm_large.npz not generated')
def test_lm_full_bank_on_an_image_larger_than_the_background_kernel():
    """Leung-Malik descriptors of a 1280 x 1280 image (both axes longer than the 1201-tap sigma-150 kernel), full bank, against
    the REFERENCE's own compute_texture_desc_lm_img2d_clr (tests/golden/make_lm_large_golden.py ran it).  Every feature within 1e-4
    of the response scale (rms = sqrt of the largest energy) of its battery and channel."""
    import sys
    sys.path.insert(0, os.path.dirname(GOLD_LM))
    from make_lm_large_golden import make_inputs
    from pyimsegm_b200 import texture
    gold = np.load(GOLD_LM)
    img, seg = make_inputs()
    assert abs(float(img.sum()) - float(gold['img_sum'])) < 1e-6 * float(gold['img_sum']) and int(seg.sum()) == int(gold['seg_sum'])
    fts, names = texture.compute_texture_desc_lm_img2d_clr(img, seg, ('mean', 'std', 'energy'), 'normal')
    assert list(names) == list(gold['names']) and fts.shape[0] == int(gold['nb_segments'])
    got, want = fts[gold['rows']], gold['features']
    rms = np.sqrt(gold['energy_max'])                       # [20 batteries, 3 channels]
    scale = np.ones((20, 3, 3))
    scale[:, 0, :] = rms
    scale[:, 1, :] = rms
    scale[:, 2, :] = rms ** 2
    err = np.abs(got - want).reshape(len(want), 20, 3, 3) / scale[None]
    assert err.max() < 1e-4, 'max error relative to the battery response scale: %g at %r' % (err.max(), np.unravel_index(err.argmax(), err.shape))


def test_config3_shaped_pipeline_with_a_shared_model(oracle):
    """BASELINE config 3 in small: colour + full Leung-Malik statistics (D = 189), 4 classes, one model shared by both sides
    (fitted on the oracle's features).  The texture features differ by ~1e-6, so superpixels whose two best classes are nearly
    tied may flip: label maps must agree on > 99.5 % of the pixels, segm_soft within 1e-3."""
    import bench
    from oracle import texture as otex
    from sklearn import mixture, pipeline, preprocessing
    from pyimsegm_b200 import pipelines as pl
    img = bench.synth_texture_image(77, 160, 224, n_classes=4, cell=32)
    feats = {'color': ('mean', 'std', 'energy'), 'tLM': ('mean', 'std', 'energy')}
    slic_o, col_o = oracle.compute_color2d_superpixels_features(img, ('mean', 'std', 'energy'), 16, 0.2)
    lm_o, _ = otex.texture_desc_lm(img, slic_o, ('mean', 'std', 'energy'), 'normal')
    fts_o = np.hstack([col_o, lm_o])
    assert fts_o.shape[1] == 189
    slic_g, fts_g = pl.compute_color2d_superpixels_features(img, feats, sp_size=16, sp_regul=0.2)
    assert np.array_equal(slic_g, slic_o) and fts_g.shape == fts_o.shape
    model = pipeline.Pipeline([('std_scaler', preprocessing.StandardScaler()),
                               ('model', mixture.GaussianMixture(4, covariance_type='diag', random_state=0, reg_covar=1e-3))]).fit(fts_o)
    proba_o = model.predict_proba(fts_o)
    labels_o = oracle.segment_graph_cut_general(slic_o, proba_o, 1., 'model')
    segm, soft = pl.segment_color2d_slic_features_model_graphcut(img, model, feats, sp_size=16, sp_regul=0.2, gc_regul=1.)
    agree = (segm == labels_o[slic_o]).mean()
    assert agree > 0.995, 'label maps agree on %.4f of the pixels' % agree
    assert np.abs(soft - proba_o[slic_o]).max() < 1e-3


def test_cuda_graph_replay_equals_eager_launches():
    """pipelines._graph_call: the device part of the path captured once and replayed per image (batch API and
    segment_resident) must give exactly what the eager launches give, for every image of the batch"""
    from pyimsegm_b200 import pipelines as pl
    imgs = [synth_regions(200, 264, seed=s)[0] for s in (31, 32, 33, 34, 35)]
    feats = {'color': ['mean']}
    pl.USE_CUDA_GRAPHS = False
    try:
        eager = pl.segment_images_batch(imgs, 3, feats, sp_size=16, sp_regul=0.2)
    finally:
        pl.USE_CUDA_GRAPHS = True
    for _ in range(3):      # eager -> capture -> replay on every one of the three stream engines
        graph = pl.segment_images_batch(imgs * 2, 3, feats, sp_size=16, sp_regul=0.2)
    assert any(isinstance(v, tuple) for v in pl._GRAPHS.values()), 'no CUDA graph was captured'
    for i, (segm, soft) in enumerate(graph):
        assert np.array_equal(segm, eager[i % len(imgs)][0])
        np.testing.assert_allclose(soft, eager[i % len(imgs)][1], rtol=1e-6, atol=1e-9)   # the statistics use floating-point atomics


def test_graph_replay_survives_other_configurations_in_between():
    """a captured graph keeps its own constants (seed grid) and buffers: running another image size / superpixel size on the same
    engine between two replays must not change what the replay computes"""
    from pyimsegm_b200 import pipelines as pl
    img, _ = synth_regions(160, 208, seed=41)
    other, _ = synth_regions(300, 260, seed=42)
    feats = {'color': ['mean']}
    runs = [pl.pipe_color2d_slic_features_model_graphcut(img, 3, feats, sp_size=16, sp_regul=0.2) for _ in range(3)]   # eager, capture, replay
    pl.pipe_color2d_slic_features_model_graphcut(other, 3, feats, sp_size=20, sp_regul=0.3)          # grows buffers, new seed grid
    pl.compute_color2d_superpixels_features(other, feats, sp_size=11, sp_regul=0.2)
    again = pl.pipe_color2d_slic_features_model_graphcut(img, 3, feats, sp_size=16, sp_regul=0.2)
    for segm, soft in runs[1:] + [again]:
        assert np.array_equal(segm, runs[0][0])
        np.testing.assert_allclose(soft, runs[0][1], rtol=1e-6, atol=1e-9)
