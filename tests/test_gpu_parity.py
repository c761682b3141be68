"""GPU parity tests proper: the CUDA path (through the C-ABI) against the CPU oracle on the same seeded inputs."""
import os

import numpy as np
import pytest

from conftest import synth_disc, synth_regions

pytestmark = pytest.mark.gpu

#: outputs of the reference's Cython module for inputs built below (tests/golden/make_cython_goldens.py)
REF_CYTHON = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden', 'reference_cython.npz'))


@pytest.fixture(scope='module')
def eng():
    from pyimsegm_b200.engine import get_engine
    return get_engine()


def _slic_both(oracle, img, sp_size, regul, slico=False):
    from pyimsegm_b200 import superpixels as sp
    got = sp.segment_slic_img2d(img, sp_size, regul, slico)
    want = oracle.segment_slic_img2d(img, sp_size, regul, slico)
    return got, want


@pytest.mark.parametrize('case', ['rand', 'disc', 'flat', 'u8', 'gray', 'odd', 'slico', 'slico_flat'])
def test_slic_label_map_bit_exact(oracle, case):
    rng = np.random.RandomState(0)
    if case == 'rand':
        img = rng.random_sample((125, 150, 3)) / 2.
        img[:, :75] += 0.5
        args = (20, 0.2)
    elif case == 'disc':
        img, args = synth_disc(256, 256), (25, 0.2)
    elif case == 'flat':
        img, args = synth_disc(200, 240, noise=0.0), (16, 0.3)
    elif case == 'u8':
        img, args = (synth_disc(256, 256) * 255).astype(np.uint8), (30, 0.3)
    elif case == 'gray':
        img, args = synth_disc(128, 160)[..., 0], (20, 0.2)
    elif case == 'slico':
        img, args = synth_regions(180, 230, seed=6)[0], (15, 0.2, True)       # SLICO / ASLIC (slic_zero=True)
    elif case == 'slico_flat':
        img, args = synth_disc(150, 170, noise=0.0), (14, 0.3, True)
    else:
        img, args = synth_regions(203, 317, seed=5)[0], (17, 0.25)
    got, want = _slic_both(oracle, img, *args)
    assert got.dtype == np.int64 and got.shape == img.shape[:2]
    assert np.array_equal(got, want)
    assert set(np.unique(got)) == set(range(got.max() + 1))


def test_color_stats_match_oracle_and_reference_module(oracle):
    from pyimsegm_b200 import descriptors as ds
    img, _ = synth_regions(300, 400, seed=3)
    seg = oracle.segment_slic_img2d(img, 20, 0.2)
    for im in (img, (img * 255).astype(np.uint8), img.astype(np.float32)):
        for name, fn_o in (('mean', oracle.color2d_mean), ('energy', oracle.color2d_energy), ('std', oracle.color2d_std)):
            got = getattr(ds, 'cython_img2d_color_%s' % name)(im, seg)
            np.testing.assert_allclose(got, fn_o(im, seg), rtol=1e-6, atol=1e-9)
    np.testing.assert_allclose(ds.cython_img2d_color_energy(img, seg), REF_CYTHON['slic_energy'], rtol=1e-6, atol=1e-9)
    fts, names = ds.compute_image2d_color_statistic(img, seg, ('mean', 'std', 'energy', 'meanGrad'))
    want = oracle.image2d_color_statistic(img, seg, ('mean', 'std', 'energy', 'meanGrad'))
    assert fts.shape == (seg.max() + 1, 12) and len(names) == 12
    np.testing.assert_allclose(fts, want, rtol=1e-6, atol=1e-9)


def test_reference_doctest_goldens_descriptors():
    """imsegm/descriptors.py:218-283 and :796-813"""
    from pyimsegm_b200 import descriptors as ds
    image = np.zeros((2, 10, 3))
    image[:, 2:6, 0] = 1
    image[:, 3:7, 1] = 3
    image[:, 4:9, 2] = 2
    segm = np.array([[0] * 5 + [1] * 5] * 2)
    np.testing.assert_allclose(ds.cython_img2d_color_mean(image, segm), [[0.6, 1.2, 0.4], [0.2, 1.2, 1.6]], rtol=1e-12)
    np.testing.assert_allclose(ds.cython_img2d_color_energy(image, segm), [[0.6, 3.6, 0.8], [0.2, 3.6, 3.2]], rtol=1e-12)
    np.testing.assert_allclose(ds.cython_img2d_color_std(image, segm),
                               [[0.48989794, 1.46969383, 0.80000003], [0.40000001, 1.46969383, 0.80000001]], rtol=1e-7)
    features, names = ds.compute_image2d_color_statistic(image, segm)
    assert names[:3] == ['color-ch1_mean', 'color-ch2_mean', 'color-ch3_mean'] and features.shape == (2, 15)
    want = [[0.6, 1.2, 0.4, 0.5, 1.5, 0.8, 0.6, 3.6, 0.8, 1.0, 0.0, 0.0, 0.2, 0.6, 0.4],
            [0.2, 1.2, 1.6, 0.4, 1.5, 0.8, 0.2, 3.6, 3.2, 0.0, 0.0, 2.0, -0.2, -0.6, -0.6]]
    assert np.round(features, 1).tolist() == want


def test_reference_doctest_goldens_graph():
    """imsegm/superpixels.py:163-168, :211-215; imsegm/graph_cuts.py:587-609, :687-716"""
    from pyimsegm_b200 import graph_cuts as gc
    from pyimsegm_b200 import superpixels as sp
    grid = np.array([[0] * 5 + [1] * 5, [2] * 5 + [3] * 5])
    v, edges = sp.make_graph_segm_connect_grid2d_conn4(grid)
    assert v.tolist() == [0, 1, 2, 3] and [list(map(int, e)) for e in edges] == [[0, 1], [0, 2], [1, 3], [2, 3]]
    segm = np.array([[0] * 6 + [1] * 5, [0] * 6 + [2] * 5])
    assert sp.superpixel_centers(segm) == [(0.5, 2.5), (0.0, 8.0), (1.0, 8.0)]
    segments = np.array([[0] * 3 + [1] * 5 + [2] * 4, [4] * 4 + [5] * 5 + [6] * 3])
    np.random.seed(0)
    _ = np.random.random(segments.shape + (3,)) * 255
    features = np.random.random((segments.max() + 1, 15)) * 10
    proba = np.random.random((segments.max() + 1, 2))
    edges, weights = gc.compute_edge_weights(segments)
    assert edges.tolist() == [[0, 1], [1, 2], [0, 4], [1, 4], [1, 5], [2, 5], [4, 5], [2, 6], [5, 6]]
    assert np.round(weights, 2).tolist() == [1.0] * 9
    _, weights = gc.compute_edge_weights(segments, edge_type='spatial')
    assert np.round(weights, 3).tolist() == [0.776, 0.69, 2.776, 0.853, 2.194, 0.853, 0.69, 2.776, 0.776]
    _, weights = gc.compute_edge_weights(segments, features=features, edge_type='features')
    assert np.round(weights, 3).tolist() == [0.031, 0.005, 0.051, 0.032, 0.096, 0.013, 0.018, 0.033, 0.013]
    _, weights = gc.compute_edge_weights(segments, proba=proba, edge_type='model')
    assert np.round(weights, 3).tolist() == [0.001, 0.028, 1.122, 0.038, 0.117, 0.688, 0.487, 1.152, 0.282]
    # graph cut goldens
    np.random.seed(0)
    segments = np.array([[0] * 3 + [2] * 3 + [4] * 3 + [6] * 3 + [8] * 3, [1] * 3 + [3] * 3 + [5] * 3 + [7] * 3 + [9] * 3])
    proba = np.array([[0.1] * 6 + [0.9] * 4, [0.9] * 6 + [0.1] * 4], dtype=float).T
    proba += (0.5 - np.random.random(proba.shape)) * 0.2
    labels = gc.segment_graph_cut_general(segments, proba, gc_regul=0., edge_type='')
    assert labels.tolist() == [1, 1, 1, 1, 1, 1, 0, 0, 0, 0]
    labels = gc.segment_graph_cut_general(segments, proba, gc_regul=1., edge_type='spatial')
    assert labels.dtype == np.int32
    assert labels[segments].tolist() == [[1] * 9 + [0] * 6] * 2


def _random_graph_problem(rng, n, k, deg=3.0, strong=True):
    m = int(n * deg)
    a = rng.randint(0, n, m)
    b = rng.randint(0, n, m)
    keep = a != b
    pairs = np.unique(np.stack([np.minimum(a, b)[keep], np.maximum(a, b)[keep]], 1), axis=0)
    w = rng.random_sample(len(pairs)) * 2 + 1e-3
    p = rng.dirichlet(np.ones(k) * (0.3 if strong else 2.0), n)
    return pairs.astype(np.int32), w, p


@pytest.mark.parametrize('n,k,regul', [(12, 2, 1.0), (300, 3, 0.8), (2000, 4, 2.0), (7000, 3, 1.5), (9000, 5, 3.0)])
def test_alpha_expansion_labels_bit_exact(oracle, n, k, regul):
    from pyimsegm_b200 import graph_cuts as gc
    rng = np.random.RandomState(n + k)
    edges, w, p = _random_graph_problem(rng, n, k)
    unary = gc.compute_unary_cost(p)
    pw = gc.compute_pairwise_cost(regul, p.shape)
    want, e_want, _ = oracle.cut_general_graph(edges, w, unary, pw, n_iter=-1, return_energy=True)
    got = gc.cut_general_graph(edges, w, unary, pw, n_iter=-1)
    assert got.dtype == np.int32
    assert np.array_equal(got, want)
    got2 = gc.cut_general_graph(edges, w, unary, pw, n_iter=999)
    want2 = oracle.cut_general_graph(edges, w, unary, pw, n_iter=999)
    assert np.array_equal(got2, want2)


def test_energies_match_oracle(oracle):
    from pyimsegm_b200 import graph_cuts as gc
    img, _ = synth_regions(256, 320, seed=4)
    seg = oracle.segment_slic_img2d(img, 16, 0.2)
    rng = np.random.RandomState(1)
    proba = rng.dirichlet(np.ones(3), seg.max() + 1)
    for et in ('model', 'model_l1', 'model_l2', 'spatial', ''):
        e_g, w_g = gc.compute_edge_weights(seg, proba=proba, edge_type=et)
        e_o, w_o = oracle.edge_weights(seg, proba, et)
        assert np.array_equal(e_g, e_o)
        np.testing.assert_allclose(w_g, w_o, rtol=1e-9)
    labels = gc.segment_graph_cut_general(seg, proba, gc_regul=2., edge_type='model')
    want = oracle.segment_graph_cut_general(seg, proba, 2., 'model')
    assert np.array_equal(labels, want)


def test_pipeline_with_shared_model_equals_oracle(oracle):
    """entry point 3.2 (imsegm/pipelines.py:160): same fitted model on both sides, label maps must be identical"""
    from sklearn import mixture, pipeline, preprocessing
    from pyimsegm_b200 import pipelines as pl
    img, _ = synth_regions(384, 512, seed=7)
    feats = {'color': ['mean']}
    slic_o, fts_o = oracle.compute_color2d_superpixels_features(img, ('mean',), 24, 0.2)
    model = pipeline.Pipeline([('std_scaler', preprocessing.StandardScaler()),
                               ('model', mixture.GaussianMixture(3, covariance_type='full', random_state=0))]).fit(fts_o)
    segm, soft = pl.segment_color2d_slic_features_model_graphcut(img, model, feats, sp_size=24, sp_regul=0.2, gc_regul=1.)
    segm_o, soft_o, _, _ = oracle.segment_with_model(img, model.predict_proba, ('mean',), 24, 0.2, 1., 'model')
    assert segm.shape == img.shape[:2] and soft.shape == img.shape[:2] + (3,)
    assert np.array_equal(segm, segm_o)
    np.testing.assert_allclose(soft, soft_o, rtol=1e-6, atol=1e-9)
    # the self-estimating pipeline: shapes + sanity (the GMM is unseeded in the reference, so no label parity)
    segm2, soft2 = pl.pipe_color2d_slic_features_model_graphcut(img, 3, feats, sp_size=24)
    assert segm2.shape == img.shape[:2] and soft2.shape == img.shape[:2] + (3,)
    np.testing.assert_allclose(soft2.sum(-1), 1.0, rtol=1e-9)


def test_device_gmm_matches_sklearn_from_shared_start():
    """estim_class_model (imsegm/graph_cuts.py:73-163): same EM as sklearn's GaussianMixture when both start from the
    same hard assignment; tolerance 1e-6 on parameters and probabilities (EM amplifies summation-order noise)"""
    from sklearn import mixture, preprocessing
    from pyimsegm_b200 import graph_cuts as gc
    rng = np.random.RandomState(3)
    K, D = 3, 3
    centers = np.array([[0.2, 0.25, 0.18], [0.5, 0.52, 0.47], [0.8, 0.83, 0.78]])
    X = np.concatenate([c + rng.normal(0, 0.04, (n, D)) for c, n in zip(centers, (1500, 2200, 1300))])
    y0 = rng.randint(0, K, len(X))
    y0[:60] = np.repeat(np.arange(K), 20)
    near = ((X[:, None, :] - centers[None]) ** 2).sum(-1).argmin(1)
    y0[::2] = near[::2]                       # a half-informed start so that EM has real work to do
    model = gc.estim_class_model_device(X, K, use_scaler=True, max_iter=99, init_labels=y0)
    scaler, gmm = model.named_steps['std_scaler'], model.named_steps['model']
    Xs = preprocessing.StandardScaler().fit(X)
    np.testing.assert_allclose(scaler.mean_, Xs.mean_, rtol=1e-12)
    np.testing.assert_allclose(scaler.scale_, Xs.scale_, rtol=1e-12)
    Z = Xs.transform(X)
    resp = np.eye(K)[y0]
    nk = resp.sum(0) + 10 * np.finfo(float).eps
    means0 = resp.T @ Z / nk[:, None]
    covs0 = np.array([((resp[:, k, None] * (Z - means0[k])).T @ (Z - means0[k])) / nk[k] + 1e-6 * np.eye(D) for k in range(K)])
    ref = mixture.GaussianMixture(K, covariance_type='full', max_iter=99, n_init=1, weights_init=nk / len(Z), means_init=means0,
                                  precisions_init=np.linalg.inv(covs0)).fit(Z)
    assert gmm.n_iter_ == ref.n_iter_ and gmm.converged_ == ref.converged_
    np.testing.assert_allclose(gmm.weights_, ref.weights_, rtol=1e-6)
    np.testing.assert_allclose(gmm.means_, ref.means_, rtol=1e-6, atol=1e-8)
    np.testing.assert_allclose(gmm.covariances_, ref.covariances_, rtol=1e-6, atol=1e-9)
    np.testing.assert_allclose(gmm.lower_bound_, ref.lower_bound_, rtol=1e-8)
    np.testing.assert_allclose(model.predict_proba(X), ref.predict_proba(Z), rtol=1e-5, atol=1e-9)
    # the unseeded-in-the-reference default: k-means++ start on the device, 9 restarts; must separate the three blobs
    model2 = gc.estim_class_model(X, K)
    lab = model2.predict_proba(X).argmax(1)
    assert len(model2.named_steps['model'].weights_) == K
    purity = sum(np.bincount(lab[near == k], minlength=K).max() for k in range(K)) / len(X)
    assert purity > 0.98


@pytest.mark.parametrize('D,K', [(40, 3), (189, 4)])
def test_device_gmm_large_d_matches_sklearn_from_shared_start(D, K):
    """the large-D path of the device class model (batched FP64 GEMMs + Cholesky; colour + Leung-Malik features give
    D = 189): same EM as sklearn from the same hard start, tolerance 1e-6 as for the small path"""
    from sklearn import mixture, preprocessing
    from pyimsegm_b200 import graph_cuts as gc
    rng = np.random.RandomState(D)
    sizes = (700, 900, 600, 800)[:K]
    centers = rng.normal(0, 1.0, (K, D))
    mix = rng.normal(0, 0.3, (K, D, D)) / np.sqrt(D)
    X = np.concatenate([c + rng.normal(0, 1.0, (n, D)) @ (np.eye(D) * 0.4 + m) for c, m, n in zip(centers, mix, sizes)])
    truth = np.repeat(np.arange(K), sizes)
    y0 = truth.copy()
    flip = rng.rand(len(X)) < 0.3
    y0[flip] = rng.randint(0, K, flip.sum())       # a 70 % informed start so that EM has real work to do
    model = gc.estim_class_model_device(X, K, use_scaler=True, max_iter=99, init_labels=y0)
    gmm = model.named_steps['model']
    Z = preprocessing.StandardScaler().fit(X).transform(X)
    resp = np.eye(K)[y0]
    nk = resp.sum(0) + 10 * np.finfo(float).eps
    means0 = resp.T @ Z / nk[:, None]
    covs0 = np.array([((resp[:, k, None] * (Z - means0[k])).T @ (Z - means0[k])) / nk[k] + 1e-6 * np.eye(D) for k in range(K)])
    ref = mixture.GaussianMixture(K, covariance_type='full', max_iter=99, n_init=1, weights_init=nk / len(Z), means_init=means0,
                                  precisions_init=np.linalg.inv(covs0)).fit(Z)
    assert gmm.n_iter_ == ref.n_iter_ and gmm.converged_ == ref.converged_
    np.testing.assert_allclose(gmm.weights_, ref.weights_, rtol=1e-6)
    np.testing.assert_allclose(gmm.means_, ref.means_, rtol=1e-6, atol=1e-8)
    np.testing.assert_allclose(gmm.covariances_, ref.covariances_, rtol=1e-6, atol=1e-8)
    np.testing.assert_allclose(gmm.lower_bound_, ref.lower_bound_, rtol=1e-8)
    np.testing.assert_allclose(gmm.precisions_cholesky_, ref.precisions_cholesky_, rtol=1e-5, atol=1e-7)
    np.testing.assert_allclose(model.predict_proba(X), ref.predict_proba(Z), rtol=1e-5, atol=1e-9)
    # unseeded default (k-means++ on the device, 9 restarts): must recover the blobs
    lab = gc.estim_class_model(X, K).predict_proba(X).argmax(1)
    purity = sum(np.bincount(lab[truth == k], minlength=K).max() for k in range(K)) / len(X)
    assert purity > 0.97


def test_fully_resident_pipeline_is_consistent(oracle):
    """pipe_color2d_slic_features_model_graphcut with the device-fitted GMM: its own model, replayed through the
    shared-model entry point and through the oracle, must give the identical label map"""
    from pyimsegm_b200 import graph_cuts as gc
    from pyimsegm_b200 import pipelines as pl
    img, truth = synth_regions(320, 448, seed=11)
    feats = {'color': ['mean']}
    segm, soft = pl.pipe_color2d_slic_features_model_graphcut(img, 3, feats, sp_size=20, sp_regul=0.2, gc_regul=1.)
    assert segm.dtype == np.int32 and segm.shape == img.shape[:2] and soft.shape == img.shape[:2] + (3,)
    np.testing.assert_allclose(soft.sum(-1), 1.0, rtol=1e-9)
    # segmentation quality on the synthetic regions (labels are a permutation of the classes)
    conf = np.array([[np.sum((segm == a) & (truth == b)) for b in range(3)] for a in range(3)])
    assert conf.max(0).sum() / truth.size > 0.95
    # replay: fit the same model through the public estimator (same seed, same features) and use entry point 3.2
    slic, fts = pl.compute_color2d_superpixels_features(img, feats, sp_size=20, sp_regul=0.2)
    model = gc.estim_class_model(fts, 3)
    segm2, soft2 = pl.segment_color2d_slic_features_model_graphcut(img, model, feats, sp_size=20, sp_regul=0.2, gc_regul=1.)
    assert np.array_equal(segm, segm2)
    segm_o, _, _, _ = oracle.segment_with_model(img, model.predict_proba, ('mean',), 20, 0.2, 1., 'model')
    assert np.array_equal(segm, segm_o)


def test_full_size_config2_bit_exact(oracle):
    """BASELINE.json configs[1] at full size (2048x2048, sp_size 29, K = 3): SLIC label map and the final segmentation with
    a shared model are identical to the oracle's, descriptors within 1e-6"""
    from sklearn import mixture, pipeline, preprocessing
    from pyimsegm_b200 import pipelines as pl
    img, _ = synth_regions(2048, 2048, seed=2)
    feats = {'color': ['mean']}
    slic, fts = pl.compute_color2d_superpixels_features(img, feats, sp_size=29, sp_regul=0.2)
    slic_o, fts_o = oracle.compute_color2d_superpixels_features(img, ('mean',), 29, 0.2)
    assert np.array_equal(slic, slic_o)
    np.testing.assert_allclose(fts, fts_o, rtol=1e-6, atol=1e-9)
    assert 4500 < slic.max() + 1 < 5500
    model = pipeline.Pipeline([('std_scaler', preprocessing.StandardScaler()),
                               ('model', mixture.GaussianMixture(3, covariance_type='full', random_state=0))]).fit(fts_o)
    segm, soft = pl.segment_color2d_slic_features_model_graphcut(img, model, feats, sp_size=29, sp_regul=0.2, gc_regul=1.)
    proba = model.predict_proba(fts_o)
    labels_o = oracle.segment_graph_cut_general(slic_o, proba, 1., 'model')
    assert np.array_equal(segm, labels_o[slic_o])
    np.testing.assert_allclose(soft[::7, ::5], proba[slic_o][::7, ::5], rtol=1e-6, atol=1e-9)


def test_config1_reference_cpu_case(oracle):
    """BASELINE.json configs[0]: 512x512 synthetic disc, 2 classes, sp_size 25 (SURVEY.md section 8d config 1)"""
    from pyimsegm_b200 import graph_cuts as gc
    from pyimsegm_b200 import pipelines as pl
    img = synth_disc(512, 512, seed=0)
    feats = {'color': ['mean']}
    segm, soft = pl.pipe_color2d_slic_features_model_graphcut(img, 2, feats, sp_size=25, sp_regul=0.2, gc_regul=1., gc_edge_type='model')
    yy, xx = np.mgrid[:512, :512]
    disc = (yy - 256) ** 2 + (xx - 256) ** 2 < 160 ** 2
    agree = max(np.mean(segm == disc), np.mean(segm == ~disc))
    assert agree > 0.98 and soft.shape == (512, 512, 2)
    slic, fts = pl.compute_color2d_superpixels_features(img, feats, sp_size=25, sp_regul=0.2)
    assert np.array_equal(slic, oracle.segment_slic_img2d(img, 25, 0.2))
    model = gc.estim_class_model(fts, 2)
    segm2, _ = pl.segment_color2d_slic_features_model_graphcut(img, model, feats, sp_size=25, sp_regul=0.2)
    segm_o, _, _, _ = oracle.segment_with_model(img, model.predict_proba, ('mean',), 25, 0.2, 1., 'model')
    assert np.array_equal(segm, segm2) and np.array_equal(segm2, segm_o)


def test_remaining_native_functions(oracle):
    """gray 3-D statistics, label histogram and ray features of imsegm/features_cython.pyx (:144-282): doctest goldens of
    imsegm/descriptors.py:470-478, :1479-1485, :1641-1653, the oracle, and stored outputs of the reference module compiled unchanged.
    Ray distances: 1e-5 relative against the compiled reference (it is built with -ffast-math, its last float ulp is
    compiler dependent); exact against the oracle and against the integer goldens."""
    from pyimsegm_b200 import descriptors as ds
    image = np.zeros((2, 3, 8))
    image[0, :, 2:6] = 1
    image[1, :, 3:7] = 3
    segm = np.array([[[0, 0, 0, 0, 1, 1, 1, 1]] * 3, [[2, 2, 2, 2, 3, 3, 3, 3]] * 3])
    np.testing.assert_allclose(ds.cython_img3d_gray_mean(image, segm), [0.5, 0.5, 0.75, 2.25], rtol=1e-12)
    rng = np.random.RandomState(0)
    vol = rng.random_sample((5, 40, 50)).astype(np.float32)
    seg = (np.arange(5)[:, None, None] * 20 + np.arange(40)[None, :, None] // 10 * 5 + np.arange(50)[None, None, :] // 10)
    for mode, fn in ((0, ds.cython_img3d_gray_mean), (1, ds.cython_img3d_gray_energy)):
        np.testing.assert_allclose(fn(vol, seg), oracle.gray3d_stat(vol, seg, mode), rtol=1e-6)
    np.testing.assert_allclose(ds.cython_img3d_gray_std(vol, seg), np.sqrt(oracle.gray3d_stat(vol, seg, 2, oracle.gray3d_stat(vol, seg, 0))), rtol=1e-6)
    s = np.array([[0, 1, 2], [1, 1, -1], [2, 2, 2]])
    assert ds.cython_label_hist_seg2d(s, np.ones((3, 3)), 3).tolist() == [1.0, 3.0, 4.0]
    big = rng.randint(-1, 6, (64, 80))
    mask = (rng.rand(64, 80) < 0.5).astype(int)
    assert ds.cython_label_hist_seg2d(big, mask, 6).tolist() == oracle.label_hist2d(big, mask, 6).astype(float).tolist()
    seg_empty = np.zeros((100, 150), dtype=bool)
    assert ds.cython_ray_features_seg2d(seg_empty, (50, 75), 90).tolist() == [-1., -1., -1., -1.]
    seg = np.ones((100, 150), dtype=bool)
    yy, xx = np.mgrid[:100, :150]
    seg[(yy - 50) ** 2 + (xx - 75) ** 2 < 40 ** 2] = False              # skimage.draw.disk((50, 75), 40)
    assert ds.cython_ray_features_seg2d(seg, (50, 75), 45).astype(int).tolist() == [40, 41, 40, 41, 40, 41, 40, 41]
    assert ds.cython_ray_features_seg2d(seg, (60, 40), 30).astype(int).tolist() == [74, 55, 28, 10, 5, 4, 4, 5, 9, 30, 57, 75]
    assert ds.cython_ray_features_seg2d(seg, (40, 60), 20).astype(int).tolist() == \
        [54, 57, 58, 55, 50, 43, 38, 31, 26, 24, 22, 22, 23, 26, 29, 34, 41, 48]
    noise = rng.rand(40, 60) < 0.08
    pos = np.stack([rng.randint(0, 40, 25), rng.randint(0, 60, 25)], 1)
    for edge, e in (('up', 1), ('down', -1)):
        got = ds.cython_ray_features_seg2d(noise, pos, 7.5, edge)
        for p, g, ref in zip(pos, got, REF_CYTHON['rays_' + edge]):
            assert np.array_equal(g, oracle.ray_features2d(noise, p, 7.5, e))
            np.testing.assert_allclose(g, ref, rtol=1e-5)


@pytest.mark.parametrize('sp_size,regul,shape', [(4, 0.3, (96, 128)), (5, 0.15, (77, 101)), (60, 0.2, (200, 260)), (9, 0.5, (33, 47))])
def test_slic_extreme_superpixel_sizes(oracle, sp_size, regul, shape):
    """tiny superpixels overflow the per-tile candidate list (resumable multi-round scan), huge ones span many tiles"""
    img, _ = synth_regions(shape[0], shape[1], seed=sp_size, cell=16)
    got, want = _slic_both(oracle, img, sp_size, regul)
    assert np.array_equal(got, want)


@pytest.mark.parametrize('min_f,max_f', [(0.05, 0.15), (0.3, 0.6), (1.5, 4.0)])
def test_connectivity_oversize_and_merge_replay(oracle, eng, min_f, max_f):
    """small max_size forces the truncated-BFS split of oversize components, large min_size forces long merge chains"""
    import torch
    from pyimsegm_b200.superpixels import slic_params
    img, _ = synth_regions(160, 208, seed=21, noise=0.12)
    n_seg, compact = slic_params(img.shape[:2], 14, 0.25)
    d_img = torch.from_numpy(img).cuda()
    labels, n_lab = eng.slic(d_img, n_seg, compact, sigma=1.0, min_size_factor=min_f, max_size_factor=max_f)
    got = labels.cpu().numpy()
    lo, hi = img.min(), img.max()
    want = oracle.slic((img - lo) / (hi - lo), n_seg, compact, sigma=1, min_size_factor=min_f, max_size_factor=max_f)
    assert np.array_equal(got, want) and int(n_lab.item()) == want.max() + 1


def test_degenerate_inputs_do_not_hang():
    from pyimsegm_b200 import pipelines as pl
    from pyimsegm_b200 import superpixels as sp
    tiny = np.random.RandomState(0).random_sample((9, 11, 3))
    seg = sp.segment_slic_img2d(tiny, 3, 0.3)
    assert seg.shape == (9, 11) and seg.min() == 0
    with pytest.raises(ValueError):
        sp.segment_slic_img2d(tiny, 50, 0.3)                    # superpixel larger than the image
    const = np.full((40, 50, 3), 0.5)
    seg = sp.segment_slic_img2d(const, 10, 0.2)                 # 0/0 in the min-max rescale: NaN colours, like the reference
    assert seg.shape == (40, 50)
    two = np.zeros((64, 64, 3)); two[:, 32:] = 1.0              # only two distinct values, flat regions tie everywhere
    segm, soft = pl.pipe_color2d_slic_features_model_graphcut(two, 2, {'color': ['mean']}, sp_size=8)
    assert len(np.unique(segm)) == 2 and (segm[:, :30] == segm[0, 0]).all() and (segm[:, 34:] == segm[0, -1]).all()


def test_region_label_histograms_reference_doctests():
    """imsegm/labeling.py:215-228 and :252-265"""
    from pyimsegm_b200 import labeling
    slic = np.array([[0] * 3 + [1] * 3 + [2] * 3] * 4 + [[4] * 3 + [5] * 3 + [6] * 3] * 4)
    segm = np.zeros(slic.shape, dtype=int)
    segm[4:, 5:] = 2
    want = [[12, 0, 0], [12, 0, 0], [12, 0, 0], [0, 0, 0], [12, 0, 0], [8, 0, 4], [0, 0, 12]]
    assert labeling.histogram_regions_labels_counts(slic, segm).tolist() == want
    norm = labeling.histogram_regions_labels_norm(slic, segm)
    np.testing.assert_allclose(norm[5], [2 / 3., 0, 1 / 3.])
    assert norm[3].tolist() == [0, 0, 0] and norm[6].tolist() == [0, 0, 1]
    rng = np.random.RandomState(0)
    a, b = rng.randint(0, 300, (257, 300)), rng.randint(0, 5, (257, 300))
    want = np.zeros((300, 5))
    np.add.at(want, (a.ravel(), b.ravel()), 1)
    assert np.array_equal(labeling.histogram_regions_labels_counts(a, b), want)
    with pytest.raises(ValueError):
        labeling.histogram_regions_labels_counts(a, b - 1)


def test_batch_api_equals_single_image_calls():
    """segment_images_batch (two streams, overlapped copies) returns exactly what the per-image calls return"""
    from pyimsegm_b200 import graph_cuts as gc
    from pyimsegm_b200 import pipelines as pl
    imgs = [synth_regions(160 + 16 * i, 200, seed=30 + i)[0] for i in range(5)]
    feats = {'color': ['mean', 'std']}
    batch = pl.segment_images_batch(imgs, nb_classes=3, dict_features=feats, sp_size=14)
    for im, (segm, soft) in zip(imgs, batch):
        s1, p1 = pl.pipe_color2d_slic_features_model_graphcut(im, 3, feats, sp_size=14)
        assert np.array_equal(segm, s1) and np.array_equal(soft, p1)
    _, fts = pl.compute_color2d_superpixels_features(imgs[0], feats, sp_size=14)
    model = gc.estim_class_model(fts, 3)
    batch = pl.segment_images_batch(imgs, dict_features=feats, sp_size=14, model_pipeline=model)
    for im, (segm, soft) in zip(imgs, batch):
        s1, p1 = pl.segment_color2d_slic_features_model_graphcut(im, model, feats, sp_size=14)
        assert np.array_equal(segm, s1) and np.allclose(soft, p1)
    with pytest.raises(ValueError):
        pl.segment_images_batch(imgs, nb_classes=3, model_pipeline=model)
