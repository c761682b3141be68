"""CPU tests: the oracle against every golden vector the reference's own doctests hold for the hot path
(SURVEY.md section 4), against stored outputs of the reference's Cython module, and against SciPy."""
import os

import numpy as np
from scipy import ndimage


def test_blur_is_bit_exact_with_scipy(oracle):
    rng = np.random.RandomState(0)
    for shape in ((37, 53, 3), (5, 7, 3), (64, 3, 3), (2, 2, 3)):
        img = rng.random_sample(shape)
        got = oracle.gaussian_blur(img, 1.0)
        want = ndimage.gaussian_filter(img[None], [1, 1, 1, 0])[0]  # skimage blurs the [1,H,W,3] array
        assert np.array_equal(got, want)


def test_rgb2lab_matches_numpy_formula(oracle):
    def rgb2lab_np(rgb):
        arr = rgb.copy()
        m = arr > 0.04045
        arr[m] = np.power((arr[m] + 0.055) / 1.055, 2.4)
        arr[~m] /= 12.92
        mat = np.array([[0.412453, 0.357580, 0.180423], [0.212671, 0.715160, 0.072169], [0.019334, 0.119193, 0.950227]])
        xyz = arr @ mat.T / np.array([0.95047, 1., 1.08883])
        m = xyz > 0.008856
        xyz[m] = np.cbrt(xyz[m])
        xyz[~m] = 7.787 * xyz[~m] + 16. / 116.
        x, y, z = xyz[..., 0], xyz[..., 1], xyz[..., 2]
        return np.stack([116 * y - 16, 500 * (x - y), 200 * (y - z)], -1)

    rng = np.random.RandomState(1)
    img = rng.random_sample((40, 50, 3))
    img[:5] *= 0.04  # exercise the linear branches
    np.testing.assert_allclose(oracle.rgb2lab_scaled(img, 1.0), rgb2lab_np(img), rtol=0, atol=1e-12)
    xs = np.linspace(0.0089, 1.2, 20001)
    c = np.array([oracle.lib().oracle_det_cbrt(x) for x in xs])
    assert np.max(np.abs(c / np.cbrt(xs) - 1)) < 4e-16
    xs = np.linspace(0.09, 1.0, 20001)
    c = np.array([oracle.lib().oracle_det_pow24(x) for x in xs])
    assert np.max(np.abs(c / xs ** 2.4 - 1)) < 2e-15


def test_slic_shape_contract_of_the_reference(oracle):
    """imsegm/superpixels.py:32-40 pins only shapes; also check label hygiene"""
    np.random.seed(0)
    img = np.random.random((100, 150, 3))
    assert oracle.segment_slic_img2d(img, 20, 0.2).shape == (100, 150)
    img = np.random.random((150, 100))
    assert oracle.segment_slic_img2d(img, 20, 0.2).shape == (150, 100)
    yy, xx = np.mgrid[:128, :128]
    img = np.full((128, 128, 3), 0.2)
    img[(yy - 64) ** 2 + (xx - 64) ** 2 < 900] = 0.8
    seg = oracle.segment_slic_img2d(img, 16, 0.3)
    assert set(np.unique(seg)) == set(range(seg.max() + 1))
    # every label is one 4-connected component
    for lb in range(seg.max() + 1):
        assert ndimage.label(seg == lb)[1] == 1


def test_enforce_connectivity_semantics(oracle):
    seg = np.zeros((6, 8), dtype=np.int64)
    seg[:, 4:] = 1
    seg[0, 0] = 1          # a 1-pixel island: no labelled neighbour yet -> merged into label 0
    seg[5, 7] = 0          # a late island: merged into the neighbour labelled last
    out = oracle.enforce_connectivity(seg, 3, 100)
    assert out[0, 0] == 0 and out[5, 7] == out[5, 6] and set(np.unique(out)) == {0, 1}
    # max_size truncation splits a big component in BFS order
    out = oracle.enforce_connectivity(np.zeros((4, 10), dtype=np.int64), 2, 16)
    assert out.tolist() == [[0, 0, 0, 0, 0, 0, 1, 1, 1, 1], [0, 0, 0, 0, 0, 1, 1, 1, 1, 1],
                            [0, 0, 0, 2, 1, 1, 1, 1, 1, 3], [0, 0, 2, 2, 2, 2, 1, 1, 3, 3]]  # diamond-shaped BFS cuts


def test_color_statistics_goldens(oracle):
    """imsegm/descriptors.py:218-226, :246-254, :275-283, :796-813"""
    image = np.zeros((2, 10, 3))
    image[:, 2:6, 0] = 1
    image[:, 3:7, 1] = 3
    image[:, 4:9, 2] = 2
    segm = np.array([[0] * 5 + [1] * 5] * 2)
    np.testing.assert_allclose(oracle.color2d_mean(image, segm), [[0.6, 1.2, 0.4], [0.2, 1.2, 1.6]], rtol=1e-12)
    np.testing.assert_allclose(oracle.color2d_energy(image, segm), [[0.6, 3.6, 0.8], [0.2, 3.6, 3.2]], rtol=1e-12)
    np.testing.assert_allclose(oracle.color2d_std(image, segm),
                               [[0.48989794, 1.46969383, 0.80000003], [0.40000001, 1.46969383, 0.80000001]], rtol=3e-8)
    fts = oracle.image2d_color_statistic(image, segm, ('mean', 'std', 'energy', 'meanGrad'))
    want = [[0.6, 1.2, 0.4, 0.5, 1.5, 0.8, 0.6, 3.6, 0.8, 0.2, 0.6, 0.4], [0.2, 1.2, 1.6, 0.4, 1.5, 0.8, 0.2, 3.6, 3.2, -0.2, -0.6, -0.6]]
    assert np.round(fts, 1).tolist() == want


def test_restatement_equals_reference_cython_module(oracle):
    """against the outputs of the reference's Cython module stored by tests/golden/make_cython_goldens.py"""
    gold = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden', 'reference_cython.npz'))
    rng = np.random.RandomState(3)
    img = rng.random_sample((60, 70, 3)).astype(np.float32)
    seg = (np.arange(60)[:, None] // 8 * 9 + np.arange(70)[None, :] // 8).astype(np.int32)
    mean_ref = gold['blocks_mean']
    np.testing.assert_allclose(oracle.color2d_mean(img, seg), mean_ref, rtol=1e-12)
    np.testing.assert_allclose(oracle.color2d_energy(img, seg), gold['blocks_energy'], rtol=1e-7)
    np.testing.assert_allclose(oracle.color2d_std(img, seg, mean_ref) ** 2, gold['blocks_variance'], rtol=1e-6)


def test_graph_goldens(oracle):
    """imsegm/superpixels.py:163-168, :211-215; imsegm/graph_cuts.py:311-319, :587-609"""
    grid = np.array([[0] * 5 + [1] * 5, [2] * 5 + [3] * 5])
    v, e = oracle.adjacency_edges(grid)
    assert v.tolist() == [0, 1, 2, 3] and e.tolist() == [[0, 1], [0, 2], [1, 3], [2, 3]]
    segm = np.array([[0] * 6 + [1] * 5, [0] * 6 + [2] * 5])
    assert oracle.superpixel_centers(segm).tolist() == [[0.5, 2.5], [0.0, 8.0], [1.0, 8.0]]
    segments = np.array([[0] * 3 + [1] * 2 + [2] * 5, [4] * 4 + [5] * 2 + [6] * 4])
    centres = oracle.superpixel_centers(segments)
    edges = np.array([[0, 1], [1, 2], [4, 5], [5, 6], [0, 4], [1, 5], [2, 6]])
    assert np.round(oracle.spatial_dist(centres, edges), 2).tolist() == [2.5, 3.5, 3.0, 3.0, 1.12, 1.41, 1.12]
    assert np.round(oracle.spatial_dist(centres, edges, True), 2).tolist() == [1.12, 1.57, 1.34, 1.34, 0.5, 0.63, 0.5]
    segments = np.array([[0] * 3 + [1] * 5 + [2] * 4, [4] * 4 + [5] * 5 + [6] * 3])
    np.random.seed(0)
    _ = np.random.random(segments.shape + (3,)) * 255
    features = np.random.random((segments.max() + 1, 15)) * 10
    proba = np.random.random((segments.max() + 1, 2))
    e, w = oracle.edge_weights(segments, edge_type='')
    assert e.tolist() == [[0, 1], [1, 2], [0, 4], [1, 4], [1, 5], [2, 5], [4, 5], [2, 6], [5, 6]]
    assert np.round(oracle.edge_weights(segments, edge_type='spatial')[1], 3).tolist() == \
        [0.776, 0.69, 2.776, 0.853, 2.194, 0.853, 0.69, 2.776, 0.776]
    assert np.round(oracle.edge_weights(segments, features=features, edge_type='features')[1], 3).tolist() == \
        [0.031, 0.005, 0.051, 0.032, 0.096, 0.013, 0.018, 0.033, 0.013]
    assert np.round(oracle.edge_weights(segments, proba=proba, edge_type='model')[1], 3).tolist() == \
        [0.001, 0.028, 1.122, 0.038, 0.117, 0.688, 0.487, 1.152, 0.282]
    # imsegm/graph_cuts.py:399-413 draws proba right after the image (no features in between)
    edges = np.array(e, dtype=int)
    np.random.seed(0)
    _ = np.random.random(segments.shape + (3,)) * 255
    proba = np.random.random((segments.max() + 1, 2))
    assert np.round(oracle.edge_model(edges, proba, 'l2'), 3).tolist() == [0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.002, 0.005, 0.0]
    assert np.round(oracle.edge_model(edges, proba, 'l1'), 3).tolist() == [0.002, 0.015, 0.001, 0.002, 0.0, 0.002, 0.015, 0.034, 0.001]
    assert np.round(oracle.edge_model(edges, proba, 'lT'), 3).tolist() == [0.0, 0.002, 0.0, 0.005, 0.0, 0.0, 0.101, 0.092, 0.001]


def test_graphcut_goldens(oracle):
    """imsegm/graph_cuts.py:687-716 (unary values, gc_regul=0 argmin, alpha-expansion on 10 nodes)"""
    np.random.seed(0)
    segments = np.array([[0] * 3 + [2] * 3 + [4] * 3 + [6] * 3 + [8] * 3, [1] * 3 + [3] * 3 + [5] * 3 + [7] * 3 + [9] * 3])
    proba = np.array([[0.1] * 6 + [0.9] * 4, [0.9] * 6 + [0.1] * 4], dtype=float).T
    proba += (0.5 - np.random.random(proba.shape)) * 0.2
    want = [[2.40531242, 0.15436155], [2.53266106, 0.11538463], [2.1604864, 0.13831863], [2.18495711, 0.19644636],
            [4.60517019, 0.0797884], [3.17833405, 0.11180231], [0.12059702, 4.20769207], [0.0143091, 1.70059894],
            [0.01005034, 3.39692559], [0.16916609, 3.64975219]]
    np.testing.assert_allclose(oracle.unary_cost(proba), want, rtol=1e-6, atol=1e-8)  # goldens are printed with 8 decimals
    assert oracle.segment_graph_cut_general(segments, proba, 0., '').tolist() == [1, 1, 1, 1, 1, 1, 0, 0, 0, 0]
    labels = oracle.segment_graph_cut_general(segments, proba, 1., 'spatial')
    assert labels.dtype == np.int32 and labels[segments].tolist() == [[1] * 9 + [0] * 6] * 2
    slic = np.array([[0] * 4 + [1] * 6 + [2] * 4, [3] * 5 + [4] * 4 + [5] * 5])
    proba = np.array([[1] * 3 + [0] * 3, [0] * 3 + [1] * 3], dtype=float).T
    proba += np.random.random(proba.shape) / 2.
    assert oracle.segment_graph_cut_general(slic, proba, 0., '').tolist() == [0, 0, 0, 1, 1, 1]


def test_alpha_expansion_is_a_local_minimum_and_matches_brute_force(oracle):
    rng = np.random.RandomState(5)
    for n, k in ((7, 2), (8, 3)):
        edges = np.array([[i, j] for i in range(n) for j in range(i + 1, n) if rng.rand() < 0.4], dtype=np.int32)
        w = rng.randint(1, 50, len(edges)).astype(np.int32)
        un = rng.randint(0, 100, (n, k)).astype(np.int32)
        pw = ((1 - np.eye(k)) * 10).astype(np.int32)
        labels, energy, _ = oracle.alpha_expansion_int(edges, w, un, pw, -1, return_energy=True)

        def E(l):
            return un[np.arange(n), l].sum() + (w * pw[l[edges[:, 0]], l[edges[:, 1]]]).sum()
        assert E(labels) == energy
        best = min(E(np.array(np.unravel_index(c, (k,) * n))) for c in range(k ** n))
        if k == 2:
            assert energy == best     # one expansion on a binary Potts problem is the global optimum
        else:
            assert energy <= 2 * best  # expansion's approximation bound for a metric


def test_label_histograms_reference_doctests(oracle):
    """imsegm/descriptors.py:1301-1325, :1406-1424, :1511-1516 -- the goldens of the label-histogram drivers"""
    segm = np.zeros((10, 10), dtype=int)
    segm[1:9, 2:8] = 1
    segm[3:7, 4:6] = 2
    points = [[3, 3], [4, 4], [2, 7], [6, 6]]
    want = np.array([[0., 0.8, 0.2, 0.12, 0.62, 0.25, 0.44, 0.41, 0.15], [0., 0.2, 0.8, 0., 0.62, 0.38, 0.22, 0.75, 0.03],
                     [0.2, 0.8, 0., 0.5, 0.5, 0., 0.46, 0.33, 0.21], [0., 0.8, 0.2, 0.12, 0.62, 0.25, 0.44, 0.41, 0.15]])
    assert np.array_equal(np.round(oracle.label_histograms_positions(segm, points, [1, 2, 4]), 2), want)
    proba = np.zeros((10, 10, 2), dtype=int)
    proba[3:7, 4:6, 1] = 1
    proba[:, :, 0] = 1 - proba[:, :, 0]
    want = np.array([[1., 0.2, 1., 0.25, 1., 0.15], [1., 0.8, 1., 0.38, 1., 0.03], [1., 0., 1., 0., 1., 0.21], [1., 0.2, 1., 0.25, 1., 0.15]])
    assert np.array_equal(np.round(oracle.label_histograms_positions(proba, points, [1, 2, 4]), 2), want)
    hist, size = oracle.label_hist_selem(segm, [6, 6], np.ones((3, 3)), 3)
    assert hist.tolist() == [0., 7., 2.] and size == 9
    hist, size = oracle.label_hist_selem(segm, [4, 4], np.ones((5, 5)), 3)
    assert hist.tolist() == [0., 17., 8.] and size == 25
    seg = np.zeros((50, 50, 2), dtype=float)
    seg[15:35, 20:40, 1] = 1
    seg[:, :, 0] = 1 - seg[:, :, 1]
    hist, size = oracle.label_hist_selem(seg, (15, 20), np.ones((12, 13), dtype=int))
    assert hist.tolist() == [114., 42.] and size == 156


def test_host_side_descriptor_helpers_reference_doctests():
    """pure-host helpers of the Ray / histogram drivers against the reference's doctest values
    (imsegm/descriptors.py:1380-1387, :1773-1786, :1905-1920, :1975-1983, :2013-2025)"""
    from pyimsegm_b200 import descriptors as ds
    assert ds.adjust_bounding_box_crop((50, 50), (7, 7), (20, 20)) == ((17, 17), (24, 24), (0, 0), (7, 7))
    assert ds.adjust_bounding_box_crop((50, 50), (15, 15), (20, 45)) == ((13, 38), (28, 50), (0, 0), (15, 12))
    assert ds.adjust_bounding_box_crop((50, 50), (15, 15), (5, 5)) == ((0, 0), (13, 13), (2, 2), (15, 15))
    assert ds.adjust_bounding_box_crop((50, 50), (80, 80), (20, 20)) == ((0, 0), (50, 50), (20, 20), (70, 70))
    vec = np.array([43, 46, 44, 39, 28, 18, 12, 10, 9, 12, 22, 28])
    ray, shift = ds.shift_ray_features(vec)
    assert abs(shift - 41.50) < 0.01 and ray.tolist() == [46, 44, 39, 28, 18, 12, 10, 9, 12, 22, 28, 43]
    ray2, shift2 = ds.shift_ray_features(ray)
    assert abs(shift2 - 11.50) < 0.01 and np.array_equal(ray, ray2)
    assert ds.shift_ray_features(vec, method='max')[1] == 30.0
    assert ds.interpolate_ray_dist([-1] * 5).tolist() == [-1] * 5
    vals = np.sin(np.linspace(0, 2 * np.pi, 20)) * 10
    vals[3:7] = -1
    vals[16:] = -1
    assert np.round(ds.interpolate_ray_dist(vals, order='spline')).astype(int).tolist() == \
        [0, 3, 6, 8, 9, 10, 9, 7, 5, 2, -2, -5, -7, -9, -10, -10, -9, -7, -5, -3]
    assert np.round(ds.interpolate_ray_dist(vals, order='cos')).astype(int).tolist() == \
        [0, 3, 6, 8, 10, 10, 9, 7, 5, 2, -2, -5, -7, -9, -10, -10, -8, -6, -3, 0]
    np.testing.assert_allclose(ds.reconstruct_ray_features_2d((10., 10), np.array([1] * 4)), [[10, 11], [11, 10], [10, 9], [9, 10]], atol=1e-12)
    np.testing.assert_allclose(ds.reconstruct_ray_features_2d((10., 10), np.array([-1, 0, 1, np.inf])), [[10, 10], [10, 9]], atol=1e-12)
    assert ds.reduce_close_points(np.array([range(10), range(10)]).T, 2).tolist() == [[0, 0], [2, 2], [4, 4], [6, 6], [8, 8]]
    assert ds.reduce_close_points(np.array([[0, 0], [1, 1], [0, 2]]), 2).tolist() == [[0, 0], [0, 2]]
    assert ds.reduce_close_points(np.ones((10, 2)), 2).tolist() == [[1., 1.]]
    # the NumPy variants of the gray-volume statistics (descriptors.py:545-676) on the doctest volume of :698-715
    img = np.array([[[0] * 3 + [1] * 3 + [2] * 2] * 3] * 2, dtype=float)[:, :, :8]
    seg = np.array([[[0] * 2 + [1] * 2 + [2] * 2 + [5] * 2] * 3] * 2)
    assert ds.numpy_img3d_gray_mean(img, seg).shape == (6, )
    np.testing.assert_allclose(ds.numpy_img3d_gray_mean(img, seg)[[0, 1, 2, 5]], [0., 0.5, 1., 2.])
    np.testing.assert_allclose(ds.numpy_img3d_gray_std(img, seg)[[0, 1, 2, 5]], [0., 0.5, 0., 0.])
    np.testing.assert_allclose(ds.numpy_img3d_gray_energy(img, seg)[[0, 1, 2, 5]], [0., 0.5, 1., 4.])


def test_color_median_reference_doctest(oracle):
    """imsegm/descriptors.py:429-437 numpy_img2d_color_median"""
    image = np.zeros((2, 10, 3))
    image[:, 2:6, 0] = 1
    image[:, 3:8, 1] = 3
    image[:, 4:9, 2] = 2
    segm = np.array([[0, 0, 0, 0, 1, 1, 1, 1, 1, 1]] * 2)
    np.testing.assert_allclose(oracle.color2d_median(image, segm), [[0.5, 0., 0.], [0., 3., 2.]])
