"""
Parity against outputs OF THE REFERENCE ITSELF: tests/golden/reference_vectors.npz was produced by tests/golden/make_goldens.py,
which imports the reference's own modules (imsegm.descriptors / graph_cuts / labeling / superpixels from /root/reference, with its
Cython module compiled unchanged) and stores inputs and outputs.  The not-gpu half pins the oracle, the gpu half the CUDA path.
"""
import os

import numpy as np
import pytest

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden', 'reference_vectors.npz')


@pytest.fixture(scope='module')
def ref():
    return np.load(GOLD)


def _lm_check(fts, want, tol):
    """errors against the response scale of the battery / channel (see tests/test_gpu_texture.py)"""
    worst = 0.0
    for b in range(fts.shape[1] // 9):
        for c in range(3):
            col = lambda i: b * 9 + i * 3 + c        # noqa: E731
            rms = np.sqrt(np.abs(want[:, col(2)]).max()) + 1e-300
            for i in range(3):
                worst = max(worst, np.abs(fts[:, col(i)] - want[:, col(i)]).max() / (rms * rms if i == 2 else rms))
    assert worst < tol, 'max error relative to the battery response scale: %g' % worst


# ------------------------------------------------------------------------------------------------------------------- oracle

def test_oracle_matches_the_reference_outputs(oracle, ref):
    from oracle import texture as otex
    img, seg = ref['color_img'], ref['color_seg']
    np.testing.assert_allclose(oracle.color2d_mean(img, seg), ref['color_mean'], rtol=1e-6, atol=1e-9)
    np.testing.assert_allclose(oracle.color2d_energy(img, seg), ref['color_energy'], rtol=1e-6, atol=1e-9)
    np.testing.assert_allclose(oracle.color2d_std(img, seg), ref['color_std'], rtol=1e-6, atol=1e-9)
    native = [list(ref['color_statistic_names']).index('color-ch%i_%s' % (c, f)) for f in ('mean', 'std', 'energy', 'meanGrad') for c in (1, 2, 3)]
    np.testing.assert_allclose(oracle.image2d_color_statistic(img, seg, ('mean', 'std', 'energy', 'meanGrad')), ref['color_statistic'][:, native],
                               rtol=1e-6, atol=1e-9)
    vol, vseg = ref['gray_vol'], ref['gray_seg']
    np.testing.assert_allclose(oracle.gray3d_stat(vol, vseg, 0), ref['gray_mean'], rtol=1e-6, atol=1e-9)
    np.testing.assert_allclose(oracle.gray3d_stat(vol, vseg, 1), ref['gray_energy'], rtol=1e-6, atol=1e-9)
    # Leung-Malik: the scipy restatement in oracle/texture.py against the reference's own descriptor (pins the texture oracle)
    bank, names = otex.filter_bank(sigmas=otex.SIGMAS_SHORT, nb_orient=4)
    np.testing.assert_allclose(np.concatenate(bank, axis=0), ref['lm_short_bank'], rtol=1e-12, atol=1e-15)
    assert list(names) == list(ref['lm_short_names'])
    want = ref['lm_short_features']
    fts, fnames = otex.texture_desc_lm(ref['lm_img'], ref['lm_seg'], ('mean', 'std', 'energy'), 'short')
    assert list(fnames) == list(ref['lm_short_feature_names']) and fts.shape == want.shape
    _lm_check(fts, want, 2e-6)          # both are float64 scipy; the statistics go through f32 in the Cython module
    # native hist / Ray kernels, energies, graph
    np.testing.assert_array_equal(oracle.label_hist2d(ref['hist_seg'], ref['hist_selem'], 4), ref['hist'])
    for k, p in enumerate(ref['ray_pos']):
        np.testing.assert_allclose(oracle.ray_features2d(ref['ray_seg'], tuple(p), 15., 1), ref['ray_up'][k], rtol=1e-5)
        np.testing.assert_allclose(oracle.ray_features2d(1 - ref['ray_seg'], tuple(p), 15., -1), ref['ray_down'][k], rtol=1e-5)
    proba, edges, centres = ref['gc_proba'], ref['gc_edges'], ref['gc_centres']
    np.testing.assert_allclose(oracle.unary_cost(proba), ref['gc_unary'], rtol=1e-12)
    np.testing.assert_allclose(oracle.pairwise_cost(2.5, 3), ref['gc_pairwise_potts'], rtol=1e-12)
    for metric in ('lT', 'l1', 'l2'):
        np.testing.assert_allclose(oracle.edge_model(edges, proba, metric), ref['gc_edge_model_' + metric], rtol=1e-10)
    np.testing.assert_allclose(oracle.spatial_dist(centres, edges), ref['gc_spatial'], rtol=1e-12)
    np.testing.assert_allclose(oracle.spatial_dist(centres, edges, relative=True), ref['gc_spatial_rel'], rtol=1e-12)
    assert oracle.adjacency_edges(seg)[1].tolist() == ref["graph_edges"].tolist()    # same order too: sorted by (b, a)


# ---------------------------------------------------------------------------------------------------------------- CUDA path

@pytest.mark.gpu
def test_device_matches_the_reference_outputs(ref):
    from pyimsegm_b200 import descriptors as ds
    from pyimsegm_b200 import graph_cuts as gc
    from pyimsegm_b200 import labeling as lb
    from pyimsegm_b200 import superpixels as sp
    img, seg = ref['color_img'], ref['color_seg']
    np.testing.assert_allclose(ds.cython_img2d_color_mean(img, seg), ref['color_mean'], rtol=1e-6, atol=1e-9)
    np.testing.assert_allclose(ds.cython_img2d_color_energy(img, seg), ref['color_energy'], rtol=1e-6, atol=1e-9)
    np.testing.assert_allclose(ds.cython_img2d_color_std(img, seg), ref['color_std'], rtol=1e-6, atol=1e-9)
    fts, names = ds.compute_image2d_color_statistic(img, seg, ('mean', 'std', 'energy', 'median', 'meanGrad'))
    assert list(names) == list(ref['color_statistic_names'])
    np.testing.assert_allclose(fts, ref['color_statistic'], rtol=1e-6, atol=1e-9)
    vol, vseg = ref['gray_vol'], ref['gray_seg']
    np.testing.assert_allclose(ds.cython_img3d_gray_mean(vol, vseg), ref['gray_mean'], rtol=1e-6, atol=1e-9)
    np.testing.assert_allclose(ds.cython_img3d_gray_energy(vol, vseg), ref['gray_energy'], rtol=1e-6, atol=1e-9)
    np.testing.assert_allclose(ds.cython_img3d_gray_std(vol, vseg), ref['gray_std'], rtol=1e-6, atol=1e-9)
    fts, names = ds.compute_image3d_gray_statistic(vol, vseg)
    assert list(names) == list(ref['gray_statistic_names'])
    np.testing.assert_allclose(fts, ref['gray_statistic'], rtol=1e-6, atol=1e-9)
    # Leung-Malik on the tensor cores against the reference's own descriptor
    bank, names = ds.create_filter_bank_lm_2d(sigmas=ds.SHORT_FILTERS_SIGMAS, nb_orient=4)
    np.testing.assert_allclose(np.concatenate(bank, axis=0), ref['lm_short_bank'], rtol=1e-12, atol=1e-15)
    fts, fnames = ds.compute_texture_desc_lm_img2d_clr(ref['lm_img'], ref['lm_seg'], ('mean', 'std', 'energy'), 'short')
    assert list(fnames) == list(ref['lm_short_feature_names'])
    _lm_check(fts, ref['lm_short_features'], 2e-4)
    np.testing.assert_allclose(ds.compute_img_filter_response2d(ref['lm_img'][..., 0], bank[0]), ref['lm_response_edge0'], rtol=1e-10, atol=1e-13)
    # native hist / Ray kernels
    np.testing.assert_array_equal(ds.cython_label_hist_seg2d(ref['hist_seg'].astype(float), ref['hist_selem'], 4), ref['hist'])
    np.testing.assert_allclose(ds.cython_ray_features_seg2d(ref['ray_seg'], ref['ray_pos'], 15., 'up'), ref['ray_up'], rtol=1e-5)
    np.testing.assert_allclose(ds.cython_ray_features_seg2d(1 - ref['ray_seg'], ref['ray_pos'], 15., 'down'), ref['ray_down'], rtol=1e-5)
    # energies: host functions of the drop-in module and the device kernel behind compute_edge_weights
    proba, edges, centres = ref['gc_proba'], ref['gc_edges'], ref['gc_centres']
    np.testing.assert_allclose(gc.compute_unary_cost(proba), ref['gc_unary'], rtol=1e-12)
    np.testing.assert_allclose(gc.compute_pairwise_cost(2.5, proba.shape), ref['gc_pairwise_potts'], rtol=1e-12)
    np.testing.assert_allclose(gc.compute_pairwise_cost([((0, 1), 2.0), ((1, 2), 0.5)], proba.shape), ref['gc_pairwise_list'], rtol=1e-12)
    for metric in ('lT', 'l1', 'l2'):
        np.testing.assert_allclose(gc.compute_edge_model(edges, proba, metric), ref['gc_edge_model_' + metric], rtol=1e-10)
    np.testing.assert_allclose(gc.compute_spatial_dist(centres, edges, relative=True), ref['gc_spatial_rel'], rtol=1e-12)
    # graph and region / annotation histogram
    assert sorted(map(tuple, np.asarray(sp.make_graph_segm_connect_grid2d_conn4(seg)[1]).tolist())) == sorted(map(tuple, ref['graph_edges'].tolist()))
    np.testing.assert_allclose(lb.histogram_regions_labels_norm(seg, ref['annot']), ref['region_hist_norm'], rtol=1e-12)


def test_volume_connectivity_oracle_reduces_to_the_2d_one(oracle):
    """oracle_enforce_connectivity3d on a one-slice volume is the 2-D pass (its z neighbours never exist)"""
    import ctypes as C
    rng = np.random.RandomState(11)
    seg = rng.randint(0, 6, (40, 52)).astype(np.int64)
    seg[10:30, 5:25] = 7
    for min_size, max_size in ((2, 30), (6, 400), (1, 3)):
        want = oracle.enforce_connectivity(seg, min_size, max_size)
        got = np.empty_like(seg)
        oracle.lib().oracle_enforce_connectivity3d(seg.ctypes.data_as(C.POINTER(C.c_int64)), 1, 40, 52, C.c_long(min_size), C.c_long(max_size),
                                                   got.ctypes.data_as(C.POINTER(C.c_int64)))
        assert np.array_equal(got, want), (min_size, max_size)
