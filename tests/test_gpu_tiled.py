"""
Row-band mode (pyimsegm_b200/tiled.py, SURVEY.md section 8e / BASELINE config 5) against the oracle and against the
single-GPU path.  On one GPU the bands live side by side in one process and are merged by isb_combine -- the same integer
sum the NCCL all_reduce does between GPUs; the real 2-GPU run is tests/run_tiled_ranks.py under torchrun (spawned by
test_two_ranks_nccl when the box has two GPUs).
"""
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT, synth_disc, synth_regions

pytestmark = pytest.mark.gpu


@pytest.fixture(scope='module')
def eng():
    from pyimsegm_b200.engine import get_engine
    return get_engine()


@pytest.mark.parametrize('case', ['regions', 'ragged', 'u8', 'gray', 'slico', 'tiny_sp', 'thin_bands'])
def test_banded_label_map_is_bit_exact(oracle, eng, case):
    from pyimsegm_b200.superpixels import slic_params
    from pyimsegm_b200.tiled import slic_tiled
    slico, bands_list = False, (2, 3, 5)
    if case == 'regions':
        img, sp_size, regul = synth_regions(512, 384, seed=11)[0], 20, 0.2
    elif case == 'ragged':
        img, sp_size, regul = synth_regions(397, 263, seed=12)[0], 17, 0.25      # H not a multiple of the band count
    elif case == 'u8':
        img, sp_size, regul = (synth_disc(320, 256) * 255).astype(np.uint8), 25, 0.3
    elif case == 'gray':
        img, sp_size, regul = synth_disc(300, 200)[..., 0], 20, 0.2
    elif case == 'slico':
        img, sp_size, regul, slico = synth_regions(360, 300, seed=13)[0], 15, 0.2, True
    elif case == 'tiny_sp':
        img, sp_size, regul = synth_regions(256, 256, seed=14, cell=16)[0], 5, 0.3
    else:
        img, sp_size, regul, bands_list = synth_regions(300, 256, seed=15)[0], 30, 0.2, (7, 12)   # bands thinner than the halo
    want = oracle.segment_slic_img2d(img, sp_size, regul, slico)
    n_seg, compact = slic_params(img.shape[:2], sp_size, regul)
    for n_bands in bands_list:
        res = slic_tiled(img, n_seg, compact, slic_zero=slico, bands_per_rank=n_bands, eng=eng)
        assert not res.fell_back
        got = eng.to_host(res.d_seg)
        assert np.array_equal(got, want), 'bands=%d' % n_bands
        assert int(eng.to_host(res.d_n_labels)[0]) == want.max() + 1


def test_banded_sweeps_without_connectivity_match_whole_image(eng):
    """the raw k-means label map (before the connectivity pass), band by band, against the single-GPU sweeps"""
    from pyimsegm_b200.superpixels import slic_params
    from pyimsegm_b200.tiled import slic_tiled
    img = synth_regions(640, 448, seed=16, noise=0.1)[0]
    n_seg, compact = slic_params(img.shape[:2], 22, 0.15)
    whole, _ = eng.slic(eng.to_device(img, 'image'), n_seg, compact, enforce_connectivity=False)
    whole = eng.to_host(whole).copy()
    for n_bands in (2, 4):
        res = slic_tiled(img, n_seg, compact, bands_per_rank=n_bands, eng=eng, enforce_connectivity=False)
        assert np.array_equal(eng.to_host(res.d_seg), whole)


def test_orphans_beyond_the_halo_fall_back(oracle, eng):
    """a constant image rescales to NaN: no window ever takes a pixel, every pixel keeps label 0 -- an orphan far from
    cluster 0's centre.  The device check must notice and the whole-image sweeps must give the oracle's answer."""
    from pyimsegm_b200.superpixels import slic_params
    from pyimsegm_b200.tiled import slic_tiled
    img = np.full((240, 200, 3), 0.5)
    want = oracle.segment_slic_img2d(img, 20, 0.2)
    n_seg, compact = slic_params(img.shape[:2], 20, 0.2)
    res = slic_tiled(img, n_seg, compact, bands_per_rank=3, eng=eng)
    assert res.fell_back
    assert np.array_equal(eng.to_host(res.d_seg), want)


@pytest.mark.parametrize('features', [['mean'], ['mean', 'std', 'energy']])
def test_banded_pipeline_matches_single_gpu_pipeline(eng, features):
    from pyimsegm_b200 import pipelines as pl
    from pyimsegm_b200.tiled import pipe_color2d_slic_features_model_graphcut_tiled
    img, truth = synth_regions(600, 512, seed=17)
    fts = {'color': features}
    segm, soft = pl.pipe_color2d_slic_features_model_graphcut(img, 3, fts, sp_size=20, sp_regul=0.2, gc_regul=1., gc_edge_type='model')
    for n_bands in (1, 3):
        got, got_soft, (lo, hi) = pipe_color2d_slic_features_model_graphcut_tiled(img, 3, fts, sp_size=20, sp_regul=0.2,
                                                                                 bands_per_rank=n_bands)
        assert (lo, hi) == (0, 600)
        assert np.array_equal(got, segm)
        np.testing.assert_allclose(got_soft, soft, rtol=1e-6, atol=1e-9)
    # and the segmentation means something: classes follow the ground-truth regions up to a permutation
    agree = max(np.mean(np.asarray(p)[truth] == segm) for p in ([0, 1, 2], [0, 2, 1], [1, 0, 2], [1, 2, 0], [2, 0, 1], [2, 1, 0]))
    assert agree > 0.9


def test_banded_colour_statistics_match_oracle(oracle, eng):
    from pyimsegm_b200.superpixels import slic_params
    from pyimsegm_b200.tiled import color_stats_tiled, slic_tiled
    img = synth_regions(420, 333, seed=18)[0].astype(np.float32)
    n_seg, compact = slic_params(img.shape[:2], 18, 0.2)
    res = slic_tiled(img, n_seg, compact, bands_per_rank=4, eng=eng)
    seg = eng.to_host(res.d_seg).copy()
    feat, centres = color_stats_tiled(res, img.dtype, 3, ('mean', 'std', 'energy'), eng=eng)
    nb = seg.max() + 1
    want = np.hstack([oracle.color2d_mean(img, seg), oracle.color2d_std(img, seg), oracle.color2d_energy(img, seg)])
    np.testing.assert_allclose(eng.to_host(feat)[:nb], want, rtol=1e-6, atol=1e-9)
    np.testing.assert_allclose(eng.to_host(centres)[:nb], np.asarray(oracle.superpixel_centers(seg)), rtol=1e-12)


@pytest.mark.parametrize('bank', ['normal', 'short'])
def test_banded_texture_statistics_match_whole_image(eng, bank):
    """Leung-Malik statistics of a banded image: bands whose slabs end INSIDE the image (rows + 616 of halo) must reproduce the
    whole-image descriptor -- same background, same responses on the owned rows, same image-wide response norms"""
    from pyimsegm_b200.superpixels import slic_params
    from pyimsegm_b200.texture import device_lm_features
    from pyimsegm_b200.tiled import LM_ROW_MARGIN, slic_tiled, texture_stats_tiled
    rng = np.random.RandomState(5)
    img = synth_regions(2000, 192, seed=21)[0] + 0.05 * rng.standard_normal((2000, 192, 3))
    n_seg, compact = slic_params(img.shape[:2], 24, 0.2)
    flags = ('mean', 'std', 'energy')
    res = slic_tiled(img, n_seg, compact, bands_per_rank=3, eng=eng, raw_margin=LM_ROW_MARGIN)
    assert res.bands[1].up_lo > 0 and res.bands[1].up_hi < 2000          # the middle band's slab has two interior edges
    got = eng.to_host(texture_stats_tiled(res, img.dtype, flags, bank, eng=eng)).copy()
    d_img = eng.to_device(img, 'image')
    want = eng.to_host(device_lm_features(eng, d_img, res.d_seg, int(res.nb_bound), flags, bank)[0]).copy()
    assert np.abs(want).max() > 0.1
    np.testing.assert_allclose(got, want, rtol=1e-7, atol=1e-9)


def test_banded_pipeline_with_texture_matches_single_gpu_pipeline(eng):
    from pyimsegm_b200 import pipelines as pl
    from pyimsegm_b200.tiled import pipe_color2d_slic_features_model_graphcut_tiled
    rng = np.random.RandomState(6)
    img = synth_regions(1500, 160, seed=22)[0] + 0.05 * rng.standard_normal((1500, 160, 3))
    fts = {'color': ['mean', 'std'], 'tLM_short': ['mean', 'energy']}
    segm, soft = pl.pipe_color2d_slic_features_model_graphcut(img, 3, fts, sp_size=20, sp_regul=0.2, gc_regul=1., gc_edge_type='model')
    got, got_soft, (lo, hi) = pipe_color2d_slic_features_model_graphcut_tiled(img, 3, fts, sp_size=20, sp_regul=0.2, bands_per_rank=2)
    assert (lo, hi) == (0, 1500)
    assert np.mean(got == segm) > 0.999
    np.testing.assert_allclose(got_soft, soft, rtol=1e-4, atol=1e-6)


def test_two_ranks_nccl():
    """the same checks with two processes, one GPU each, merged by NCCL all_reduce / broadcast"""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip('needs two GPUs')
    cmd = [sys.executable, '-m', 'torch.distributed.run', '--nnodes=1', '--nproc-per-node=2', '--master-addr', '127.0.0.1',
           '--master-port', '29571', os.path.join(ROOT, 'tests', 'run_tiled_ranks.py')]
    out = subprocess.run(cmd, cwd=ROOT, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, timeout=600)
    text = out.stdout.decode(errors='replace')
    assert out.returncode == 0, text[-3000:]
    assert 'TILED-RANKS-OK' in text, text[-3000:]
