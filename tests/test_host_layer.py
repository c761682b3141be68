"""The host layer over the C-ABI: only engine.py (and the binding table in _lib.py) calls the library, the small rules every
caller shares, and the recovery from an overflowed device edge table."""
import ast
import glob
import os

import numpy as np
import pytest

from conftest import ROOT, synth_regions

PKG = os.path.join(ROOT, 'pyimsegm_b200')


def test_only_the_engine_calls_the_library():
    offenders = []
    for path in sorted(glob.glob(os.path.join(PKG, '*.py'))):
        if os.path.basename(path) in ('engine.py', '_lib.py'):
            continue
        with open(path) as f:
            tree = ast.parse(f.read(), path)
        for node in ast.walk(tree):
            if isinstance(node, ast.Attribute) and node.attr.startswith('isb_'):
                offenders.append('%s:%d .%s' % (os.path.basename(path), node.lineno, node.attr))
            elif isinstance(node, ast.Import) and any(a.name.split('.')[0] == 'ctypes' for a in node.names):
                offenders.append('%s:%d import ctypes' % (os.path.basename(path), node.lineno))
            elif isinstance(node, ast.ImportFrom) and (node.module or '').split('.')[0] == 'ctypes':
                offenders.append('%s:%d from ctypes' % (os.path.basename(path), node.lineno))
    assert not offenders, offenders


def test_flag_bits():
    from pyimsegm_b200.engine import flag_bits
    assert flag_bits(()) == (0, 0)
    assert flag_bits(['mean']) == (1, 1)
    assert flag_bits(('energy', 'mean')) == (5, 2)
    assert flag_bits(['mean', 'std', 'energy']) == (7, 3)
    assert flag_bits(['std', 'std']) == (2, 1)
    with pytest.raises(KeyError):
        flag_bits(['median'])


def test_dtype_code():
    import torch
    from pyimsegm_b200.engine import dtype_code
    for code, np_t, torch_t in ((0, np.uint8, torch.uint8), (1, np.uint16, torch.uint16), (2, np.float32, torch.float32),
                                (3, np.float64, torch.float64)):
        assert dtype_code(np.dtype(np_t)) == code
        assert dtype_code(np_t) == code
        assert dtype_code(torch_t) == code
    with pytest.raises(KeyError):
        dtype_code(np.int32)


def test_edge_capacity_rule(monkeypatch):
    from pyimsegm_b200 import engine
    assert engine.edge_capacity(1) == 64
    assert engine.edge_capacity(1000) == 8000
    assert engine.edge_capacity(1000, ndim=3) == 16000
    assert engine.grown_edge_capacity(8000) == 32000
    monkeypatch.setattr(engine, 'EDGE_CAP_PER_NODE', 1)
    assert engine.edge_capacity(1000) == 1000
    assert engine.edge_capacity(10) == 64


# ---------------------------------------------------------------------------------------------------------------------------
# the overflow recovery: with one edge per node the first table of every graph below overflows; the kernels bound their writes
# at the capacity, every consumer skips an overflowed table and the host redoes the graph larger.  The images hold multiples of
# 1/64, so the colour means the device GMM is fitted on are exact whatever order the floating-point atomics add in: two runs
# then fit the same model and must give the same label map.

def _image(h, w, seed):
    return np.round(synth_regions(h, w, seed=seed)[0] * 64) / 64


def _small_cap(monkeypatch):
    from pyimsegm_b200 import engine
    monkeypatch.setattr(engine, 'EDGE_CAP_PER_NODE', 1)


def _same(got, want):
    assert np.array_equal(got[0], want[0])
    np.testing.assert_allclose(got[1], want[1], rtol=1e-6, atol=1e-9)   # the statistics use floating-point atomics


@pytest.mark.gpu
@pytest.mark.parametrize('graphs', [True, False])
def test_overflow_single_image(monkeypatch, graphs):
    from pyimsegm_b200 import pipelines as pl
    img = _image(256, 320, 51)
    feats = {'color': ['mean']}
    monkeypatch.setattr(pl, 'USE_CUDA_GRAPHS', graphs)
    want = pl.pipe_color2d_slic_features_model_graphcut(img, 3, feats, sp_size=12, sp_regul=0.2)
    _small_cap(monkeypatch)
    for _ in range(3):          # eager, captured, replayed when the graphs are on
        _same(pl.pipe_color2d_slic_features_model_graphcut(img, 3, feats, sp_size=12, sp_regul=0.2), want)


@pytest.mark.gpu
def test_overflow_batch(monkeypatch):
    from pyimsegm_b200 import pipelines as pl
    imgs = [_image(200, 264, s) for s in (52, 53, 54, 55)]
    feats = {'color': ['mean']}
    want = pl.segment_images_batch(imgs, 3, feats, sp_size=12, sp_regul=0.2)
    _small_cap(monkeypatch)
    for got, ref in zip(pl.segment_images_batch(imgs, 3, feats, sp_size=12, sp_regul=0.2), want):
        _same(got, ref)


@pytest.mark.gpu
def test_overflow_banded(monkeypatch):
    from pyimsegm_b200 import tiled
    img = _image(320, 256, 56)
    want = tiled.pipe_color2d_slic_features_model_graphcut_tiled(img, 3, sp_size=12, bands_per_rank=2)
    _small_cap(monkeypatch)
    got = tiled.pipe_color2d_slic_features_model_graphcut_tiled(img, 3, sp_size=12, bands_per_rank=2)
    assert got[2] == want[2]
    _same(got[:2], want[:2])


@pytest.mark.gpu
def test_overflow_region_adjacency_graph(monkeypatch):
    from pyimsegm_b200.superpixels import make_graph_segm_connect_grid2d_conn4, segment_slic_img2d
    slic = segment_slic_img2d(synth_regions(256, 256, seed=57)[0], sp_size=10, relative_compact=0.2)
    want = make_graph_segm_connect_grid2d_conn4(slic)
    _small_cap(monkeypatch)
    got = make_graph_segm_connect_grid2d_conn4(slic)
    assert np.array_equal(got[0], want[0]) and got[1] == want[1]


@pytest.mark.gpu
def test_overflow_volume_edge_weights(monkeypatch):
    from pyimsegm_b200.graph_cuts import compute_edge_weights
    rng = np.random.RandomState(58)
    seg = np.kron(np.arange(6 * 8 * 8).reshape(6, 8, 8), np.ones((3, 4, 4), dtype=int))      # 384 boxes, 6-connected
    proba = rng.dirichlet(np.ones(3), seg.max() + 1)
    want = compute_edge_weights(seg, proba=proba, edge_type='model')
    _small_cap(monkeypatch)
    got = compute_edge_weights(seg, proba=proba, edge_type='model')
    assert np.array_equal(got[0], want[0])
    np.testing.assert_array_equal(got[1], want[1])
