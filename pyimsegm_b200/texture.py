"""
Leung-Malik texture descriptors on the GPU (reference ``imsegm/descriptors.py:880-1106``).

Host side: the filter bank is built with numpy/scipy exactly like the reference does at run time
(``create_filter_bank_lm_2d``, descriptors.py:903-948), then laid out for the tensor-core contraction of
``isb_lm_texture`` (correlation form, oriented batteries first, tf32 hi/lo split, operand layout).  The contraction, the battery max,
the log-norm scaling and the per-superpixel statistics run in CUDA (``csrc/lm_texture.cu``).
"""
import itertools

import numpy as np

from .engine import dtype_code, flag_bits, get_engine

#: sigma of the background that is subtracted before filtering (descriptors.py:1078)
BACKGROUND_SIGMA = 150
_KW, _KWP = 33, 40
_BANK_CACHE = {}


def make_gaussian_filter1d(vals, sigma, order=0):
    """ sampled Gaussian (derivative of order 0..2) normalised to unit L1 norm (descriptors.py:880-891) """
    if order > 2:
        raise ValueError("Only orders up to 2 are supported")
    resp = np.exp(-vals ** 2 / (2. * sigma ** 2))
    if order == 1:
        resp = -resp * vals
    elif order == 2:
        resp = resp * (vals ** 2 - sigma ** 2)
    return resp / np.abs(resp).sum()


def make_edge_filter2d(sig, phase, points, sup):
    """ anisotropic (3 sigma x sigma) Gaussian derivative on the rotated grid ``points`` (descriptors.py:894-900) """
    ft = (make_gaussian_filter1d(points[0, :], sigma=3 * sig) * make_gaussian_filter1d(points[1, :], sigma=sig, order=phase))
    ft = ft.reshape(sup, sup)
    return ft / np.abs(ft).sum()


def create_filter_bank_lm_2d(radius=16, sigmas=None, nb_orient=8):
    """ Leung-Malik bank: per sigma 'edge' and 'bar' batteries of ``nb_orient`` rotated kernels, a Gaussian and two
    Laplacians of Gaussian (descriptors.py:903-948)

    :return tuple(list(ndarray),list(str)): batteries [n_kernels, 2r+1, 2r+1] and their names
    """
    from scipy.ndimage import gaussian_filter, gaussian_laplace
    from .descriptors import DEFAULT_FILTERS_SIGMAS
    sigmas = DEFAULT_FILTERS_SIGMAS if sigmas is None else sigmas
    support = 2 * radius + 1
    gx, gy = np.mgrid[-radius:radius + 1, radius:-radius - 1:-1]
    grid = np.vstack([gx.ravel(), gy.ravel()])
    impulse = np.zeros((support, support))
    impulse[radius, radius] = 1
    filters, names = [], []
    for sigma in sigmas:
        edges, bars = [], []
        for k in range(nb_orient):
            angle = np.pi * k / nb_orient  # half turn only: the kernels are symmetric
            rot = np.dot(np.array([[np.cos(angle), -np.sin(angle)], [np.sin(angle), np.cos(angle)]]), grid)
            edges.append(make_edge_filter2d(sigma, 1, rot, support))
            bars.append(make_edge_filter2d(sigma, 2, rot, support))
        filters += [np.asarray(edges), np.asarray(bars), gaussian_filter(impulse, sigma)[np.newaxis],
                    gaussian_laplace(impulse, sigma)[np.newaxis], gaussian_laplace(impulse, sigma ** 2)[np.newaxis]]
        names += ['sigma%.1f-%s' % (sigma, n) for n in ('edge', 'bar', 'Gauss', 'GaussLap', 'GaussLap2')]
    return filters, names


def _round_tf32(x):
    """cvt.rna.tf32.f32: round a float32 to 10 explicit mantissa bits, ties away from zero"""
    bits = np.ascontiguousarray(x, dtype=np.float32).view(np.uint32)
    out = ((bits + np.uint32(0x1000)) & np.uint32(0xFFFFE000)).view(np.float32)
    return out


def bank_operand_layout(bank_type):
    """(names, w_tc, NP, orient, n_batt) for 'normal' / 'short' on the HOST.  ``w_tc`` holds, per kernel row, the weights in the operand
    layout of the tensor-core contraction (see isb_lm_texture): float32 [33 kernel rows][hi | lo][10 k-chunks][NP / 8][8 filters][4 taps],
    correlation form (kernels flipped), tf32-rounded value and tf32-rounded remainder, taps 33..39 and the padding filters zero"""
    from .descriptors import SHORT_FILTERS_SIGMAS
    if bank_type == 'short':
        filters, names = create_filter_bank_lm_2d(sigmas=SHORT_FILTERS_SIGMAS, nb_orient=4)
        orient, NP = 4, 48
    else:
        filters, names = create_filter_bank_lm_2d()
        orient, NP = 8, 80
    n_sig = len(filters) // 5
    cols = []
    for s in range(n_sig):      # oriented batteries first: edge s0 | bar s0 | edge s1 | ...
        cols += list(filters[5 * s]) + list(filters[5 * s + 1])
    for s in range(n_sig):      # then Gauss, LoG(sigma), LoG(sigma^2) per sigma
        cols += [filters[5 * s + 2][0], filters[5 * s + 3][0], filters[5 * s + 4][0]]
    assert len(cols) <= NP
    w = np.zeros((_KW, _KWP, NP), dtype=np.float64)
    for j, f in enumerate(cols):
        w[:, :_KW, j] = f[::-1, ::-1]          # ndimage.convolve == correlation with the flipped kernel
    w32 = w.astype(np.float32)
    hi = _round_tf32(w32)
    lo = _round_tf32((w32 - hi).astype(np.float32))
    # [dy][dx][n] -> [dy][half][dx // 4][n // 8][n % 8][dx % 4]: K-major core matrices of 8 filters x 4 taps (16 bytes)
    both = np.stack([hi, lo], axis=1).reshape(_KW, 2, _KWP // 4, 4, NP // 8, 8)
    w_tc = np.ascontiguousarray(both.transpose(0, 1, 2, 4, 5, 3))
    return names, w_tc, NP, orient, len(filters)


def _device_bank(bank_type):
    """(names, d_w_tc, NP, orient, n_batt) for 'normal' / 'short', cached per device (:func:`bank_operand_layout` uploaded once)"""
    eng = get_engine()
    key = (bank_type, eng.device.index)
    if key in _BANK_CACHE:
        return _BANK_CACHE[key]
    names, w_tc, NP, orient, n_batt = bank_operand_layout(bank_type)
    d_w = eng.torch.from_numpy(w_tc).to(eng.device)
    _BANK_CACHE[key] = (names, d_w, NP, orient, n_batt)
    return _BANK_CACHE[key]


def background_kernel(sigma=BACKGROUND_SIGMA, truncate=4.0):
    """scipy.ndimage's 1-D Gaussian (full, 2r+1 taps) and the same kernel folded onto a reflected length-3 axis (3x3)"""
    radius = int(truncate * float(sigma) + 0.5)
    x = np.arange(-radius, radius + 1)
    w = np.exp(-0.5 / (sigma * sigma) * x ** 2)
    w = w / w.sum()
    mix = np.zeros((3, 3))
    for c in range(3):
        idx = (c + x) % 6
        idx = np.where(idx < 3, idx, 5 - idx)        # reflect: (c b a | a b c | c b a)
        for cp in range(3):
            mix[c, cp] = w[idx == cp].sum()
    return np.ascontiguousarray(w), radius, np.ascontiguousarray(mix)


def lm_setup(eng, bank_type, flags):
    """what every launch of the Leung-Malik kernels takes besides the image: (names, d_w, NP, orient, n_batt, w_bg, radius, mix,
    bits, ncol) -- the uploaded bank (:func:`_device_bank`), the background kernel (:func:`background_kernel`; the caller puts its
    taps ``w_bg`` on the device with ``eng.const_device(w_bg, 'lm_bg_w')``), the statistics' bit mask and the number of feature
    columns"""
    names, d_w, NP, orient, n_batt = _device_bank(bank_type)
    w_bg, radius, mix = background_kernel()
    bits, n = flag_bits(flags)
    return names, d_w, NP, orient, n_batt, w_bg, radius, mix, bits, n_batt * 3 * n


def device_lm_features(eng, d_img, d_seg, nb, flags, bank_type='normal', feat=None, col0=0):
    """run isb_lm_texture on device buffers; returns (feat tensor [nb, ld], names, n_cols)"""
    names, d_w, NP, orient, n_batt, w_bg, radius, mix, bits, ncol = lm_setup(eng, bank_type, flags)
    nb = int(nb)
    if feat is None:
        feat = eng.buf('feat_lm', (nb, ncol), eng.torch.float64)
    H, W = int(d_seg.shape[0]), int(d_seg.shape[1])
    d_wbg = eng.const_device(w_bg, 'lm_bg_w')
    ws, wsb = eng.workspace('ws_lm', 'lm_workspace_bytes', H, W, nb, n_batt)
    eng.call('lm_texture', d_img, dtype_code(d_img.dtype), d_seg, H, W, nb, d_wbg, radius, mix, d_w, NP, orient, n_batt, bits, feat,
             int(feat.shape[1]), int(col0), ws, wsb)
    return feat, names, ncol


def _texture_desc_lm_materialised(img, seg, feature_flags, bank_type):
    """ the reference's own sequence (descriptors.py:1078-1098) with every array in memory: background (sigma 150 on all three
    axes), per battery the strongest response per channel (FP64 on the device, ``isb_filter_response_2d``), clip, log-norm
    scaling, then :func:`compute_image2d_color_statistic` -- the route for the statistics the fused kernel does not produce
    (``median``, ``meanGrad``) """
    from .descriptors import (MAX_SIGNAL_RESPONSE, SHORT_FILTERS_SIGMAS, _gauss_smooth_slices, compute_image2d_color_statistic,
                              compute_img_filter_response3d)
    img = np.asarray(img, dtype=np.float64)
    _, _, mix = background_kernel()
    roll = np.ascontiguousarray(np.rollaxis(img, -1, 0))
    smooth = _gauss_smooth_slices(roll, BACKGROUND_SIGMA)          # the two image axes ...
    roll = roll - np.tensordot(mix, smooth, axes=(1, 0))           # ... and the reflected length-3 channel axis
    if bank_type == 'short':
        filters, fl_names = create_filter_bank_lm_2d(sigmas=SHORT_FILTERS_SIGMAS, nb_orient=4)
    else:
        filters, fl_names = create_filter_bank_lm_2d()
    features, names = [], []
    for battery, fl_name in zip(filters, fl_names):
        resp = compute_img_filter_response3d(roll, battery)
        resp[resp > MAX_SIGNAL_RESPONSE] = MAX_SIGNAL_RESPONSE
        norm = np.sqrt(np.sum(resp ** 2))
        if norm == 0 or abs(norm) == np.inf:
            resp = np.zeros(resp.shape)
        else:
            resp = (resp * (np.log(1 + norm) / 0.03)) / norm
        fts, ns = compute_image2d_color_statistic(np.rollaxis(resp, 0, 3), seg, feature_flags, fl_name)
        features.append(fts)
        names += ns
    features = np.nan_to_num(np.concatenate(tuple(features), axis=1))
    features[features == 0] = 0
    names = ['tLM_%s' % n for n in names]
    if features.shape[1] != len(names):
        raise ValueError('features: %r and names %r' % (features.shape, names))
    return features, names


def compute_texture_desc_lm_img2d_clr(img, seg, feature_flags, bank_type='normal'):
    """ texture descriptors of a colour image: statistics of the Leung-Malik filter-bank responses per segment
    (reference descriptors.py:1041-1106)

    :param ndarray img: image [H, W, 3]
    :param ndarray seg: segmentation [H, W]
    :param list(str) feature_flags: subset of ('mean', 'std', 'energy') -- the statistics the device computes
    :param str bank_type: 'normal' (4 sigmas x 8 orientations, 20 batteries) or 'short' (3 x 4, 15 batteries)
    :return tuple(ndarray,list(str)): features [nb_segments, n_batteries * 3 * n_flags], names
    """
    from .descriptors import NAMES_FEATURE_FLAGS, _check_color_image, _check_color_image_segm, _check_unrecognised_feature_names, _device_dtype
    img, seg = _device_dtype(img), np.asarray(seg)
    _check_color_image(img)
    _check_color_image_segm(img, seg)
    if any(f in ('median', 'meanGrad') for f in feature_flags):
        # these two statistics need the filter responses in memory: per-battery path, exactly the reference's sequence
        return _texture_desc_lm_materialised(img, seg, feature_flags, bank_type)
    flags = [f for f in ('mean', 'std', 'energy') if f in feature_flags]
    _check_unrecognised_feature_names(feature_flags)
    eng = get_engine()
    nb = int(seg.max()) + 1
    d_img = eng.to_device(img, 'image')
    d_seg = eng.to_device(seg.astype(np.int32, copy=False), 'seg_in')
    feat, fl_names, ncol = device_lm_features(eng, d_img, d_seg, nb, flags, bank_type)
    features = eng.to_host(feat).copy()
    order = [f for f in NAMES_FEATURE_FLAGS if f in flags]
    names = list(itertools.chain.from_iterable(
        ['tLM_%s-ch%i_%s' % (n, c + 1, f) for f in order for c in range(3)] for n in fl_names))
    features = np.nan_to_num(features)
    features[features == 0] = 0
    if features.shape[1] != len(names):
        raise ValueError('features: %r and names %r' % (features.shape, names))
    return features, names
