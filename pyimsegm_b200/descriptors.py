"""
Per-superpixel descriptors on the GPU.

Mirror of the reference module ``imsegm/descriptors.py`` for the colour / texture statistics that the
SLIC -> features -> GraphCut pipeline uses (same public names, feature-dictionary grammar, column order and
error types).  The reference computes them in its only native module ``imsegm/features_cython.pyx``; here
they come from ``isb_segment_stats_2d`` (``include/imsegm_b200.h``).
"""
import itertools
import logging

import numpy as np

from .engine import FLAG_BITS, dtype_code, flag_bits, get_engine
from .utilities import ImageDimensionError

#: kept for API compatibility with the reference (descriptors.py:25-33); the native path here is CUDA and it
#: is always on -- there is no Python/NumPy fallback behind this switch
USE_CYTHON = True

#: all statistics computable on superpixels (reference descriptors.py:36)
NAMES_FEATURE_FLAGS = ('mean', 'std', 'energy', 'median', 'meanGrad')
#: sigmas of the Leung-Malik filter bank (reference descriptors.py:38-40)
DEFAULT_FILTERS_SIGMAS = (np.sqrt(2), 2, 2 * np.sqrt(2), 4)
SHORT_FILTERS_SIGMAS = (np.sqrt(2), 2, 4)
#: feature sets (reference descriptors.py:42-52)
FEATURES_SET_ALL = {
    'color': ('mean', 'std', 'energy', 'median', 'meanGrad'),
    'tLM': ('mean', 'std', 'energy', 'median', 'meanGrad'),
}
FEATURES_SET_COLOR = {'color': ('mean', 'std', 'energy')}
FEATURES_SET_TEXTURE = {'tLM': ('mean', 'std', 'energy')}
FEATURES_SET_TEXTURE_SHORT = {'tLM_short': ('mean', 'std', 'energy')}
HIST_CIRCLE_DIAGONALS = (10, 20, 30, 40, 50)
#: filter responses are clipped at this value (reference descriptors.py:55)
MAX_SIGNAL_RESPONSE = 1.e6


def _check_color_image_segm(image, segm):
    if image.shape[:2] != segm.shape:
        raise ImageDimensionError('ndarrays - image and segmentation do not match %r vs %r' % (image.shape, segm.shape))
    return True


def _check_gray_image_segm(image, segm):
    if image.shape != segm.shape:
        raise ImageDimensionError('ndarrays - image and segmentation do not match %r vs %r' % (image.shape, segm.shape))
    return True


def _check_color_image(image):
    if image.ndim != 3 or image.shape[2] != 3:
        raise ImageDimensionError('image is not RGB with dims %s' % repr(image.shape))
    return True


def _check_unrecognised_feature_group(feature_flags):
    unknown = [k for k in feature_flags if not (k.startswith('color') or k.startswith('tLM'))]
    if unknown:
        logging.warning('unrecognised following feature groups: %r', unknown)
    return unknown


def _check_unrecognised_feature_names(feature_flags):
    unknown = [k for k in feature_flags if k not in NAMES_FEATURE_FLAGS]
    if unknown:
        logging.warning('unrecognised following feature names: %r', unknown)
    return unknown


def _device_dtype(img):
    img = np.asarray(img)
    if img.dtype in (np.uint8, np.uint16, np.float32, np.float64):
        return img
    return img.astype(np.float64)


def _device_stats(img, seg, flags):
    """[nb, 3 * len(flags)] statistics in the order mean, std, energy (only those requested)"""
    img, seg = _device_dtype(img), np.asarray(seg)
    _check_color_image_segm(img, seg)
    eng = get_engine()
    nb = int(seg.max()) + 1
    d_img = eng.to_device(img, 'image')
    d_seg = eng.to_device(seg.astype(np.int32, copy=False), 'seg_in')
    feat, _, _ = eng.segment_stats(d_img, d_seg, nb, flags)
    return eng.to_host(feat).copy()


def cython_img2d_color_mean(img, seg):
    """ mean colour per segment, f32 pixels accumulated in f64 (reference descriptors.py:209-234) """
    return _device_stats(img, seg, ('mean', ))


def cython_img2d_color_energy(img, seg):
    """ mean squared colour per segment (reference descriptors.py:237-262) """
    return _device_stats(img, seg, ('energy', ))


def cython_img2d_color_std(img, seg, means=None):
    """ colour standard deviation per segment, two-pass about the f32 mean (reference descriptors.py:265-296).
    ``means`` is accepted for signature compatibility; the device path recomputes it in the same launch family """
    return _device_stats(img, seg, ('std', ))


def _host_label_sums(values, seg, nb):
    return np.stack([np.bincount(seg.ravel(), weights=values[..., c].ravel(), minlength=nb) for c in range(3)], axis=1)


def numpy_img2d_color_mean(img, seg):
    """ f64 host computation of the mean colour (the reference's NumPy variant, descriptors.py:299-332) """
    img, seg = np.asarray(img, dtype=float), np.asarray(seg)
    _check_color_image_segm(img, seg)
    nb = int(seg.max()) + 1
    cnt = np.bincount(seg.ravel(), minlength=nb).astype(float)
    cnt[cnt == 0] = -1
    return _host_label_sums(img, seg, nb) / cnt[:, None]


def numpy_img2d_color_std(img, seg, means=None):
    """ f64 host computation of the colour STD (reference descriptors.py:335-376) """
    img, seg = np.asarray(img, dtype=float), np.asarray(seg)
    _check_color_image_segm(img, seg)
    if means is None:
        means = numpy_img2d_color_mean(img, seg)
    nb = int(seg.max()) + 1
    if len(means) < nb:
        raise ValueError('number of means (%i) should be equal to number of labels (%i)' % (len(means), nb))
    cnt = np.bincount(seg.ravel(), minlength=nb).astype(float)
    cnt[cnt == 0] = -1
    var = _host_label_sums((img - np.asarray(means)[seg]) ** 2, seg, nb) / cnt[:, None]
    var[var == 0] = 0
    return np.sqrt(var)


def numpy_img2d_color_energy(img, seg):
    """ f64 host computation of the colour energy (reference descriptors.py:379-417) """
    img, seg = np.asarray(img, dtype=float), np.asarray(seg)
    _check_color_image_segm(img, seg)
    nb = int(seg.max()) + 1
    cnt = np.bincount(seg.ravel(), minlength=nb).astype(float)
    cnt[cnt == 0] = -1
    return _host_label_sums(img ** 2, seg, nb) / cnt[:, None]


def _device_median(img, seg, channels):
    """per-label median of every channel on the device (``isb_segment_median``: counting sort by label + radix select)"""
    eng = get_engine()
    img = _device_dtype(img)
    n_px = int(seg.size)
    nb = int(seg.max()) + 1
    d_img = eng.to_device(img, 'median_img')
    d_seg = eng.to_device(np.ascontiguousarray(seg, dtype=np.int32), 'seg_in')
    out = eng.buf('median_out', (nb, channels), eng.torch.float64)
    ws, wsb = eng.workspace('ws_median', 'segment_median_workspace_bytes', n_px, nb)
    eng.call('segment_median', d_img, dtype_code(img.dtype), d_seg, n_px, channels, nb, out, ws, wsb)
    return eng.to_host(out).copy()


def numpy_img2d_color_median(img, seg):
    """ per-segment, per-channel median (reference descriptors.py:420-455: a pure-Python loop over the pixels there, no native
    path); NaN for labels without pixels """
    img, seg = np.asarray(img), np.asarray(seg)
    _check_color_image_segm(img, seg)
    return _device_median(img, seg, 3)


def _device_gray_stats(img, seg, flags):
    img, seg = _device_dtype(img), np.asarray(seg)
    _check_gray_image_segm(img, seg)
    eng = get_engine()
    nb = int(seg.max()) + 1
    d_img = eng.to_device(img, 'image_gray')
    d_seg = eng.to_device(seg.astype(np.int32, copy=False), 'seg_in')
    bits, n = flag_bits(flags)
    feat = eng.buf('feat_gray', (nb, n), eng.torch.float64)
    ws, wsb = eng.workspace('ws_gray', 'gray_stats_workspace_bytes', nb)
    eng.call('gray_stats', d_img, dtype_code(img.dtype), d_seg, img.size, nb, bits, feat, n, 0, ws, wsb)
    return eng.to_host(feat).copy()


def cython_img3d_gray_mean(img, seg):
    """ mean intensity per segment of a gray volume (reference descriptors.py:458-487) """
    return _device_gray_stats(img, seg, ('mean', ))[:, 0]


def cython_img3d_gray_energy(img, seg):
    """ mean squared intensity per segment of a gray volume (reference descriptors.py:490-515) """
    return _device_gray_stats(img, seg, ('energy', ))[:, 0]


def cython_img3d_gray_std(img, seg, mean=None):
    """ intensity STD per segment of a gray volume, two-pass about the f32 mean (reference descriptors.py:518-551) """
    return _device_gray_stats(img, seg, ('std', ))[:, 0]


def cython_label_hist_seg2d(segm_select, struc_elem, nb_labels):
    """ histogram of the labels under a structuring element (reference descriptors.py:1479-1498) """
    segm_select, struc_elem = np.array(segm_select, dtype=float), np.asarray(struc_elem)
    if segm_select.shape != struc_elem.shape:
        raise ValueError('segm. %r and mask %r sizes do not match' % (segm_select.shape, struc_elem.shape))
    segm_select[np.isnan(segm_select)] = -1
    eng = get_engine()
    d_a = eng.to_device(segm_select.astype(np.int16), 'hist_segm')
    d_b = eng.to_device(struc_elem.astype(np.int16), 'hist_selem')
    hist = eng.buf('hist_out', (int(nb_labels),), eng.torch.int32)
    eng.call('label_hist_2d', d_a, d_b, segm_select.shape[0], segm_select.shape[1], int(nb_labels), hist)
    return eng.to_host(hist).astype(float)


def ray_angle_tables(angle_step):
    """(sin, cos) float32 tables of the ray directions exactly as features_cython.pyx:247-268 forms them"""
    angles = np.arange(0, 360, angle_step, dtype=np.float32)
    rads = [float(np.float32(np.deg2rad(a))) for a in angles]
    return np.array([np.sin(r) for r in rads], dtype=np.float32), np.array([np.cos(r) for r in rads], dtype=np.float32)


def cython_ray_features_seg2d(seg_binary, position, angle_step=5., edge='up'):
    """ Ray features: distance from ``position`` to the first boundary along rays every ``angle_step`` degrees
    (reference descriptors.py:1628-1660).  ``position`` may also be an [n, 2] array: all positions run in one launch.

    :return ndarray: ray distances, float32 [n_angles] (or [n, n_angles])
    """
    edge_int = {'down': -1, 'up': 1}[edge]
    seg = np.array(seg_binary, dtype=np.int8)
    pos = np.atleast_2d(np.array(position, dtype=np.int32))
    sin_a, cos_a = ray_angle_tables(float(angle_step))
    eng = get_engine()
    d_seg, d_pos = eng.to_device(seg, 'ray_seg'), eng.to_device(pos, 'ray_pos')
    d_s, d_c = eng.to_device(sin_a, 'ray_sin'), eng.to_device(cos_a, 'ray_cos')
    out = eng.buf('ray_out', (len(pos), len(sin_a)), eng.torch.float32)
    eng.call('ray_features_2d', d_seg, seg.shape[0], seg.shape[1], d_pos, len(pos), d_s, d_c, len(sin_a), edge_int, out)
    res = eng.to_host(out).copy()
    return res[0] if np.ndim(position) == 1 else res


# ---------------------------------------------------------------------------------------------------------------------
# gray volumes: host (NumPy) variants and the statistic driver (reference descriptors.py:545-787)
# ---------------------------------------------------------------------------------------------------------------------

def _gray_counts(seg):
    nb = int(np.max(seg)) + 1
    cnt = np.bincount(np.ravel(seg), minlength=nb).astype(float)
    cnt[cnt == 0] = -1          # "just for not dividing by 0"
    return nb, cnt


def numpy_img3d_gray_mean(img, seg):
    """ f64 host computation of the mean intensity per segment of a gray volume (reference descriptors.py:545-580) """
    img, seg = np.asarray(img, dtype=float), np.asarray(seg)
    _check_gray_image_segm(img, seg)
    nb, cnt = _gray_counts(seg)
    return np.bincount(seg.ravel(), weights=img.ravel(), minlength=nb) / cnt


def numpy_img3d_gray_std(img, seg, means=None):
    """ f64 host computation of the intensity STD per segment of a gray volume (reference descriptors.py:583-617) """
    img, seg = np.asarray(img, dtype=float), np.asarray(seg)
    _check_gray_image_segm(img, seg)
    if means is None:
        means = numpy_img3d_gray_mean(img, seg)
    nb, cnt = _gray_counts(seg)
    if len(means) < nb:
        raise ValueError('number of means (%i) should be equal to number of labels (%i)' % (len(means), nb))
    var = np.bincount(seg.ravel(), weights=((img - np.asarray(means)[seg]) ** 2).ravel(), minlength=nb) / cnt
    var[var == 0] = 0
    return np.sqrt(var)


def numpy_img3d_gray_energy(img, seg):
    """ f64 host computation of the mean squared intensity per segment of a gray volume (reference descriptors.py:620-648) """
    img, seg = np.asarray(img, dtype=float), np.asarray(seg)
    _check_gray_image_segm(img, seg)
    nb, cnt = _gray_counts(seg)
    return np.bincount(seg.ravel(), weights=(img ** 2).ravel(), minlength=nb) / cnt


def numpy_img3d_gray_median(img, seg):
    """ median intensity per segment of a gray volume (reference descriptors.py:651-676; NaN for absent labels) """
    img, seg = np.asarray(img), np.asarray(seg)
    _check_gray_image_segm(img, seg)
    return _device_median(img, seg, 1)[:, 0]


def compute_image3d_gray_statistic(image, segm, feature_flags=NAMES_FEATURE_FLAGS, ch_name='gray'):
    """ statistics of a gray volume over the segments (reference descriptors.py:679-784); mean / std / energy run in
    ``isb_gray_stats`` (or the NumPy variants when ``USE_CYTHON`` is off, as in the reference)

    :return tuple(ndarray,list(str)): features [nb_segments, nb_statistics], column names
    """
    image, segm = np.asarray(image), np.asarray(segm)
    _check_gray_image_segm(image, segm)
    if not list(feature_flags):
        raise ValueError('some features has to be selected')
    image = np.nan_to_num(image)
    fn_mean = cython_img3d_gray_mean if USE_CYTHON else numpy_img3d_gray_mean
    columns = {}
    native = [f for f in ('mean', 'std', 'energy') if f in feature_flags]
    if native and USE_CYTHON:
        stats = _device_gray_stats(image, segm, native)       # one launch family for all three
        for i, f in enumerate(native):
            columns[f] = stats[:, i]
    elif native:
        mean = numpy_img3d_gray_mean(image, segm) if 'mean' in native else None
        if 'mean' in native:
            columns['mean'] = mean
        if 'std' in native:
            columns['std'] = numpy_img3d_gray_std(image, segm, mean)
        if 'energy' in native:
            columns['energy'] = numpy_img3d_gray_energy(image, segm)
    if 'median' in feature_flags:
        columns['median'] = numpy_img3d_gray_median(image, segm)
    if 'meanGrad' in feature_flags:
        grad = np.zeros(image.shape, dtype=image.dtype if image.dtype.kind == 'f' else float)
        for i in range(image.shape[0]):
            grad[i] = np.sum(np.gradient(image[i]), axis=0)
        columns['meanGrad'] = fn_mean(grad, segm)
    order = [f for f in NAMES_FEATURE_FLAGS if f in feature_flags]
    names = ['%s_%s' % (ch_name, f) for f in order]
    _check_unrecognised_feature_names(feature_flags)
    nb = int(segm.max()) + 1
    features = np.stack([columns[f] for f in order], axis=1) if order else np.empty((nb, 0))
    features = np.nan_to_num(features)
    features[features == 0] = 0
    if features.shape[1] != len(names):
        raise ValueError('features: %r and names %r' % (features.shape, names))
    return features, names


def _as_slices(img):
    img = np.ascontiguousarray(img, dtype=np.float64)
    if img.ndim not in (2, 3):
        raise ValueError('expected a 2-D image or a stack of 2-D slices, got shape %r' % (img.shape, ))
    return img, (img[np.newaxis] if img.ndim == 2 else img)


def compute_img_filter_response2d(img, filter_battery):
    """ the strongest response of a 2-D image over a battery of filters, ``max_f convolve(img, filter_f)`` (true convolution,
    mode 'reflect'; reference descriptors.py:951-966) -- FP64 on the device (``isb_filter_response_2d``) """
    filter_battery = np.ascontiguousarray(filter_battery, dtype=np.float64)
    if filter_battery.ndim != 3:
        raise ValueError('wrong battery dim %r' % (filter_battery.shape, ))
    if np.ndim(img) != 2:
        raise ValueError('expected a 2-D image, got shape %r' % (np.shape(img), ))
    return compute_img_filter_response3d(np.asarray(img)[np.newaxis], filter_battery)[0]


def compute_img_filter_response3d(img, filter_battery):
    """ :func:`compute_img_filter_response2d` of every slice ``img[i]`` in one launch (reference descriptors.py:969-983) """
    filter_battery = np.ascontiguousarray(filter_battery, dtype=np.float64)
    if filter_battery.ndim != 3:
        raise ValueError('wrong battery dim %r' % (filter_battery.shape, ))
    img = np.ascontiguousarray(img, dtype=np.float64)
    if img.ndim != 3:
        raise ValueError('expected a stack of 2-D slices, got shape %r' % (img.shape, ))
    eng = get_engine()
    d_img = eng.to_device(img, 'resp_img')
    d_ker = eng.to_device(filter_battery, 'resp_kernels')
    out = eng.buf('resp_out', img.shape, eng.torch.float64)
    eng.call('filter_response_2d', d_img, img.shape[0], img.shape[1], img.shape[2], d_ker, filter_battery.shape[0], filter_battery.shape[1],
             filter_battery.shape[2], out)
    return eng.to_host(out).copy()


def _gauss_smooth_slices(stack, sigma):
    """scipy ``gaussian_filter(slice, sigma)`` of every 2-D slice of a float64 stack [n, H, W], FP64 on the device"""
    from .engine import gaussian_half_kernel
    w_half, radius = gaussian_half_kernel(sigma)
    eng = get_engine()
    d_img = eng.to_device(stack, 'smooth_img')
    d_w = eng.to_device(w_half, 'smooth_w')
    tmp = eng.buf('smooth_tmp', stack.shape, eng.torch.float64)
    out = eng.buf('smooth_out', stack.shape, eng.torch.float64)
    eng.call('gaussian_filter_2d', d_img, stack.shape[0], stack.shape[1], stack.shape[2], d_w, radius, tmp, out)
    return eng.to_host(out).copy()


def image_subtract_gauss_smooth(img, sigma):
    """ subtract from every slice ``img[i]`` its own Gaussian-smoothed copy -- a high-pass per slice (reference
    descriptors.py:986-1000; scipy's ``gaussian_filter`` semantics, FP64 on the device) """
    if sigma <= 0:
        return img
    src, stack = _as_slices(img)
    if src.ndim != 3:
        raise ValueError('expected a stack of 2-D slices, got shape %r' % (src.shape, ))
    return np.asarray(img) - _gauss_smooth_slices(stack, sigma).reshape(src.shape)


def compute_texture_desc_lm_img3d_val(img, seg, feature_flags, bank_type='normal'):
    """ Leung-Malik texture statistics of a gray VOLUME (reference descriptors.py:1003-1038): slice-wise high-pass (sigma 150),
    slice-wise battery responses, clipping, log-norm scaling over the whole volume, statistics over the 3-D segments.
    Generic FP64 kernels (``isb_gaussian_filter_2d``, ``isb_filter_response_2d``, ``isb_gray_stats``): this is the completeness
    path for volumes -- the tensor-core kernel of the hot path is :func:`compute_texture_desc_lm_img2d_clr`.

    :return tuple(ndarray,list(str)): features [nb_segments, nb_batteries * nb_statistics], names
    """
    img, seg = np.asarray(img), np.asarray(seg)
    _check_gray_image_segm(img, seg)
    img = image_subtract_gauss_smooth(img, 150)
    if bank_type == 'short':
        filters, fl_names = create_filter_bank_lm_2d(sigmas=SHORT_FILTERS_SIGMAS, nb_orient=4)
    else:
        filters, fl_names = create_filter_bank_lm_2d()
    features, names = [], []
    for battery, fl_name in zip(filters, fl_names):
        response = compute_img_filter_response3d(img, battery)
        response[response > MAX_SIGNAL_RESPONSE] = MAX_SIGNAL_RESPONSE
        l_n = np.sqrt(np.sum(np.power(response, 2)))
        if l_n == 0 or abs(l_n) == np.inf:
            response = np.zeros(response.shape)
        else:
            response = (response * (np.log(1 + l_n) / 0.03)) / l_n
        fts, ns = compute_image3d_gray_statistic(response, seg, feature_flags, fl_name)
        features.append(fts)
        names += ns
    features = np.nan_to_num(np.concatenate(tuple(features), axis=1))
    features[features == 0] = 0
    names = ['tLM_%s' % name for name in names]
    if features.shape[1] != len(names):
        raise ValueError('features: %r and names %r' % (features.shape, names))
    return features, names


def compute_selected_features_gray3d(img, segments, feature_flags=FEATURES_SET_COLOR):
    """ selected features of a gray volume (reference descriptors.py:1109-1164): ``{'color': flags}`` -> intensity statistics,
    ``{'tLM[_short]': flags}`` -> texture statistics (see :func:`compute_texture_desc_lm_img3d_val`)

    :return tuple(ndarray,list(str)): features [nb_segments, nb_features], names
    """
    img, segments = np.asarray(img), np.asarray(segments)
    _check_gray_image_segm(img, segments)
    if not feature_flags:
        raise ValueError('some features has to be selected')
    features, names = [], []
    if any(k.startswith('color') for k in feature_flags):
        flags = np.unique([feature_flags[k] for k in feature_flags if k.startswith('color')])
        fts, ns = compute_image3d_gray_statistic(img, segments, flags)
        features.append(fts)
        names += ns
    for k in [k for k in feature_flags if k.startswith('tLM')]:
        bank_type = k.split('_')[-1] if '_' in k else 'normal'
        fts, ns = compute_texture_desc_lm_img3d_val(img, segments, feature_flags[k], bank_type)
        features.append(fts)
        names += ns
    _check_unrecognised_feature_group(feature_flags)
    if not features:
        return np.array([[]] * (int(segments.max()) + 1)), []
    features = np.nan_to_num(np.concatenate(tuple(features), axis=1))
    features[features == 0] = 0          # -0 -> +0
    if features.shape[1] != len(names):
        raise ValueError('features: %r and names %r' % (features.shape, names))
    return features, names


# ---------------------------------------------------------------------------------------------------------------------
# label histograms about positions (reference descriptors.py:1288-1528)
# ---------------------------------------------------------------------------------------------------------------------

def adjust_bounding_box_crop(image_size, bbox_size, position):
    """ the part of a box of ``bbox_size`` centred on ``position`` that lies inside an image, as index ranges of the image
    and of the box (reference descriptors.py:1355-1393)

    :return tuple: im_begin, im_end, bb_begin, bb_end
    """
    if len(image_size) != len(bbox_size):
        raise ValueError('incompatible sizes %r != %r' % (image_size, bbox_size))
    im_size, bb_size, pos = np.asarray(image_size), np.asarray(bbox_size), np.asarray(position)
    half_lo, half_hi = np.floor(bb_size / 2.).astype(int), np.ceil(bb_size / 2.).astype(int)
    im_begin = np.maximum(pos - half_lo, 0)
    im_end = np.minimum(pos + half_hi, im_size)
    bb_begin = np.where(im_begin == 0, half_lo - pos, 0)
    bb_end = np.where(im_end == im_size, half_lo + (im_size - pos), bb_size)
    if not np.array_equal(im_end - im_begin, bb_end - bb_begin):
        raise ValueError('different sizes of image %r and bounding box %r mask' % (im_end - im_begin, bb_end - bb_begin))
    return tuple(int(v) for v in im_begin), tuple(int(v) for v in im_end), tuple(int(v) for v in bb_begin), tuple(int(v) for v in bb_end)


def _device_label_hists(segm, positions, nb_labels, diameters=None, struc_elem=None):
    """label histograms under discs (``diameters``) or one explicit structuring element about every position, one launch
    (``isb_disc_label_hist``).  ``segm`` is [H, W] labels or [H, W, K] per-label maps.
    Returns (hist [n_pos, n_elems, nb_labels], sizes [n_pos, n_elems])."""
    segm = np.asarray(segm)
    pos = np.ascontiguousarray(np.atleast_2d(np.asarray(positions)).astype(np.int32))
    if pos.shape[1] != 2:
        raise ValueError('positions have to be (row, col) pairs, got shape %r' % (pos.shape, ))
    H, W = int(segm.shape[0]), int(segm.shape[1])
    eng = get_engine()
    torch = eng.torch
    d_pos = eng.to_device(pos, 'hist_pos')
    d_seg = d_proba = None
    if segm.ndim == 2:
        lab = np.array(segm, dtype=float)
        lab[np.isnan(lab)] = -1
        d_seg = eng.to_device(lab.astype(np.int32), 'hist_segm32')
    else:
        d_proba = eng.to_device(np.ascontiguousarray(segm, dtype=np.float64), 'hist_proba')
    d_diam = d_sel = None
    mh = mw = 0
    if struc_elem is not None:
        sel = np.ascontiguousarray(np.asarray(struc_elem) == 1, dtype=np.uint8)
        mh, mw = int(sel.shape[0]), int(sel.shape[1])
        d_sel = eng.to_device(sel, 'hist_selem8')
        n_el = 1
    else:
        diam = np.ascontiguousarray(np.asarray(diameters, dtype=np.int32))
        d_diam = eng.to_device(diam, 'hist_diam')
        n_el = len(diam)
    hist = eng.buf('hist_out64', (len(pos), n_el, int(nb_labels)), torch.float64)
    sizes = eng.buf('hist_sizes', (len(pos), n_el), torch.float64)
    eng.call('disc_label_hist', d_seg, d_proba, H, W, d_pos, len(pos), d_diam, n_el, d_sel, mh, mw, int(nb_labels), hist, sizes)
    return eng.to_host(hist).copy(), eng.to_host(sizes).copy()


def _check_position_inside(shape, position):
    if any(p < 0 or p >= s for p, s in zip(position, shape)):
        raise ValueError('position %r lies outside the segmentation %r' % (position, tuple(shape)))


def compute_label_hist_segm(segm, position, struc_elem, nb_labels):
    """ histogram of the labels under a structuring element centred on ``position`` (reference descriptors.py:1396-1441)

    :return tuple(ndarray,float): counts per label, number of element pixels inside the image
    """
    segm, struc_elem = np.asarray(segm), np.asarray(struc_elem)
    if segm.ndim != len(position):
        raise ValueError('dim of position %r should match the segmentation %r dim' % (position, segm.shape))
    position = [int(p) for p in position]
    _check_position_inside(segm.shape, position)
    hist, sizes = _device_label_hists(segm, [position], nb_labels, struc_elem=struc_elem)
    return hist[0, 0], struc_elem.dtype.type(sizes[0, 0])


def compute_label_hist_proba(segm, position, struc_elem):
    """ sums of the per-label maps ``segm[..., l]`` under a structuring element centred on ``position``
    (reference descriptors.py:1501-1528)

    :return tuple(ndarray,int): sums per label, number of element pixels inside the image
    """
    segm, struc_elem = np.asarray(segm), np.asarray(struc_elem)
    if segm.ndim != (len(position) + 1):
        raise ValueError('segment. (%r) should have larger (+1) dim than position %i' % (segm.shape, len(position)))
    position = [int(p) for p in position]
    _check_position_inside(segm.shape[:2], position)
    hist, sizes = _device_label_hists(segm, [position], segm.shape[-1], struc_elem=struc_elem)
    return hist[0, 0], struc_elem.dtype.type(sizes[0, 0])


def compute_label_histograms_positions(segm, positions, diameters=HIST_CIRCLE_DIAGONALS, nb_labels=None):
    """ label frequencies in concentric rings (discs of growing ``diameters`` minus the previous disc) about the positions
    (reference descriptors.py:1288-1352); every disc of every position is counted in one kernel launch

    :param ndarray segm: labels [H, W] or per-label maps [H, W, K]
    :return tuple(ndarray,list(str)): features [nb_positions, nb_diameters * nb_labels], names
    """
    segm = np.asarray(segm)
    pos_dim = np.asarray(positions).shape[1]
    if (segm.ndim - pos_dim) not in (0, 1):
        raise ValueError('dimension %r and %r difference should be 0 or 1' % (segm.ndim, pos_dim))
    if nb_labels is None:
        nb_labels = int(segm.max()) + 1 if segm.ndim == pos_dim else segm.shape[-1]
    int_pos = [[int(p) for p in pos] for pos in positions]
    for pos in int_pos:
        _check_position_inside(segm.shape[:2], pos)
    hist, sizes = _device_label_hists(segm, int_pos, nb_labels, diameters=list(diameters))
    ring_size = np.diff(np.concatenate([np.zeros((len(int_pos), 1)), sizes], axis=1), axis=1)
    if np.any(ring_size <= 0):
        raise ValueError('norm or element should be positive')
    ring_hist = np.diff(np.concatenate([np.zeros((len(int_pos), 1, nb_labels)), hist], axis=1), axis=1)
    if np.any(ring_hist < 0):
        raise ValueError('outer elem should have more labels then the inter')
    pos_hists = (ring_hist / ring_size[:, :, None]).reshape(len(int_pos), -1)
    feature_names = ['hist-d_%i-lb_%i' % (d, lb) for d in diameters for lb in range(nb_labels)]
    if pos_hists.shape[1] != len(feature_names):
        raise ValueError('histogram: %r and names %r' % (pos_hists.shape, feature_names))
    return pos_hists, feature_names


# ---------------------------------------------------------------------------------------------------------------------
# Ray features about positions (reference descriptors.py:1545-2041)
# ---------------------------------------------------------------------------------------------------------------------

def numpy_ray_features_seg2d(seg_binary, position, angle_step=5., edge='up'):
    """ the reference keeps a NumPy twin of its Cython ray tracer (descriptors.py:1663-1708); here both names run the CUDA kernel """
    return cython_ray_features_seg2d(seg_binary, position, angle_step, edge)


def _smooth_rays(ray_dist, smooth_coef):
    if smooth_coef is not None and smooth_coef > 0:
        from scipy.ndimage import gaussian_filter1d
        return gaussian_filter1d(ray_dist, smooth_coef)
    return ray_dist


def compute_ray_features_segm_2d(seg_binary, position, angle_step=5., smooth_coef=0, edge='up'):
    """ Ray features of one position: distance to the first boundary every ``angle_step`` degrees, optionally smoothed along
    the angle (reference descriptors.py:1711-1759) """
    seg_binary = np.asarray(seg_binary)
    if seg_binary.ndim != len(position):
        raise ValueError('Segmentation dim of %r and position (%i) does not match' % (seg_binary.ndim, len(position)))
    ray_dist = cython_ray_features_seg2d(seg_binary.astype(bool), tuple(map(int, position)), angle_step, edge)
    return _smooth_rays(ray_dist, smooth_coef)


def shift_ray_features(ray_dist, method='phase'):
    """ rotate a Ray feature vector to start at its dominant direction -- rotation invariance (reference descriptors.py:1762-1802)

    :param str method: 'phase' (phase of the strongest Fourier component) or 'max' (largest distance)
    :return tuple(ndarray,float): shifted vector, shift in degrees
    """
    ray_dist = np.asarray(ray_dist)
    angle_step = 360 / len(ray_dist)
    if method == 'phase':
        ext = np.hstack([ray_dist] * 5)
        spectrum = np.fft.fft(ext - np.mean(ext)) / float(len(ext))
        half = len(ext) // 2
        idx = np.argmax(np.abs(spectrum)[:half])
        shift = np.rad2deg(-np.angle(spectrum)[:half][idx])
        shift = (360 + shift) if shift < 0 else shift
    else:
        shift = float(np.argmax(ray_dist) * angle_step)
    step = int(round(shift / angle_step))
    return np.array(ray_dist[step:].tolist() + ray_dist[:step].tolist()), shift


def compute_ray_features_positions(segm, list_positions, angle_step=5., border_labels=None, segm_open=None, smooth_ray=None,
                                   shifting=True, edge='up'):
    """ Ray features of many positions of a segmentation whose ``border_labels`` form the boundary
    (reference descriptors.py:1805-1884); the rays of ALL positions are traced in one kernel launch

    :return tuple(ndarray,list(float),list(str)): rays [nb_positions, nb_angles], shifts, names
    """
    segm = np.asarray(segm)
    pos_dim = np.asarray(list_positions).shape[1]
    if (segm.ndim - pos_dim) not in (0, 1):
        raise ValueError('dimension %s and %s difference should be 0 or 1' % (segm.ndim, pos_dim))
    border_labels = border_labels if border_labels is not None else [0]
    if segm.ndim > pos_dim:
        segm = np.argmax(segm, axis=-1)
    seg_binary = np.isin(segm, list(border_labels))
    if isinstance(segm_open, int):
        seg_binary = binary_opening_disk(seg_binary, segm_open)     # skimage.morphology.opening(mask, disk(r)) on the device
    positions = [tuple(map(int, pos)) for pos in list_positions]
    rays = np.atleast_2d(cython_ray_features_seg2d(seg_binary, np.asarray(positions), angle_step, edge))
    pos_rays, pos_shift = [], []
    for ray_dist in rays:
        ray_dist = _smooth_rays(ray_dist, smooth_ray)
        shift = 0
        if shifting:
            ray_dist, shift = shift_ray_features(ray_dist)
        pos_rays.append(ray_dist)
        pos_shift.append(float(shift))
    nb_rays = rays.shape[1]
    feature_names = ['ray-lb_%s-agl_%i' % (''.join(map(str, border_labels)), int(a)) for a in np.linspace(0, 360 - angle_step, nb_rays)]
    pos_rays = np.array(pos_rays)
    if pos_rays.shape[1] != len(feature_names):
        raise ValueError('Ray features: %r and names %r' % (pos_rays.shape, feature_names))
    return pos_rays, pos_shift, feature_names


def binary_opening_disk(mask, radius):
    """ morphological opening of a binary 2-D mask with a disc of ``radius`` pixels, borders reflected -- what the reference gets
    from ``skimage.morphology.opening(mask, morphology.disk(radius))`` (descriptors.py:1873-1876); ``isb_binary_opening_disk`` """
    mask = np.ascontiguousarray(mask, dtype=np.uint8)
    if mask.ndim != 2:
        raise ValueError('expected a 2-D mask, got shape %r' % (mask.shape, ))
    eng = get_engine()
    d_in = eng.to_device(mask, 'morph_in')
    tmp = eng.buf('morph_tmp', mask.shape, eng.torch.uint8)
    out = eng.buf('morph_out', mask.shape, eng.torch.uint8)
    eng.call('binary_opening_disk', d_in, mask.shape[0], mask.shape[1], int(radius), tmp, out)
    return eng.to_host(out).astype(bool)


def compute_ray_features_segm_2d_vectors(seg_binary, position, angle_step=5., smooth_coef=0, edge='up'):
    """ the reference's legacy Ray tracer (descriptors.py:1545-1625, "USES WHOLE IMAGE ROTATION SO IT IS VERY SLOW"): the mask is
    shifted so that ``position`` is the image centre and rotated (nearest neighbour) once per angle; the distances are read along the
    four half-axes of every rotated copy.  Kept for API completeness on scipy's ``ndimage.shift`` / ``rotate`` like the original --
    it is not on any accelerated path; :func:`compute_ray_features_segm_2d` is the device tracer.

    :return ndarray: distances, -1 where no boundary is met
    """
    from scipy import ndimage
    seg_binary = np.asarray(seg_binary).astype(bool)
    angle_range = 90 if (90 % angle_step) == 0 else 180
    nb_steps = int(angle_range / angle_step)
    ray_dist = np.full(int(nb_steps * 2 * (180 / angle_range)), -1)
    if bool(seg_binary[int(position[0]), int(position[1])]) and edge == 'up':
        return ray_dist * 0            # the position already sits on the boundary label
    size = np.array(seg_binary.shape)
    shift = size / 2 - np.asarray(position)
    pad = np.abs(shift).astype(int)
    canvas = np.zeros(size + 2 * pad)
    canvas[pad[0]:pad[0] + size[0], pad[1]:pad[1] + size[1]] = seg_binary
    centred = ndimage.shift(canvas, shift.tolist(), order=0, cval=True)

    def first_edge(line):
        """distance to the first boundary pixel ('up') or to the end of the first boundary run ('down') along a half-axis"""
        hits = np.flatnonzero(line)
        if not hits.size:
            return None
        if edge == 'up':
            return int(hits[0])
        if edge == 'down':
            gaps = np.flatnonzero(~line[hits[0]:])
            return int(hits[0] + gaps[0]) if gaps.size else None
        return None

    for i, ang in enumerate(np.arange(0, angle_range, angle_step)):
        rot = ndimage.rotate(centred, ang + 90, order=0, reshape=True, cval=True).astype(bool)
        cy, cx = (np.array(rot.shape) / 2).astype(int)
        half_axes = [rot[:cy, cx][::-1], rot[cy, cx:], rot[cy:, cx], rot[cy, :cx][::-1]]
        if angle_range == 180:
            half_axes = [half_axes[0], half_axes[2]]
        for j, line in enumerate(half_axes):
            dist = first_edge(line)
            if dist is not None:
                ray_dist[i + j * nb_steps] = dist
    if smooth_coef > 0:
        ray_dist = ndimage.gaussian_filter1d(ray_dist, smooth_coef)
    return np.array(ray_dist)


def interpolate_ray_dist(ray_dists, order='spline'):
    """ fill the missing (-1) entries of a periodic Ray vector (reference descriptors.py:1887-1951)

    :param str|int order: polynomial degree, 'spline' (periodic interpolating spline) or 'cos' (fitted sinusoid)
    """
    ray_dists = np.array(ray_dists)
    x_space = np.arange(len(ray_dists))
    missing = ray_dists == -1
    x_train, y_train = x_space[~missing], ray_dists[~missing]
    if not y_train.size:
        return ray_dists
    if isinstance(order, int):
        ray_dists[missing] = np.poly1d(np.polyfit(x_train, y_train, order))(x_space[missing])
    elif order == 'spline':
        from scipy import interpolate
        n = len(x_space)
        spline = interpolate.InterpolatedUnivariateSpline(np.hstack((x_train - n, x_train, x_train + n)), np.tile(y_train, 3))
        ray_dists[missing] = spline(x_space[missing])
    elif order == 'cos':
        from scipy import optimize

        def _wave(x, t):
            return x[0] + x[1] * np.sin(x[2] + x[3] * t)

        x0 = np.array([np.mean(y_train), (y_train.max() - y_train.min()) / 2., 0, len(x_space) / np.pi])
        fit = optimize.least_squares(lambda x, t, y: _wave(x, t) - y, x0, gtol=1e-1, args=(x_train, y_train))
        ray_dists[missing] = _wave(fit.x, x_space[missing])
    return ray_dists


def reconstruct_ray_features_2d(position, ray_features, shift=0):
    """ the boundary points a Ray vector describes about ``position`` (reference descriptors.py:1954-1999)

    :return ndarray: points [nb_valid_rays, 2]
    """
    if len(position) != 2:
        raise ValueError('positions has to have 2 coordinates')
    if len(ray_features) <= 2:
        raise ValueError('required at least 2 features')
    ray_features = np.asarray(ray_features)
    angles = (np.pi / 2.) - np.linspace(0, 2 * np.pi, len(ray_features), endpoint=False) - np.deg2rad(shift)
    valid = np.logical_and(ray_features >= 0, ~np.isinf(ray_features))
    angles, rays = angles[valid], ray_features[valid]
    return np.tile(position, (len(rays), 1)) + np.array([np.cos(angles) * rays, np.sin(angles) * rays]).T


def reduce_close_points(points, dist_thr):
    """ drop points until no two of them are closer than ``dist_thr``; of the closest pair the later one goes
    (reference descriptors.py:2002-2041) """
    if len(points) <= 2:
        raise ValueError('too few point to be reduced')
    from scipy import spatial
    points = np.asarray(points)
    dist = spatial.distance.cdist(points, points, metric='euclidean')
    np.fill_diagonal(dist, np.inf)
    while len(points) > 0 and dist.size and np.min(dist) < dist_thr:
        drop = max(np.unravel_index(dist.argmin(), dist.shape))
        points = np.delete(points, drop, axis=0)
        dist = np.delete(np.delete(dist, drop, axis=0), drop, axis=1)
    return points


def compute_image2d_color_statistic(image, segm, feature_flags=NAMES_FEATURE_FLAGS, color_name='color'):
    """ statistics of a colour image over the segments; columns are statistic-major, channel-minor
    (reference descriptors.py:787-863)

    :return tuple(ndarray,list(str)): features [nb_segments, 3 * nb_statistics], column names
    """
    image, segm = np.asarray(image), np.asarray(segm)
    _check_color_image(image)
    _check_color_image_segm(image, segm)
    ch_names = ['%s-ch%i' % (color_name, i + 1) for i in range(3)]
    native = [f for f in ('mean', 'std', 'energy') if f in feature_flags]
    blocks = {}
    if native:
        stats = _device_stats(image, segm, native)
        for i, f in enumerate(native):
            blocks[f] = stats[:, 3 * i:3 * i + 3]
    if 'median' in feature_flags:
        blocks['median'] = numpy_img2d_color_median(np.nan_to_num(image), segm)
    if 'meanGrad' in feature_flags:
        clean = np.nan_to_num(image)
        grad = np.zeros(clean.shape, dtype=clean.dtype if clean.dtype.kind == 'f' else float)
        for i in range(3):
            grad[:, :, i] = np.sum(np.gradient(clean[:, :, i]), axis=0)
        blocks['meanGrad'] = _device_stats(grad, segm, ('mean', ))
    order = [f for f in NAMES_FEATURE_FLAGS if f in feature_flags]
    nb = int(segm.max()) + 1
    features = np.hstack([blocks[f] for f in order]) if order else np.empty((nb, 0))
    names = list(itertools.chain.from_iterable(['%s_%s' % (n, f) for n in ch_names] for f in order))
    _check_unrecognised_feature_names(feature_flags)
    features = np.nan_to_num(features)
    features[features == 0] = 0
    if features.shape[1] != len(names):
        raise ValueError('features: %r and names %r' % (features.shape, names))
    return features, names


def norm_features(features, scaler=None):
    """ standardise the features (reference descriptors.py:866-877) """
    from sklearn import preprocessing
    if not scaler:
        scaler = preprocessing.StandardScaler()
        scaler.fit(features)
    return scaler.transform(features), scaler


def compute_selected_features_color2d(img, segments, feature_flags=FEATURES_SET_ALL):
    """ features of a colour image selected by the dictionary grammar ``{'color[_<space>]': flags, 'tLM[_short]': flags}``
    (reference descriptors.py:1207-1270)
    """
    img = np.asarray(img)
    _check_color_image(img)
    features, names = [], []
    for k in [k for k in feature_flags if k.startswith('color')]:
        clr = k.split('_')[-1] if '_' in k else 'rgb'
        if '_' in k:
            from .color import convert_img_color_from_rgb
            img_color = convert_img_color_from_rgb(img, clr)
        else:
            img_color = img
        fts, ns = compute_image2d_color_statistic(img_color, segments, feature_flags[k], color_name=clr)
        features.append(fts)
        names += ns
    for k in [k for k in feature_flags if k.startswith('tLM')]:
        bank_type = k.split('_')[-1] if '_' in k else 'normal'
        from .texture import compute_texture_desc_lm_img2d_clr
        fts, ns = compute_texture_desc_lm_img2d_clr(img, segments, feature_flags[k], bank_type)
        features.append(fts)
        names += ns
    _check_unrecognised_feature_group(feature_flags)
    features = np.concatenate(tuple(features), axis=1)
    features = np.nan_to_num(features)
    features[features == 0] = 0
    if not features.size:
        logging.error('not supported features: %r', feature_flags)
    if features.shape[1] != len(names):
        raise ValueError('features: %r and names %r' % (features.shape, names))
    return features, names


def compute_selected_features_gray2d(img, segments, features_flags=FEATURES_SET_ALL):
    """ selected features of a gray 2-D image: the reference treats it as a one-slice volume
    (reference descriptors.py:1167-1204; golden values :1179-1197)

    :return tuple(ndarray,list(str)): features [nb_segments, nb_features], names
    """
    img, segments = np.asarray(img), np.asarray(segments)
    _check_gray_image_segm(img, segments)
    features, names = compute_selected_features_gray3d(img[np.newaxis, ...], segments[np.newaxis, ...], features_flags)
    if features.shape[1] != len(names):
        raise ValueError('features: %r and names %r' % (features.shape, names))
    return features, names


def compute_selected_features_img2d(image, segm, features_flags=FEATURES_SET_COLOR):
    """ dispatch on the image kind (reference descriptors.py:1273-1285) """
    image = np.asarray(image)
    if image.ndim == 3 and image.shape[2] == 3:
        return compute_selected_features_color2d(image, segm, features_flags)
    if image.ndim == 2:
        return compute_selected_features_gray2d(image, segm, features_flags)
    logging.error('invalid image size - %r', image.shape)


def flags_are_native(dict_features):
    """True when every requested feature group / statistic is one the resident device path computes
    ('color', 'tLM', 'tLM_short' with mean / std / energy)"""
    return bool(dict_features) and all(k in ('color', 'tLM', 'tLM_short') and all(f in FLAG_BITS for f in v)
                                       for k, v in dict_features.items())


def native_feature_layout(dict_features):
    """[(key, flags, first column, n columns)] in the reference's column order: colour groups first, then texture"""
    layout, col = [], 0
    for k in [k for k in dict_features if k.startswith('color')] + [k for k in dict_features if k.startswith('tLM')]:
        flags = [f for f in ('mean', 'std', 'energy') if f in dict_features[k]]
        n = 3 * len(flags) * (1 if k == 'color' else (15 if k.endswith('_short') else 20))
        layout.append((k, flags, col, n))
        col += n
    return layout, col


# the Leung-Malik bank lives in texture.py (it shares the device layout code); the reference keeps it in this module
from .texture import (compute_texture_desc_lm_img2d_clr, create_filter_bank_lm_2d, make_edge_filter2d,  # noqa: E402,F401
                      make_gaussian_filter1d)
