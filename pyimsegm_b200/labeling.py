"""
Labelling helpers on the superpixel level (the part of the reference's ``imsegm/labeling.py`` that the supervised
pipeline calls per image: ``wrapper_compute_color2d_slic_features_labels``, reference pipelines.py:272-290).
"""
import numpy as np

from .engine import get_engine
from .utilities import ImageDimensionError


def histogram_regions_labels_counts(slic, segm):
    """ overlap counts between superpixels and an annotation: ``hist[a, b]`` = pixels with superpixel ``a`` and label ``b``
    (reference labeling.py:206-240, a per-pixel Python loop there)

    :param ndarray slic: superpixel map
    :param ndarray segm: annotation, non-negative labels
    :return ndarray: float matrix [slic.max() + 1, segm.max() + 1]
    """
    slic, segm = np.asarray(slic), np.asarray(segm)
    if slic.shape != segm.shape:
        raise ImageDimensionError('dimension does not agree')
    if segm.min() < 0:
        raise ValueError('only positive labels are allowed')
    if slic.ndim != 2:
        slic, segm = slic.reshape(1, -1), segm.reshape(1, -1)
    eng = get_engine()
    nb_a, nb_b = int(slic.max()) + 1, int(segm.max()) + 1
    d_a = eng.to_device(slic.astype(np.int32, copy=False), 'hist_slic')
    d_b = eng.to_device(segm.astype(np.int32, copy=False), 'hist_annot')
    hist = eng.buf('hist_joint', (nb_a, nb_b), eng.torch.int32)
    eng.call('region_label_hist', d_a, d_b, slic.shape[0], slic.shape[1], nb_a, nb_b, hist)
    return eng.to_host(hist).astype(float)


def histogram_regions_labels_norm(slic, segm):
    """ relative overlap of every superpixel with the annotation labels, rows sum to 1 (reference labeling.py:243-283) """
    slic, segm = np.asarray(slic), np.asarray(segm)
    if slic.shape != segm.shape:
        raise ImageDimensionError('dimension of SLIC %r and segm %r should match' % (slic.shape, segm.shape))
    if segm.min() < 0:
        raise ValueError('only positive labels are allowed')
    hist = histogram_regions_labels_counts(slic, segm)
    sums = hist.sum(axis=1, keepdims=True)
    sums[sums == 0] = -1.
    hist = np.nan_to_num(hist / sums)
    hist[hist == 0] = 0
    return hist
