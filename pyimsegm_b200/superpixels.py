"""
Superpixels: SLIC on the GPU and the superpixel adjacency graph.

Mirror of the reference module ``imsegm/superpixels.py`` (same public names, argument meaning and return
types); the work is done by the CUDA kernels behind ``include/imsegm_b200.h``:

* :func:`segment_slic_img2d`  -> ``isb_slic_prepare`` / ``isb_slic_kmeans`` / ``isb_enforce_connectivity``
  (replaces ``skimage.segmentation.slic``, reference ``imsegm/superpixels.py:22-69``)
* :func:`make_graph_segm_connect_grid2d_conn4` -> ``isb_adjacency_edges`` (reference ``:115-177``)
* :func:`superpixel_centers` -> ``isb_segment_stats_2d`` centroids (reference ``:205-242``)
"""
import logging

import numpy as np

from .engine import get_engine, grown_edge_capacity

#: spacing among neighboring pixels in axes X, Y, Z  (reference superpixels.py:19)
IMAGE_SPACING = (1, 1, 1)


def _as_rgb_like(img):
    img = np.asarray(img)
    if img.ndim == 2:
        # gray is processed as three equal channels (reference superpixels.py:50-51); the kernel replicates C=1
        return img
    if img.ndim != 3 or img.shape[2] != 3:
        raise ValueError('expected a 2-D gray or [H, W, 3] colour image, got shape %r' % (img.shape, ))
    return img


def _supported_dtype(img):
    if img.dtype in (np.uint8, np.uint16, np.float32, np.float64):
        return img
    if np.issubdtype(img.dtype, np.integer) or img.dtype == bool:
        return img.astype(np.float64)
    return img.astype(np.float64)


def slic_params(shape_hw, sp_size, relative_compact):
    """native SLIC parameters from the reference's (size, regularisation) pair (superpixels.py:57-58)"""
    nb_pixels = int(np.prod(shape_hw))
    return int(nb_pixels / (sp_size ** 2)), (sp_size * relative_compact) ** 1.5


def segment_slic_img2d(img, sp_size=50, relative_compact=0.1, slico=False):
    """ SLIC superpixels of a 2-D colour (or gray) image, computed on the GPU

    :param ndarray img: input image [H, W, 3] or [H, W]
    :param int sp_size: superpixel initial size
    :param float relative_compact: relative regularisation in range (0, 1)
    :param bool slico: parameter-free SLICO / ASLIC variant (skimage's slic_zero)
    :return ndarray: segmentation [H, W], labels 0..N-1
    """
    img = _supported_dtype(_as_rgb_like(img))
    eng = get_engine()
    n_seg, compact = slic_params(img.shape[:2], sp_size, relative_compact)
    logging.debug('SLIC 2d: NB=%i compact=%f image %r', n_seg, compact, img.shape)
    if n_seg < 1:
        raise ValueError('superpixel size %r is larger than the image %r' % (sp_size, img.shape))
    d_img = eng.to_device(img, 'image')
    labels, _ = eng.slic(d_img, n_seg, compact, sigma=1.0, enforce_connectivity=True, slic_zero=slico)
    return eng.to_host(labels).astype(np.int64)


def segment_slic_img3d_gray(im, sp_size=50, relative_compact=0.1, space=IMAGE_SPACING):
    """ SLIC superpixels of a gray volume with anisotropic voxel spacing, computed on the GPU (reference superpixels.py:72-112)

    :param ndarray im: input volume [D, H, W]
    :param int sp_size: superpixel initial size
    :param float relative_compact: relative regularisation in range (0, 1)
    :param tuple(int,int,int) space: voxel spacing (z, y, x)
    :return ndarray: labels [D, H, W], int64

    The reference closes with ``skimage.measure.label`` (:111): with full connectivity and background 0 it renumbers the labels in
    the order of their first voxel and leaves label 0 alone -- the order the connectivity pass has already produced, so the map
    is returned as it is (oracle/__init__.py ``segment_slic_img3d_gray``, tests/test_oracle_goldens.py).
    """
    im = np.asarray(im)
    if im.ndim != 3:
        raise ValueError('expected a gray volume [D, H, W], got shape %r' % (im.shape, ))
    nb_pixels = np.prod(im.shape)
    size = np.prod(sp_size / np.asarray(space, dtype=np.float32) * min(space))
    n_seg = int(nb_pixels / size)
    compact = int((size * relative_compact) ** 1.5)
    logging.debug('SLIC 3d gray: NB=%i compact=%f spacing=%r volume %r', n_seg, compact, space, im.shape)
    if n_seg < 1 or compact < 1:
        raise ValueError('superpixel size %r / compactness do not fit the volume %r' % (sp_size, im.shape))
    eng = get_engine()
    d_vol = eng.to_device(_supported_dtype(im), 'volume')
    labels, _ = eng.slic3d(d_vol, n_seg, compact, space, sigma=1.0)
    return eng.to_host(labels).astype(np.int64)


def make_graph_segment_connect_edges(vertices, all_edges):
    """ unique undirected edges from a list of label pairs (reference superpixels.py:115-131)

    :param ndarray vertices: unique labels (sorted)
    :param ndarray all_edges: [M, 2] pairs of vertex INDEXES
    :return tuple(ndarray,list): vertices, [[a, b], ...] with a < b sorted by (b, a)
    """
    vertices = np.asarray(vertices)
    pairs = np.asarray(all_edges)
    pairs = pairs[pairs[:, 0] != pairs[:, 1]]
    lo, hi = pairs.min(axis=1), pairs.max(axis=1)
    n = len(vertices)
    codes = np.unique(lo.astype(np.int64) + n * hi.astype(np.int64))
    edges = [[vertices[int(c % n)], vertices[int(c // n)]] for c in codes]
    return vertices, edges


def get_segment_diffs_2d_conn4(grid):
    """ all horizontally / vertically adjacent label pairs (reference superpixels.py:134-142) """
    grid = np.asarray(grid)
    right = np.stack([grid[:, :-1].ravel(), grid[:, 1:].ravel()], axis=1)
    down = np.stack([grid[:-1, :].ravel(), grid[1:, :].ravel()], axis=1)
    return np.vstack([right, down])


def get_segment_diffs_3d_conn6(grid):
    """ 6-connected label pairs of a volume (reference superpixels.py:145-154) """
    grid = np.asarray(grid)
    below = np.stack([grid[:-1].ravel(), grid[1:].ravel()], axis=1)
    down = np.stack([grid[:, :-1].ravel(), grid[:, 1:].ravel()], axis=1)
    right = np.stack([grid[:, :, :-1].ravel(), grid[:, :, 1:].ravel()], axis=1)
    return np.vstack([below, right, down])


def device_adjacency(eng, d_seg, nb):
    """(device edges [cap, 2] int32, E) of a device label map or volume with labels in [0, nb); grows the table on overflow"""
    cap = None
    while True:
        edges, n_edges, cap = eng.adjacency(d_seg, nb, cap)
        E = int(eng.to_host(n_edges)[0])
        if E <= cap:
            return edges, E
        cap = grown_edge_capacity(cap)


def make_graph_segm_connect_grid2d_conn4(grid):
    """ region adjacency graph of a 2-D segmentation, 4-connectivity (reference superpixels.py:157-177)

    :param ndarray grid: segmentation
    :return tuple(ndarray,list): unique labels, list of [a, b] edges (a < b, ordered by b then a)

    >>> # doctest values of the reference: grid [[0]*5+[1]*5, [2]*5+[3]*5] -> [[0, 1], [0, 2], [1, 3], [2, 3]]
    """
    grid = np.asarray(grid)
    if grid.ndim != 2:
        raise ValueError('2-D segmentation expected, got %r' % (grid.shape, ))
    vertices, inverse = np.unique(grid, return_inverse=True)
    compact = inverse.reshape(grid.shape).astype(np.int32)
    eng = get_engine()
    d_seg = eng.to_device(compact, 'seg_in')
    d_edges, E = device_adjacency(eng, d_seg, len(vertices))
    pairs = eng.to_host(d_edges[:E]) if E else np.zeros((0, 2), dtype=np.int32)
    edges = [[vertices[a], vertices[b]] for a, b in pairs.tolist()]
    return vertices, edges


def make_graph_segm_connect_grid3d_conn6(grid):
    """ region adjacency graph of a 3-D segmentation (reference superpixels.py:180-202); host implementation,
    the 3-D path is not part of the accelerated hot path """
    grid = np.asarray(grid)
    vertices, inverse = np.unique(grid, return_inverse=True)
    return make_graph_segment_connect_edges(vertices, get_segment_diffs_3d_conn6(inverse.reshape(grid.shape)))


def superpixel_centers(segments):
    """ centre (mean row, mean column) of every label 0..max (reference superpixels.py:205-242)

    :param ndarray segments: segmentation [H, W]
    :return list(tuple(float,float)): centres; labels that do not occur give [-1, -1]
    """
    segments = np.asarray(segments)
    if segments.ndim == 3:
        nb = int(segments.max()) + 1
        centres = [[-1] * 3 for _ in range(nb)]
        idx = np.indices(segments.shape).reshape(3, -1)
        flat = segments.ravel()
        cnt = np.bincount(flat, minlength=nb)
        for lb in np.nonzero(cnt)[0]:
            centres[lb] = [float(np.bincount(flat, weights=idx[d], minlength=nb)[lb] / cnt[lb]) for d in range(3)]
        return centres
    if segments.ndim != 2:
        logging.error('not supported image dim: %r', segments.shape)
        return [[-1] * segments.ndim for _ in range(int(np.max(segments)) + 1)]
    eng = get_engine()
    nb = int(segments.max()) + 1
    d_seg = eng.to_device(segments.astype(np.int32), 'seg_in')
    _, centres, counts = eng.segment_stats(None, d_seg, nb, (), want_centres=True, want_counts=True)
    cen = eng.to_host(centres)
    cnt = eng.to_host(counts)
    return [(float(r), float(c)) if n > 0 else [-1, -1] for (r, c), n in zip(cen.tolist(), cnt.tolist())]


def get_neighboring_segments(edges):
    """ neighbour lists per vertex from an edge list (reference superpixels.py:245-259) """
    edges = np.asarray(edges)
    neighbours = [[] for _ in range(int(edges.max()) + 1)]
    for a, b in edges.tolist():
        neighbours[a].append(b)
        neighbours[b].append(a)
    return neighbours
