"""
Row-band mode: ONE image cut into horizontal bands, one band (or a few) per GPU -- BASELINE config 5 (a single 8192 x 8192
image over 8 GPUs), SURVEY.md section 8(e) "one huge image".

What shards and what does not (reference call stack ``imsegm/pipelines.py:46-110``):

* pixel-sized work is banded: H2D of the band, min-max / blur / rgb2lab, the 10 SLIC sweeps, the colour statistics, the
  final LUT gathers and their D2H.  Per sweep the bands exchange one buffer of 6 int64 words per cluster (the centroids as
  bit patterns; summed as integers, which is an exact merge because every cluster has exactly one owner) -- the one real
  exchange step of the path, an ``all_reduce`` over NCCL.
* superpixel-sized work is replicated: every GPU gets the whole k-means label map (band broadcasts over NVLink), runs the
  connectivity pass, the adjacency extraction, the class model and the alpha-expansion on it.  These are small next to the
  pixel work and identical on every rank, so nothing has to be sent back.

The label map is bit-identical to the single-GPU path (tests/test_gpu_tiled.py): the pixel-centric assignment does not care
how the pixels are partitioned, and the raster-order sequential centroid sums are formed by the one band that owns the
cluster, over a slab that holds every member (checked on the device; an orphan pixel outside the slab makes every rank fall
back to the whole image on its own GPU).

Several bands may live on one GPU (``bands_per_rank``); the merge between them is the same integer sum done by
``isb_combine`` -- that is also how the single-GPU tests exercise every code path of the exchange.
"""
import logging

import numpy as np

from . import _lib
from .engine import dtype_code, flag_bits, get_engine, grown_edge_capacity

OP_SUM_I64, OP_MAX_I64, OP_MIN_F64, OP_MAX_F64, OP_SUM_F64 = 0, 1, 2, 3, 4


class Band(object):
    """rows of one band: owned [own_lo, own_hi), k-means slab [km_lo, km_hi) = owned +- halo, raw slab = k-means slab +-
    blur radius, uploaded rows [up_lo, up_hi) = the raw slab or owned +- ``margin`` (what a descriptor with a wide footprint
    asks for), whichever reaches further (all clipped to the image)"""

    def __init__(self, index, own_lo, own_hi, H, halo, radius, margin=0):
        self.index = index
        self.own_lo, self.own_hi = own_lo, own_hi
        self.km_lo, self.km_hi = max(own_lo - halo, 0), min(own_hi + halo, H)
        self.raw_lo, self.raw_hi = max(self.km_lo - radius, 0), min(self.km_hi + radius, H)
        self.up_lo, self.up_hi = min(self.raw_lo, max(own_lo - margin, 0)), max(self.raw_hi, min(own_hi + margin, H))

    def __repr__(self):
        return 'Band(%d: own %d:%d, slab %d:%d, raw %d:%d)' % (self.index, self.own_lo, self.own_hi, self.km_lo, self.km_hi,
                                                            self.raw_lo, self.raw_hi)


def plan_bands(H, n_bands, halo, radius, margin=0):
    """equal bands of ceil(H / n_bands) rows (the last one takes what is left); every band must own at least one row"""
    rows = -(-int(H) // int(n_bands))
    bands = []
    for b in range(n_bands):
        lo, hi = b * rows, min((b + 1) * rows, H)
        if lo >= hi:
            raise ValueError('an image of %d rows cannot be cut into %d bands of %d rows' % (H, n_bands, rows))
        bands.append(Band(b, lo, hi, H, halo, radius, margin))
    return bands


class LoopbackComm(object):
    """world of one process"""
    rank, world = 0, 1

    def all_reduce(self, t, op):
        pass

    def broadcast(self, t, src):
        pass


class GroupComm(object):
    """torch.distributed process group (NCCL on the GPUs); tensors are reduced in place"""

    def __init__(self, group=None):
        import torch.distributed as dist
        self.dist, self.group = dist, group
        self.rank, self.world = dist.get_rank(group), dist.get_world_size(group)
        self._ops = {'sum': dist.ReduceOp.SUM, 'max': dist.ReduceOp.MAX, 'min': dist.ReduceOp.MIN}

    def all_reduce(self, t, op):
        self.dist.all_reduce(t, op=self._ops[op], group=self.group)

    def broadcast(self, t, src):
        src = src if self.group is None else self.dist.get_global_rank(self.group, src)
        self.dist.broadcast(t, src=src, group=self.group)


def default_comm(group=None):
    import torch.distributed as dist
    if dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
        return GroupComm(group)
    return LoopbackComm()


class TiledSuperpixels(object):
    """device-resident result of :func:`slic_tiled`"""
    shape = bands = local = d_raw = d_seg = d_n_labels = nb_bound = d_feat = d_centres = d_err = None
    fell_back = False


def slic_tiled(image, n_segments, compactness, sigma=1.0, max_iter=10, slic_zero=False, rescale=True, comm=None,
               bands_per_rank=1, eng=None, min_size_factor=0.5, max_size_factor=3, enforce_connectivity=True, defer_check=False,
               force_whole=False, raw_margin=0):
    """ SLIC of one host image over the bands of ``comm`` (every rank passes the same image; it uploads only its rows)

    :param ndarray image: [H, W, C] host array, C in {1, 3}, dtype uint8 / uint16 / float32 / float64
    :return TiledSuperpixels: ``d_seg`` = the whole label map on this GPU (identical on every rank), ``d_raw[i]`` = the raw
        image rows ``bands[local[i]].up_lo:up_hi`` still on the device for the descriptors
    :param bool defer_check: do not synchronise to read the orphan counter ``res.d_err``; the caller reads it with its own
        results and calls again with ``force_whole=True`` when it is not zero
    :param bool force_whole: skip the banded sweeps, every rank runs them on the whole image (the fallback)
    :param int raw_margin: keep at least this many raw rows above and below the owned ones on the device (``d_raw[i]`` then holds
        the rows ``bands[local[i]].up_lo:up_hi``) -- the Leung-Malik descriptor needs its background radius + 16
    """
    eng = eng or get_engine()
    torch = eng.torch
    comm = comm or default_comm()
    image = np.asarray(image)
    if image.ndim == 2:
        image = image[:, :, None]
    H, W, Cn = int(image.shape[0]), int(image.shape[1]), int(image.shape[2])
    code = dtype_code(image.dtype)
    w_half, radius, seeds, ty, tx, step = eng.slic_setup(H, W, n_segments, sigma)
    n_seeds = len(seeds)
    halo = 2 * ty + 1
    n_bands = comm.world * int(bands_per_rank)
    bands = plan_bands(H, n_bands, halo, radius, int(raw_margin))
    local = list(range(comm.rank * bands_per_rank, (comm.rank + 1) * bands_per_rank))
    owner = lambda b: b // bands_per_rank  # noqa: E731

    res = TiledSuperpixels()
    res.shape, res.bands, res.local = (H, W), bands, local
    d_seeds = eng.to_device(seeds, 'seeds')
    mm = eng.buf('tb_minmax', (4,), torch.float64)
    mm_b = eng.buf('tb_minmax_b', (4,), torch.float64)
    wsb = eng.query('slic_kmeans_workspace_bytes', H, W, n_seeds, ty, tx)

    # 1) upload the raw rows, extrema of the owned rows
    res.d_raw = []
    for i, b in enumerate(local):
        bd = bands[b]
        raw = eng.to_device(image[bd.up_lo:bd.up_hi], 'tb%d_raw' % i)
        res.d_raw.append(raw)
        if rescale:
            eng.call('image_minmax', raw[bd.own_lo - bd.up_lo:bd.own_hi - bd.up_lo], code, (bd.own_hi - bd.own_lo) * W * Cn,
                     mm if i == 0 else mm_b)
            if i > 0:
                eng.call('combine', mm, mm_b, 1, OP_MIN_F64)
                eng.call('combine', mm[1:2], mm_b[1:2], 1, OP_MAX_F64)
    if rescale:
        comm.all_reduce(mm[0:1], 'min')
        comm.all_reduce(mm[1:2], 'max')

    # 2) blur + rgb2lab of every raw slab, band descriptors
    descs, keep = [], []
    xchg = [eng.buf('tb%d_xchg' % i, (6 * n_seeds + 1,), torch.int64) for i in range(len(local))]
    mdc = [eng.buf('tb%d_maxdc' % i, (n_seeds,), torch.int64) for i in range(len(local))] if slic_zero else [None] * len(local)
    err = eng.buf('tb_err', (1,), torch.int64)
    err.zero_()
    for i, b in enumerate([] if force_whole else local):
        bd = bands[b]
        hraw = bd.raw_hi - bd.raw_lo
        lab = eng.buf('tb%d_lab' % i, (3, hraw, W), torch.float64)
        eng.call('slic_prepare', res.d_raw[i][bd.raw_lo - bd.up_lo:bd.raw_hi - bd.up_lo], code, hraw, W, Cn, w_half, radius,
                 1.0 / compactness, 2 if rescale else 0, lab, mm)
        slab_rows = bd.km_hi - bd.km_lo
        labels = eng.buf('tb%d_labels' % i, (slab_rows, W), torch.int32)
        ws = eng.buf('tb%d_ws' % i, (wsb,), torch.uint8)
        d = _lib.SlicBand(slab_rows=slab_rows, width=W, image_rows=H, y_off=bd.km_lo, own_lo=bd.own_lo, own_hi=bd.own_hi, halo=halo,
                          n_seeds=n_seeds, step_y=ty, step_x=tx, slic_zero=int(bool(slic_zero)), step=step,
                          lab_slab=lab[:, bd.km_lo - bd.raw_lo:].data_ptr(), plane_stride=hraw * W,
                          seeds_yx=d_seeds.data_ptr(), labels_slab=labels.data_ptr(), ws=ws.data_ptr(), ws_bytes=wsb)
        descs.append(d)
        keep.append((lab, labels, ws))
        eng.call('slic_band_begin', d)

    # 3) the sweeps: assign, sum the owned clusters, merge, take the merged centroids
    for _ in range(0 if force_whole else int(max_iter)):
        for i, d in enumerate(descs):
            eng.call('slic_band_assign', d)
            eng.call('slic_band_update', d, xchg[i])
            if i > 0:
                eng.call('combine', xchg[0], xchg[i], 6 * n_seeds + 1, OP_SUM_I64)
        comm.all_reduce(xchg[0], 'sum')
        eng.call('combine', err, xchg[0][6 * n_seeds:], 1, OP_SUM_I64)
        for i, d in enumerate(descs):
            eng.call('slic_band_import', d, xchg[0], mdc[i])
            if slic_zero and i > 0:
                eng.call('combine', mdc[0], mdc[i], n_seeds, OP_MAX_I64)
        if slic_zero:
            comm.all_reduce(mdc[0], 'max')
        for d in descs:
            eng.call('slic_band_finalize', d, mdc[0])

    # 4) the whole k-means label map on every GPU
    full = eng.buf('tb_full', (H, W), torch.int32)
    res.d_err = err
    if not force_whole:
        for i, b in enumerate(local):
            bd = bands[b]
            full[bd.own_lo:bd.own_hi].copy_(keep[i][1][bd.own_lo - bd.km_lo:bd.own_hi - bd.km_lo])
        if comm.world > 1:
            for bd in bands:
                comm.broadcast(full[bd.own_lo:bd.own_hi], owner(bd.index))
    if force_whole or (not defer_check and int(eng.to_host(err)[0]) != 0):
        # some pixel kept the label of a cluster centred beyond the halo (no window covers it -- only degenerate inputs do
        # that): the banded sums are not trustworthy, every rank redoes the sweeps on the whole image on its own GPU
        logging.warning('slic_tiled: orphan pixels beyond the halo, redoing the sweeps on the whole image on every GPU')
        res.fell_back = True
        d_img = eng.to_device(image if Cn == 3 else image[:, :, 0], 'image')
        km, _ = eng.slic(d_img, n_segments, compactness, sigma=sigma, max_iter=max_iter, enforce_connectivity=False,
                         slic_zero=slic_zero, rescale=rescale)
        full.copy_(km)
    if not enforce_connectivity:
        res.d_seg = full
        return res
    res.d_seg, res.d_n_labels = eng.connectivity(full, n_segments, min_size_factor, max_size_factor)
    res.nb_bound = eng.slic_label_bound(H, W, n_segments, min_size_factor)
    return res


def color_stats_tiled(res, image_dtype, channels, flags, comm=None, eng=None, feat=None, col0=0):
    """colour statistics + centroids of the banded image over ``res.d_seg``: every band accumulates its owned rows, the
    accumulators are summed over the GPUs, every GPU finishes the same [nb, 3*len(flags)] table"""
    eng = eng or get_engine()
    torch = eng.torch
    comm = comm or default_comm()
    W = res.shape[1]
    if channels != 3:
        raise ValueError('the colour statistics need a 3-channel image')
    code = dtype_code(image_dtype)
    nb = int(res.nb_bound)
    bits, n = flag_bits(flags)
    acc = eng.buf('tb_acc', (nb, 6), torch.float64)
    iacc = eng.buf('tb_iacc', (nb, 3), torch.int64)
    acc.zero_()
    iacc.zero_()

    def rows(i, b):
        bd = res.bands[b]
        return bd, res.d_raw[i][bd.own_lo - bd.up_lo:bd.own_hi - bd.up_lo], res.d_seg[bd.own_lo:bd.own_hi]

    for i, b in enumerate(res.local):
        bd, img, seg = rows(i, b)
        eng.call('segment_stats_accumulate', img, code, seg, bd.own_hi - bd.own_lo, W, bd.own_lo, nb, acc, iacc)
    comm.all_reduce(acc, 'sum')
    comm.all_reduce(iacc, 'sum')
    var = None
    if bits & 2:
        var = eng.buf('tb_var', (nb, 3), torch.float64)
        meanf = eng.buf('tb_meanf', (nb, 3), torch.float32)
        var.zero_()
        for i, b in enumerate(res.local):
            bd, img, seg = rows(i, b)
            eng.call('segment_stats_deviation', img, code, seg, bd.own_hi - bd.own_lo, W, nb, acc, iacc, meanf, var)
        comm.all_reduce(var, 'sum')
    if feat is None:
        feat = eng.buf('feat', (nb, max(3 * n, 1)), torch.float64)
    centres = eng.buf('centres', (nb, 2), torch.float64)
    eng.call('segment_stats_finish', nb, bits, acc, var, iacc, feat, int(feat.shape[1]), int(col0), centres, None)
    res.d_feat, res.d_centres = feat, centres
    return feat, centres


LM_ROW_MARGIN = 616     # rows of the Leung-Malik descriptor's footprint: sigma-150 background (radius 600) + half a 33 x 33 kernel


def texture_stats_tiled(res, image_dtype, flags, bank_type='normal', comm=None, eng=None, feat=None, col0=0):
    """Leung-Malik texture statistics (reference descriptors.py:1041-1106) of the banded image over ``res.d_seg``: every band runs
    the background subtraction and the filter-bank contraction on its rows + ``LM_ROW_MARGIN`` rows of halo (``slic_tiled`` must
    have been called with ``raw_margin=LM_ROW_MARGIN``) and accumulates the sums of the rows it owns; the accumulators -- the
    per-superpixel sums and the per-battery response norms of the WHOLE image -- are summed over the GPUs, every GPU finishes
    the same [nb, n_batteries * 3 * len(flags)] block of ``feat``"""
    from .texture import lm_setup
    eng = eng or get_engine()
    torch = eng.torch
    comm = comm or default_comm()
    H, W = res.shape
    code = dtype_code(image_dtype)
    nb = int(res.nb_bound)
    _, d_w, NP, orient, n_batt, w_bg, radius, mix, bits, ncol = lm_setup(eng, bank_type, flags)
    d_wbg = eng.const_device(w_bg, 'lm_bg_w')
    acc = eng.buf('tb_lm_acc', (int(eng.query('lm_acc_doubles', nb, n_batt)),), torch.float64)
    counts = eng.buf('tb_lm_counts', (nb,), torch.int32)
    acc.zero_()
    counts.zero_()
    for i, b in enumerate(res.local):
        bd = res.bands[b]
        lo, hi = max(bd.own_lo - LM_ROW_MARGIN, 0), min(bd.own_hi + LM_ROW_MARGIN, H)
        if lo < bd.up_lo or hi > bd.up_hi:
            raise ValueError('the band keeps the raw rows %d:%d, the texture descriptor needs %d:%d (slic_tiled raw_margin)'
                             % (bd.up_lo, bd.up_hi, lo, hi))
        ws, wsb = eng.workspace('ws_lm', 'lm_workspace_bytes', hi - lo, W, nb, n_batt)
        eng.call('lm_texture_accumulate', res.d_raw[i][lo - bd.up_lo:hi - bd.up_lo], code, res.d_seg[lo:hi], hi - lo, W, bd.own_lo - lo,
                 bd.own_hi - lo, nb, d_wbg, radius, mix, d_w, NP, orient, n_batt, acc, counts, ws, wsb)
    comm.all_reduce(acc, 'sum')
    comm.all_reduce(counts, 'sum')
    if feat is None:
        feat = eng.buf('feat_lm', (nb, ncol), torch.float64)
    eng.call('lm_texture_finish', nb, n_batt, bits, acc, counts, feat, int(feat.shape[1]), int(col0))
    return feat


def features_tiled(res, image_dtype, channels, layout, ncol, comm=None, eng=None):
    """the [nb, ncol] feature table of ``native_feature_layout`` over the banded image (``res.d_feat``) + the centroids"""
    eng = eng or get_engine()
    feat = eng.buf('feat', (int(res.nb_bound), max(ncol, 1)), eng.torch.float64)
    centres = None
    for key, flags, col0, _ in layout:
        if key == 'color':
            _, centres = color_stats_tiled(res, image_dtype, channels, flags, comm=comm, eng=eng, feat=feat, col0=col0)
        else:
            texture_stats_tiled(res, image_dtype, flags, 'short' if key.endswith('_short') else 'normal', comm=comm, eng=eng, feat=feat,
                                col0=col0)
    if centres is None:
        _, centres = color_stats_tiled(res, image_dtype, channels, (), comm=comm, eng=eng, feat=eng.buf('feat_none', (int(res.nb_bound), 1),
                                                                                                         eng.torch.float64))
    res.d_feat, res.d_centres = feat, centres
    return feat, centres


def pipe_color2d_slic_features_model_graphcut_tiled(image, nb_classes, dict_features=None, sp_size=30, sp_regul=0.2, use_scaler=True,
                                                    gc_regul=1., gc_edge_type='model', max_iter=99, comm=None, bands_per_rank=1,
                                                    want_soft=True, gather_segm=False):
    """ ``pipe_color2d_slic_features_model_graphcut`` (reference pipelines.py:46-110) for one image banded over the GPUs of
    ``comm``.  Every rank passes the same host image and gets the rows it owns:

    :return tuple: (segm [rows, W] int32, segm_soft [rows, W, K] float64 or None, (row_lo, row_hi)); with ``gather_segm``
        ``segm`` is the whole [H, W] map on every rank (``segm_soft`` stays banded: it is 8*K bytes per pixel)
    """
    return _banded_pipeline(image, ('fit', nb_classes, use_scaler, max_iter), dict_features, sp_size, sp_regul, gc_regul,
                            gc_edge_type, comm, bands_per_rank, want_soft, gather_segm)


def segment_color2d_slic_features_model_graphcut_tiled(image, model, dict_features=None, sp_size=30, sp_regul=0.2, gc_regul=1.,
                                                       gc_edge_type='model', comm=None, bands_per_rank=1, want_soft=True,
                                                       gather_segm=False):
    """ ``segment_color2d_slic_features_model_graphcut`` (reference pipelines.py:160-241) -- a model fitted beforehand, e.g. by
    ``estim_model_classes_group`` on other images -- for one image banded over the GPUs of ``comm``, as
    :func:`pipe_color2d_slic_features_model_graphcut_tiled`.  The class probabilities are evaluated on the device.

    :param model: a :class:`graph_cuts.DeviceClassModel`, or a fitted mixture model it can wrap (wrapped on entry)
    :return tuple: (segm [rows, W], segm_soft [rows, W, K] float64 or None, (row_lo, row_hi)); ``segm`` maps through the
        model's ``classes_`` when it has them
    """
    from .graph_cuts import DeviceClassModel
    model = model if isinstance(model, DeviceClassModel) else DeviceClassModel(model)
    segm, soft, rows = _banded_pipeline(image, model, dict_features, sp_size, sp_regul, gc_regul, gc_edge_type, comm, bands_per_rank,
                                        want_soft, gather_segm)
    classes = getattr(model, 'classes_', None)
    return (segm if classes is None else np.asarray(classes)[segm]), soft, rows


def _banded_pipeline(image, model, dict_features, sp_size, sp_regul, gc_regul, gc_edge_type, comm, bands_per_rank, want_soft,
                     gather_segm):
    """the banded pipeline; ``model`` is ('fit', nb_classes, use_scaler, max_iter) -- the default GMM fitted on the device -- or a
    DeviceClassModel evaluated on the device"""
    from . import graph_cuts
    from .descriptors import flags_are_native, native_feature_layout
    from .pipelines import _check_model_width, _device_graphcut, _soft_on_side_stream
    from .superpixels import _as_rgb_like, _supported_dtype, slic_params
    if sp_regul <= 0.:
        raise ValueError('slic. regularisation must be positive')
    dict_features = {'color': ['mean']} if dict_features is None else dict_features
    layout, ncol = native_feature_layout(dict_features)
    if not layout or not flags_are_native(dict_features):
        raise NotImplementedError('the banded path computes mean / std / energy of the colours and of the Leung-Malik responses (got %r)'
                                  % dict_features)
    margin = LM_ROW_MARGIN if any(k.startswith('tLM') for k, _, _, _ in layout) else 0
    eng = get_engine()
    comm = comm or default_comm()
    image = _supported_dtype(_as_rgb_like(np.asarray(image)))
    H, W = int(image.shape[0]), int(image.shape[1])
    n_seg, compact = slic_params((H, W), sp_size, sp_regul)
    if n_seg < 1:
        raise ValueError('superpixel size %r is larger than the image %r' % (sp_size, tuple(image.shape)))
    if isinstance(model, graph_cuts.DeviceClassModel):
        _check_model_width(model, dict_features)
        d_model = model.device_params(eng)

        def class_proba(res):
            return eng.gmm_predict(res.d_feat, d_model, model.n_classes, d_n=res.d_n_labels)
    else:
        _, K, use_scaler, max_iter = model
        K = int(K)
        n_init = max(1, int(np.sqrt(max_iter)))

        def class_proba(res):
            return eng.gmm_fit_predict(res.d_feat, K, n_init, max_iter, use_scaler, graph_cuts.RANDOM_SEED, d_n=res.d_n_labels)[0]
    force_whole, redo_front, cap = False, True, None
    while True:
        if redo_front:
            res = slic_tiled(image, n_seg, compact, sigma=1.0, comm=comm, bands_per_rank=bands_per_rank, eng=eng, defer_check=True,
                             force_whole=force_whole, raw_margin=margin)
            features_tiled(res, image.dtype, int(image.shape[2]), layout, ncol, comm=comm, eng=eng)
            nb = int(res.nb_bound)
            d_proba = class_proba(res)          # the model fitted on this image, or the given one evaluated
            redo_front = False
        lo, hi = res.bands[res.local[0]].own_lo, res.bands[res.local[-1]].own_hi
        h_soft = soft_done = None
        if want_soft:
            h_soft, soft_done = _soft_on_side_stream(eng, res.d_seg[lo:hi], d_proba)
        # 5) graph cut, LUT gather of the owned rows
        _, d_segm, _, d_n_edges, cap = _device_graphcut(eng, res, nb, d_proba, gc_regul, gc_edge_type, d_n_nodes=res.d_n_labels,
                                                        want_soft=False, edge_cap=cap, rows=(lo, hi), whole_segm=gather_segm)
        d_full = eng.buf('segm', (H, W), eng.torch.int32) if gather_segm else None
        if gather_segm and comm.world > 1:
            for r in range(comm.world):
                blo = res.bands[r * bands_per_rank].own_lo
                bhi = res.bands[(r + 1) * bands_per_rank - 1].own_hi
                comm.broadcast(d_full[blo:bhi], r)
        (h_segm, h_n_edges, h_err), done = eng.download([d_segm if d_full is None else d_full, d_n_edges, res.d_err])
        done.synchronize()
        if soft_done is not None:
            soft_done.synchronize()
        if int(h_err[0]) != 0 and not force_whole:
            # orphan pixels beyond the halo (see slic_tiled): same answer on every rank, so every rank takes this branch
            logging.warning('banded SLIC met orphan pixels beyond the halo, redoing the sweeps on the whole image on every GPU')
            force_whole = redo_front = True
            continue
        if int(h_n_edges[0]) <= cap:
            break
        cap = grown_edge_capacity(cap)
    return h_segm.numpy(), (h_soft.numpy() if want_soft else None), (lo, hi)
