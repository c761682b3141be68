"""
Segmentation pipelines: SLIC -> per-superpixel features -> class model -> GraphCut, resident on the GPU.

Mirror of the reference module ``imsegm/pipelines.py`` for the unsupervised hot path (same names, arguments
and return values):

* :func:`pipe_color2d_slic_features_model_graphcut`     (reference pipelines.py:46-110)
* :func:`estim_model_classes_group`                     (reference pipelines.py:113-157)
* :func:`segment_color2d_slic_features_model_graphcut`  (reference pipelines.py:160-241)
* :func:`compute_color2d_superpixels_features`          (reference pipelines.py:244-270)

The image goes to the device once; label map, features, class model, graph, energies and the cut never leave it and the
host synchronises ONCE, when the results are downloaded.  (A user-supplied model, or one the device GMM does not cover, costs
one round trip: features [N, D] down, probabilities [N, K] up -- unless it is wrapped in ``graph_cuts.DeviceClassModel``, whose
probabilities are computed on the device.)
"""
import logging

import numpy as np

from .descriptors import FEATURES_SET_COLOR, compute_selected_features_img2d, flags_are_native, native_feature_layout
from .engine import edge_capacity, get_engine, grown_edge_capacity
from .graph_cuts import (DeviceClassModel, _edge_mode, compute_pairwise_cost, device_gmm_applicable, estim_class_model,
                         segment_graph_cut_general)
from .superpixels import _as_rgb_like, _supported_dtype, slic_params

#: basic features extracted from superpixels (reference pipelines.py:35)
FTS_SET_SIMPLE = FEATURES_SET_COLOR
#: default clustering for unsupervised segmentation (reference pipelines.py:39 -> classification.DEFAULT_CLUSTERING)
#: default classifier of the supervised path (reference classification.py:54; the classifier zoo itself is out of scope)
CLASSIF_NAME = 'RandForest'
CLUSTER_METHOD = 'kMeans'
#: images left out during cross-validation training (reference pipelines.py:41)
CROSS_VAL_LEAVE_OUT = 2
#: default number of workers of the reference's process pool (pipelines.py:43); the GPU path shards images over
#: devices instead, the value is kept for signature compatibility
NB_WORKERS = 1


class DeviceSuperpixels(object):
    """device-resident result of SLIC + descriptors for one image"""
    __slots__ = ('d_img', 'd_seg', 'd_n_labels', 'nb_bound', 'd_feat', 'd_centres', 'shape', 'd_params', 'd_n_edges', 'edge_cap')


def _device_slic_features(eng, image, dict_features, sp_size, sp_regul):
    """H2D, SLIC, fused colour statistics + centroids; everything stays on the device"""
    if sp_regul <= 0.:
        raise ValueError('slic. regularisation must be positive')
    on_device = hasattr(image, 'is_cuda')
    if not on_device:
        image = _supported_dtype(_as_rgb_like(image))
    H, W = int(image.shape[0]), int(image.shape[1])
    n_seg, compact = slic_params((H, W), sp_size, sp_regul)
    if n_seg < 1:
        raise ValueError('superpixel size %r is larger than the image %r' % (sp_size, tuple(image.shape)))
    res = DeviceSuperpixels()
    res.shape = (H, W)
    res.d_img = image if on_device else eng.to_device(image, 'image')
    res.d_seg, res.d_n_labels = eng.slic(res.d_img, n_seg, compact, sigma=1.0)
    res.nb_bound = eng.slic_label_bound(H, W, n_seg)
    layout, ncol = native_feature_layout(dict_features)
    res.d_feat = eng.buf('feat', (res.nb_bound, max(ncol, 1)), eng.torch.float64)
    res.d_centres = None
    for key, flags, col0, _ in layout:
        if key == 'color':
            _, res.d_centres, _ = eng.segment_stats(res.d_img, res.d_seg, res.nb_bound, flags, feat=res.d_feat, col0=col0,
                                                    want_centres=True)
        else:
            from .texture import device_lm_features
            device_lm_features(eng, res.d_img, res.d_seg, res.nb_bound, flags, 'short' if key.endswith('_short') else 'normal',
                               feat=res.d_feat, col0=col0)
    if res.d_centres is None:
        _, res.d_centres, _ = eng.segment_stats(None, res.d_seg, res.nb_bound, (), want_centres=True)
    return res


def compute_color2d_superpixels_features(image, dict_features, sp_size=30, sp_regul=0.2):
    """ segment the image into superpixels and estimate features per superpixel (reference pipelines.py:244-270)

    :return tuple(ndarray,ndarray): superpixel map [H, W], features [N, D]
    """
    if sp_regul <= 0.:
        raise ValueError('slic. regularisation must be positive')
    image = np.asarray(image)
    eng = get_engine()
    if image.ndim == 3 and flags_are_native(dict_features):
        res = _device_slic_features(eng, image, dict_features, sp_size, sp_regul)
        nb = int(eng.to_host(res.d_n_labels)[0])
        slic = eng.to_host(res.d_seg).astype(np.int64)
        features = eng.to_host(res.d_feat[:nb]).copy()
    else:
        if sp_regul <= 0.:
            raise ValueError('slic. regularisation must be positive')
        from .superpixels import segment_slic_img2d
        slic = segment_slic_img2d(image, sp_size=sp_size, relative_compact=sp_regul)
        features, _ = compute_selected_features_img2d(image, slic, dict_features)
    features[np.isnan(features)] = 0
    return slic, features


def _device_graphcut(eng, res, nb, d_proba, gc_regul, gc_edge_type, d_n_nodes=None, want_soft=True, edge_cap=None, rows=None,
                     whole_segm=False):
    """device tail of the pipeline: adjacency, energies, alpha-expansion, LUT gathers (all asynchronous).
    ``nb`` (= the rows of ``d_proba``) may be an upper bound of the label count when ``d_n_nodes`` (device scalar) carries the real
    one.  ``rows`` = (lo, hi): gather only these rows of the label map, into rows lo:hi of a whole-image 'segm' when ``whole_segm``.
    Returns (d_labels, d_segm, d_soft, d_n_edges, edge_cap)."""
    pairwise = compute_pairwise_cost(gc_regul, d_proba.shape)
    d_edges, d_n_edges, edge_cap = eng.adjacency(res.d_seg, nb, edge_cap)
    d_labels, _, _ = eng.graph_cut(d_proba, d_edges, edge_cap, d_n_edges, res.d_centres, _edge_mode(gc_edge_type), 1.0, pairwise,
                                   d_n_nodes=d_n_nodes)
    d_seg = res.d_seg if rows is None else res.d_seg[rows[0]:rows[1]]
    out_segm = eng.buf('segm', res.d_seg.shape, eng.torch.int32)[rows[0]:rows[1]] if whole_segm else None
    d_segm, d_soft = eng.gather(d_seg, d_labels, d_proba if want_soft else None, out_i=out_segm)
    return d_labels, d_segm, d_soft, d_n_edges, edge_cap


def _soft_on_side_stream(eng, d_seg, d_proba):
    """segm_soft = proba[d_seg] needs only the class probabilities: its gather and its (large) download run on the engine's side
    stream while the main stream builds and cuts the graph.  Returns (pinned host tensor, event of the download)."""
    torch = eng.torch
    side = eng.side_stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        _, d_soft = eng.gather(d_seg, None, d_proba)
        (host, ), event = eng.download([d_soft])
    return host, event


def _argmin_labels_device(eng, proba):
    graph_labels = np.argmin(np.abs(-np.log(np.clip(proba, 0.01, 0.99))), axis=-1).astype(np.int32)
    return eng.to_device(graph_labels, 'gc_labels_in')


#: start the download of segm_soft (it only needs the class probabilities) on a side stream while the graph is cut
EARLY_SOFT_DOWNLOAD = True

#: replay the device part of the path as CUDA graphs once a configuration has been seen twice (the ~70 kernel launches of an image
#: cost more host time than the GPU needs for them when images are processed back to back, and the gaps between them add up)
USE_CUDA_GRAPHS = True
_GRAPHS = {}


def _graph_call(eng, key, fn):
    """``fn()`` -- a sequence of C-ABI launches that never touches the host and writes into the engine's cached buffers -- run
    eagerly the first time ``key`` is seen (this also sizes every buffer), captured as a CUDA graph the second time, replayed
    afterwards.  Returns what ``fn`` returned (device tensors that every replay refills)."""
    if not USE_CUDA_GRAPHS:
        return fn()
    entry = _GRAPHS.get(key)
    if entry is None:
        _GRAPHS[key] = 'seen'
        return fn()
    torch = eng.torch
    if entry == 'seen':
        graph = torch.cuda.CUDAGraph()
        n0 = eng.query('launch_count')
        cur = torch.cuda.current_stream()
        side = torch.cuda.Stream(device=eng.device)
        side.wait_stream(cur)
        with torch.cuda.graph(graph, stream=side):
            out = fn()
        cur.wait_stream(side)
        eng.graphs_captured = getattr(eng, 'graphs_captured', 0) + 1      # from now on the engine never frees a buffer it outgrows
        entry = _GRAPHS[key] = (graph, out, int(eng.query('launch_count') - n0))
    graph, out, n_kernels = entry
    graph.replay()
    eng.query('note_graph_replay', n_kernels)
    return out


def _features_key(dict_features):
    return tuple(sorted((k, tuple(v)) for k, v in dict_features.items()))


def _check_model_width(model, dict_features):
    """ValueError when a DeviceClassModel was fitted on another number of features than ``dict_features`` gives"""
    ncol = native_feature_layout(dict_features)[1]
    if ncol != model.n_features:
        raise ValueError('the class model takes %d features, %r gives %d' % (model.n_features, dict_features, ncol))


def _run_resident(eng, image, model, dict_features, sp_size, sp_regul, gc_regul, gc_edge_type, soft_sink=None, edge_cap=None):
    """the whole hot path on the device.  ``model`` is either ('fit', nb_classes, use_scaler, max_iter) -> the default
    GMM is fitted on the GPU and NOTHING syncs with the host until the results are ready; or a :class:`DeviceClassModel` -> its
    probabilities are evaluated on the GPU (isb_gmm_predict), again without a synchronisation; or a callable
    proba_fn(features) -> one round trip (features down, probabilities up) as in the reference.
    ``soft_sink(d_seg, d_proba)``: the caller takes ``segm_soft = proba[slic]`` itself as soon as the probabilities exist
    (it does not depend on the graph cut) -- then ``d_soft`` is returned as None.
    With a device model and colour features the two halves -- image -> class probabilities, probabilities -> cut and LUT
    gathers -- are CUDA-graph replays (:func:`_graph_call`); the image then has to sit in one of the engine's cached buffers.
    (The large-D fit synchronises once per EM iteration, so a fitted model is only captured up to 16 features; the prediction
    never synchronises and is captured at any width.)
    ``edge_cap``: capacity of the edge table (default :func:`engine.edge_capacity` of the superpixel count).
    Returns (d_segm, d_soft, check): ``check`` is None or (d_n_edges, edge_cap) still to be verified by the caller."""
    no_cut = (not isinstance(gc_regul, (list, np.ndarray))) and gc_regul <= 0
    if isinstance(model, (tuple, DeviceClassModel)):
        from . import graph_cuts
        if not hasattr(image, 'is_cuda'):
            image = eng.to_device(_supported_dtype(_as_rgb_like(np.asarray(image))), 'image')
        graphable = (USE_CUDA_GRAPHS and not no_cut and all(k == 'color' for k in dict_features) and flags_are_native(dict_features))
        if isinstance(model, DeviceClassModel):
            _check_model_width(model, dict_features)
            nb_classes = model.n_classes
            d_model = model.device_params(eng)      # before any capture: const_device refuses a new constant while capturing
            model_key = ('predict', model.digest)

            def class_proba(res):
                return eng.gmm_predict(res.d_feat, d_model, nb_classes, d_n=res.d_n_labels)
        else:
            _, nb_classes, use_scaler, max_iter = model
            n_init = max(1, int(np.sqrt(max_iter)))
            graphable = graphable and native_feature_layout(dict_features)[1] <= graph_cuts.DEVICE_GMM_SINGLE_KERNEL_MAX_FEATURES
            model_key = model

            def class_proba(res):
                return eng.gmm_fit_predict(res.d_feat, nb_classes, n_init, max_iter, use_scaler, graph_cuts.RANDOM_SEED,
                                           d_n=res.d_n_labels)[0]

        def first_half():
            res = _device_slic_features(eng, image, dict_features, sp_size, sp_regul)
            return res, class_proba(res)

        key1 = ('probabilities', id(eng), image.data_ptr(), tuple(image.shape), str(image.dtype), model_key, _features_key(dict_features),
                sp_size, sp_regul)
        res, d_proba = _graph_call(eng, key1, first_half) if graphable else first_half()
        if no_cut:
            nb = int(eng.to_host(res.d_n_labels)[0])
            d_labels = _argmin_labels_device(eng, eng.to_host(d_proba[:nb]))
            return eng.gather(res.d_seg, d_labels, d_proba) + (None, )
        cap = edge_cap or edge_capacity(res.nb_bound)
        if soft_sink is not None:
            soft_sink(res.d_seg, d_proba)

        def second_half():
            return _device_graphcut(eng, res, res.nb_bound, d_proba, gc_regul, gc_edge_type, d_n_nodes=res.d_n_labels,
                                    want_soft=soft_sink is None, edge_cap=cap)

        key2 = ('cut', id(eng), res.d_seg.data_ptr(), d_proba.data_ptr(), res.d_centres.data_ptr(), res.shape, res.nb_bound, nb_classes,
                float(gc_regul) if graphable else None, gc_edge_type, cap, soft_sink is None)
        _, d_segm, d_soft, d_n_edges, cap = _graph_call(eng, key2, second_half) if graphable else second_half()
        return d_segm, d_soft, (d_n_edges, cap)
    res = _device_slic_features(eng, image, dict_features, sp_size, sp_regul)
    nb = int(eng.to_host(res.d_n_labels)[0])
    features = eng.to_host(res.d_feat[:nb]).copy()
    features[np.isnan(features)] = 0
    proba = np.ascontiguousarray(model(features), dtype=np.float64)
    logging.debug('list of probabilities: %r', proba.shape)
    d_proba = eng.to_device(proba, 'proba')
    if no_cut:
        return eng.gather(res.d_seg, _argmin_labels_device(eng, proba), d_proba) + (None, )
    cap = edge_cap or edge_capacity(nb)
    if soft_sink is not None:
        soft_sink(res.d_seg, d_proba)
    _, d_segm, d_soft, d_n_edges, cap = _device_graphcut(eng, res, nb, d_proba, gc_regul, gc_edge_type, want_soft=soft_sink is None,
                                                         edge_cap=cap)
    return d_segm, d_soft, (d_n_edges, cap)


def _download_results(eng, tensors):
    """D2H into pinned buffers with ONE synchronisation; returns numpy views"""
    hosts, event = eng.download(tensors)
    event.synchronize()
    return [h.numpy() for h in hosts]


def _segment(image, model, dict_features, sp_size, sp_regul, gc_regul, gc_edge_type, debug_visual, classes=None, edge_cap=None):
    image = np.asarray(image)
    eng = get_engine()
    native = image.ndim == 3 and flags_are_native(dict_features) and gc_edge_type not in ('color', 'features')
    if not native or debug_visual is not None:
        # general path: every stage still runs on the device, but through the numpy-facing stage functions
        if isinstance(model, DeviceClassModel):
            proba_fn = model.predict_proba
        else:
            proba_fn = model if callable(model) else (lambda f: estim_class_model(f, model[1], 'GMM', None, model[2], model[3]).predict_proba(f))
        slic, features = compute_color2d_superpixels_features(image, dict_features, sp_size=sp_size, sp_regul=sp_regul)
        if debug_visual is not None:
            img3 = image if image.ndim == 3 else np.stack([image] * 3, axis=-1)
            debug_visual['image'] = img3
            debug_visual['slic'] = slic
            means = np.stack([np.bincount(slic.ravel(), weights=img3[..., c].ravel()) for c in range(3)], 1)
            debug_visual['slic_mean'] = (means / np.maximum(np.bincount(slic.ravel()), 1)[:, None])[slic]
        proba = proba_fn(features)
        segm_soft = proba[slic]
        graph_labels = segment_graph_cut_general(slic, proba, image, features, gc_regul, gc_edge_type, debug_visual=debug_visual)
        if classes is not None:
            graph_labels = classes[graph_labels]
        return graph_labels[slic], segm_soft
    early = {}

    def soft_sink(d_seg, d_proba):
        early['host'], early['event'] = _soft_on_side_stream(eng, d_seg, d_proba)

    while True:
        early.clear()
        d_segm, d_soft, check = _run_resident(eng, image, model, dict_features, sp_size, sp_regul, gc_regul, gc_edge_type,
                                              soft_sink=soft_sink if EARLY_SOFT_DOWNLOAD else None, edge_cap=edge_cap)
        if check is None:       # no graph cut: both gathers were done at the end of the main stream
            segm, soft = _download_results(eng, (d_segm, d_soft))
            break
        if early:
            segm, n_edges = _download_results(eng, (d_segm, check[0]))
            early['event'].synchronize()
            soft = early['host'].numpy()
            # the next call reuses the buffers the side stream has just read: nothing of this call is left in flight
        else:                   # overlap switched off: segm_soft was gathered at the end of the main stream
            segm, soft, n_edges = _download_results(eng, (d_segm, d_soft, check[0]))
        if int(n_edges[0]) <= check[1]:
            break
        edge_cap = grown_edge_capacity(check[1])     # the device edge table overflowed: redo larger
    if classes is not None:
        segm = np.asarray(classes)[segm]
    return segm, soft


_BATCH_ENGINES = {}


def _batch_engines(nb_streams):
    """independent Engine instances (own buffers) with one CUDA stream each, cached per device"""
    from .engine import Engine
    torch = get_engine().torch
    dev = torch.cuda.current_device()
    pool = _BATCH_ENGINES.setdefault(dev, [])
    while len(pool) < nb_streams:
        pool.append((Engine(dev), torch.cuda.Stream(device=dev)))
    return pool[:nb_streams]


def _run_batch(list_images, nb_streams, max_in_flight, launch, finish):
    """consecutive images alternate over ``nb_streams`` engines with a CUDA stream each, at most ``max_in_flight`` of them
    unfinished.  ``launch(eng, image)`` queues one image's work and downloads on the current stream and returns (pinned host
    tensors, their event, extra); ``finish(index, host arrays, extra)`` runs once the event has fired and gives the image's result.
    Returns the results in input order."""
    engines = _batch_engines(nb_streams)
    torch = engines[0][0].torch
    results, pending = [None] * len(list_images), []

    def _finish(item):
        idx, hosts, event, extra = item
        event.synchronize()
        results[idx] = finish(idx, [h.numpy() for h in hosts], extra)

    caller_stream = torch.cuda.current_stream()
    for i, image in enumerate(list_images):
        eng, stream = engines[i % nb_streams]
        stream.wait_stream(caller_stream)
        with torch.cuda.stream(stream):
            pending.append((i, ) + launch(eng, np.asarray(image)))
        while len(pending) > max_in_flight:
            _finish(pending.pop(0))
    while pending:
        _finish(pending.pop(0))
    return results


def segment_images_batch(list_images, nb_classes=None, dict_features=FTS_SET_SIMPLE, sp_size=30, sp_regul=0.2, use_scaler=True,
                         gc_regul=1., gc_edge_type='model', model_pipeline=None, nb_streams=3, max_in_flight=6):
    """ the hot path over a LIST of images, the way the reference's experiment scripts run it through a process pool
    (``run_segm_slic_model_graphcut.py:461-466``): here consecutive images alternate over ``nb_streams`` CUDA streams with
    their own buffers, so the upload of image i+1 and the download of image i-1 overlap the kernels of image i.

    :param int nb_classes: fit the default GMM per image on the GPU (as ``pipe_color2d_slic_features_model_graphcut``), or
    :param model_pipeline: a fitted model used for every image (as ``segment_color2d_slic_features_model_graphcut``)
    :return list(tuple(ndarray,ndarray)): (segm, segm_soft) per image, in input order
    """
    if (nb_classes is None) == (model_pipeline is None):
        raise ValueError('give either nb_classes (per-image GMM) or model_pipeline')
    native = flags_are_native(dict_features) and gc_edge_type not in ('color', 'features')
    nb_fts = native_feature_layout(dict_features)[1] if native else 10 ** 6
    if model_pipeline is None and not (native and device_gmm_applicable(nb_fts, nb_classes)):
        return [pipe_color2d_slic_features_model_graphcut(im, nb_classes, dict_features, sp_size, sp_regul, None, use_scaler, 'GMM',
                                                          gc_regul, gc_edge_type) for im in list_images]
    if not native:
        return [segment_color2d_slic_features_model_graphcut(im, model_pipeline, dict_features, sp_size, sp_regul, gc_regul, gc_edge_type)
                for im in list_images]
    if model_pipeline is None:
        model = ('fit', nb_classes, use_scaler, 99)
    else:
        model = model_pipeline if isinstance(model_pipeline, DeviceClassModel) else model_pipeline.predict_proba
    classes = getattr(model_pipeline, 'classes_', None)

    def launch(eng, image):
        d_segm, d_soft, check = _run_resident(eng, image, model, dict_features, sp_size, sp_regul, gc_regul, gc_edge_type)
        return eng.download((d_segm, d_soft) + ((check[0], ) if check is not None else ())) + (check, )

    def finish(idx, hosts, check):
        segm, soft = hosts[0], hosts[1]
        if check is not None and int(hosts[2][0]) > check[1]:
            # edge table overflow (not seen in practice): redo this image through the single-image path with a larger table
            return _segment(list_images[idx], model, dict_features, sp_size, sp_regul, gc_regul, gc_edge_type, None, classes=classes,
                            edge_cap=grown_edge_capacity(check[1]))
        if classes is not None:
            segm = np.asarray(classes)[segm]
        return segm, soft

    return _run_batch(list_images, nb_streams, max_in_flight, launch, finish)


def compute_features_batch(list_images, dict_features, sp_size=30, sp_regul=0.2, nb_streams=3, max_in_flight=6):
    """ superpixel features of a LIST of images (the per-image half of ``estim_model_classes_group``, which the reference hands to
    a process pool, pipelines.py:139-147): consecutive images alternate over ``nb_streams`` CUDA streams with their own buffers,
    nothing synchronises with the host until an image's feature table is downloaded

    :return list(ndarray): features [N_i, D] per image, in input order
    """
    if not flags_are_native(dict_features) or any(np.ndim(im) != 3 for im in list_images):
        return [compute_color2d_superpixels_features(im, dict_features, sp_size=sp_size, sp_regul=sp_regul)[1] for im in list_images]

    def launch(eng, image):
        res = _device_slic_features(eng, image, dict_features, sp_size, sp_regul)
        return eng.download((res.d_feat, res.d_n_labels)) + (None, )

    def finish(idx, hosts, _):
        features = hosts[0][:int(hosts[1][0])].copy()
        features[np.isnan(features)] = 0
        return features

    return _run_batch(list_images, nb_streams, max_in_flight, launch, finish)


def wrapper_compute_color2d_slic_features_labels(img_annot, sp_size, sp_regul, dict_features, label_purity):
    """ superpixels, their features and one training label per superpixel from an annotated image -- the data step of the
    supervised path (reference pipelines.py:272-290): a superpixel takes the annotation label that covers most of it, or -1
    when that share is below ``label_purity`` (or the winner is the negative / unknown label)

    :param tuple(ndarray,ndarray) img_annot: image and its annotation (negative values = unknown)
    :return tuple(ndarray,ndarray,ndarray): slic [H, W], features [N, D], labels [N]
    """
    from .labeling import histogram_regions_labels_norm
    from .utilities import ImageDimensionError
    img, annot = img_annot
    annot = np.asarray(annot).astype(int)
    if np.shape(img)[:2] != annot.shape[:2]:
        raise ImageDimensionError('image %r and annot %r should match' % (np.shape(img), annot.shape))
    slic, features = compute_color2d_superpixels_features(img, dict_features, sp_size=sp_size, sp_regul=sp_regul)
    neg_label = int(np.max(annot)) + 1 if np.any(annot < 0) else None
    if neg_label is not None:
        annot = np.where(annot < 0, neg_label, annot)
    label_hist = histogram_regions_labels_norm(slic, annot)       # joint histogram on the device (isb_region_label_hist)
    labels = np.argmax(label_hist, axis=1)
    purity = np.max(label_hist, axis=1)
    if neg_label is not None:
        labels[labels == neg_label] = -1
    labels[purity < label_purity] = -1
    return slic, features, labels


def train_classif_color2d_slic_features(list_images, list_annots, dict_features, sp_size=30, sp_regul=0.2, clf_name=CLASSIF_NAME,
                                        label_purity=0.9, feature_balance='unique', pca_coef=None, nb_classif_search=1,
                                        nb_hold_out=CROSS_VAL_LEAVE_OUT, nb_workers=1):
    """ the supervised training wrapper of the reference (pipelines.py:293-379).  Its data step is available here
    (:func:`wrapper_compute_color2d_slic_features_labels`); the classifier zoo, hyper-parameter search and dataset balancing it
    hands the data to (``imsegm/classification.py``) are outside the accelerated hot path (SURVEY.md section 2, row 8) """
    raise NotImplementedError('supervised classifier training (imsegm.classification) is outside the B200 hot path; '
                              'use wrapper_compute_color2d_slic_features_labels for the features and labels')


def pipe_gray3d_slic_features_model_graphcut(image, nb_classes, dict_features, spacing=(12, 1, 1), sp_size=15, sp_regul=0.2,
                                             gc_regul=0.1):
    """ the pipeline for a gray VOLUME: 3-D SLIC supervoxels, their features, a class model, GraphCut over the 6-connected
    supervoxel graph (reference pipelines.py:382-431)

    :param ndarray image: gray volume [D, H, W]
    :param tuple(int,int,int) spacing: voxel spacing (z, y, x)
    :return ndarray: class per voxel [D, H, W]
    """
    from .descriptors import compute_selected_features_gray3d, norm_features
    from .superpixels import segment_slic_img3d_gray
    image = np.asarray(image)
    slic = segment_slic_img3d_gray(image, sp_size=sp_size, relative_compact=sp_regul, space=spacing)
    features, _ = compute_selected_features_gray3d(image, slic, dict_features)
    features[np.isnan(features)] = 0
    features, _ = norm_features(features)
    model = estim_class_model(features, nb_classes)
    proba = model.predict_proba(features)
    graph_labels = segment_graph_cut_general(slic, proba, image, features, gc_regul)
    return graph_labels[slic]


def segment_resident(d_image, model, dict_features, sp_size=30, sp_regul=0.2, gc_regul=1., gc_edge_type='model'):
    """ the same hot path with the image ALREADY on the device (a cuda tensor [H, W, 3]) and the results left
    there: returns (segm int32 [H, W], segm_soft float64 [H, W, K]) device tensors.  ``model`` is a callable
    proba_fn(features), a :class:`graph_cuts.DeviceClassModel` (evaluated on the GPU) or ('fit', nb_classes, use_scaler, max_iter)
    for the GPU-fitted default GMM. """
    return _run_resident(get_engine(), d_image, model, dict_features, sp_size, sp_regul, gc_regul, gc_edge_type)[:2]


def pipe_color2d_slic_features_model_graphcut(image, nb_classes, dict_features, sp_size=30, sp_regul=0.2, pca_coef=None,
                                              use_scaler=True, estim_model='GMM', gc_regul=1., gc_edge_type='model',
                                              debug_visual=None):
    """ complete pipeline: superpixels, features, class model estimated on this image, GraphCut
    (reference pipelines.py:46-110)

    :param ndarray image: input RGB image
    :param int nb_classes: number of classes to be segmented
    :param dict dict_features: {'color': [...], ...}
    :return tuple(ndarray,ndarray): segmentation [H, W] int32, soft segmentation [H, W, nb_classes] float64
    """
    logging.info('PIPELINE Superpixels-Features-GMM-GraphCut')
    nb_fts = native_feature_layout(dict_features)[1] if flags_are_native(dict_features) else 10 ** 6
    if flags_are_native(dict_features) and device_gmm_applicable(nb_fts, nb_classes, estim_model, pca_coef):
        model = ('fit', nb_classes, use_scaler, 99)
    else:
        def model(features):
            return estim_class_model(features, nb_classes, estim_model, pca_coef, use_scaler).predict_proba(features)
    return _segment(image, model, dict_features, sp_size, sp_regul, gc_regul, gc_edge_type, debug_visual)


def estim_model_classes_group(list_images, nb_classes, dict_features, sp_size=30, sp_regul=0.2, use_scaler=True,
                              pca_coef=None, model_type='GMM', nb_workers=NB_WORKERS):
    """ one class model from the superpixel features of a sequence of images (reference pipelines.py:113-157);
    the per-image work that the reference spreads over a process pool runs back to back on the GPU

    :return tuple(model, list(ndarray)): fitted sklearn pipeline, list of per-image features
    """
    list_features = compute_features_batch(list_images, dict_features, sp_size=sp_size, sp_regul=sp_regul)
    features = np.nan_to_num(np.concatenate(tuple(list_features), axis=0))
    model = estim_class_model(features, nb_classes, model_type, pca_coef, use_scaler)
    return model, list_features


def segment_color2d_slic_features_model_graphcut(image, model_pipeline, dict_features, sp_size=30, sp_regul=0.2, gc_regul=1.,
                                                 gc_edge_type='model', debug_visual=None):
    """ complete pipeline with a given (already fitted) model (reference pipelines.py:160-241)

    :param model_pipeline: a fitted model with ``predict_proba`` (evaluated on the host, as in the reference), or a
        :class:`graph_cuts.DeviceClassModel` wrapping one (evaluated on the GPU: the path never leaves the device)
    :return tuple(ndarray,ndarray): segmentation [H, W], soft segmentation [H, W, K]
    """
    logging.info('PIPELINE Superpixels-Features-Model-GraphCut')
    classes = getattr(model_pipeline, 'classes_', None)
    model = model_pipeline if isinstance(model_pipeline, DeviceClassModel) else model_pipeline.predict_proba
    return _segment(image, model, dict_features, sp_size, sp_regul, gc_regul, gc_edge_type, debug_visual,
                    classes=classes)
