"""
GraphCut on the superpixel graph, on the GPU.

Mirror of the reference module ``imsegm/graph_cuts.py`` (same public names, arguments, error types).  The graph,
the energies and the alpha-expansion itself run in CUDA behind ``include/imsegm_b200.h``
(``isb_adjacency_edges`` / ``isb_gc_energies`` / ``isb_alpha_expansion``); the class model stays scikit-learn
exactly as in the reference (``estim_class_model``, reference graph_cuts.py:73-163), fitted on the device when it is the default GMM
(``isb_gmm_fit_predict``); a fitted mixture wrapped in :class:`DeviceClassModel` is evaluated on the device (``isb_gmm_predict``).
"""
import logging

import numpy as np

from .engine import EDGE_MODES, get_engine
from .superpixels import (
    device_adjacency,
    make_graph_segm_connect_grid2d_conn4,
    make_graph_segm_connect_grid3d_conn6,
    superpixel_centers,
)

#: number of iterations in Graph-Cut optimisation (reference graph_cuts.py:32)
DEFAULT_GC_ITERATIONS = 25
#: minimal probability of a class in the unary term (reference graph_cuts.py:36)
MIN_UNARY_PROB = 0.01
#: cap of the pairwise (smoothness) term (reference graph_cuts.py:38)
MAX_PAIRWISE_COST = 1e5
#: edge weights are clamped to [1 / val, val] (reference graph_cuts.py:40)
MIN_MAX_EDGE_WEIGHT = 1e3
#: the default 'GMM' class model is fitted on the GPU (isb_gmm_fit_predict) when it fits the device kernel
#: (<= 16 features, <= 8 classes, no PCA); set False to force scikit-learn on the host
USE_DEVICE_GMM = True
#: seed of the device k-means++ initialisation (the reference leaves its model unseeded)
RANDOM_SEED = 0
#: D <= 16 runs as one kernel (a CTA per restart), 16 < D <= 256 (colour + Leung-Malik = 189) as batched FP64 GEMMs
DEVICE_GMM_MAX_FEATURES, DEVICE_GMM_MAX_CLASSES = 232, 8   # = DBIG of csrc/gmm.cu
#: up to this many features the fit is one kernel without any host synchronisation (csrc/gmm.cu DMAX)
DEVICE_GMM_SINGLE_KERNEL_MAX_FEATURES = 16


# ---------------------------------------------------------------------------------------------------------------------
# class model (host, scikit-learn -- unchanged behaviour of the reference)
# ---------------------------------------------------------------------------------------------------------------------

def estim_gmm_params(features, prob):
    """ GMM parameters from a soft labelling, hard-assigned by argmax (reference graph_cuts.py:43-70) """
    nb_samples, nb_classes = prob.shape
    labels = np.argmax(prob, axis=1)
    params = {'weights': [], 'means': [], 'covars': []}
    for lb in range(nb_classes):
        sel = labels == lb
        params['weights'].append(np.sum(sel) / float(nb_samples))
        params['means'].append(np.mean(features[sel], axis=0))
        params['covars'].append(np.cov(features[sel]))
    for n in ('means', 'covars'):
        params[n] = np.array([m.tolist() for m in params[n]])
    return params


def compute_multivarian_otsu(features):
    """ per-dimension Otsu split combined by majority vote (reference graph_cuts.py:166-193) """
    features = np.asarray(features)
    votes = np.zeros(features.shape)
    for i in range(features.shape[-1]):
        assign = features[:, i] > _threshold_otsu(features[:, i])
        if i > 0:
            m = np.mean(votes[:, :i], axis=1)
            if np.mean(np.abs(~assign - m)) < np.mean(np.abs(assign - m)):
                assign = ~assign
        votes[:, i] = assign
    return np.mean(votes, axis=1) > 0.5


def _threshold_otsu(values, nbins=256):
    """Otsu threshold on a 1-D sample (the reference takes it from skimage.filters, graph_cuts.py:183)"""
    hist, edges = np.histogram(np.asarray(values, dtype=float).ravel(), bins=nbins)
    centers = (edges[:-1] + edges[1:]) / 2.
    hist = hist.astype(float)
    w1 = np.cumsum(hist)
    w2 = np.cumsum(hist[::-1])[::-1]
    m1 = np.cumsum(hist * centers) / np.maximum(w1, 1e-300)
    m2 = (np.cumsum((hist * centers)[::-1]) / np.maximum(w2[::-1], 1e-300))[::-1]
    var12 = w1[:-1] * w2[1:] * (m1[:-1] - m2[1:]) ** 2
    return centers[:-1][np.argmax(var12)]


def estim_class_model_gmm(features, nb_classes, init='kmeans'):
    """ GMM over the features, optionally initialised by k-means (reference graph_cuts.py:221-249) """
    from sklearn import cluster, mixture
    gmm = mixture.GaussianMixture(n_components=nb_classes, covariance_type='full', max_iter=99)
    if init == 'kmeans':
        y = cluster.KMeans(n_clusters=nb_classes, init='k-means++').fit_predict(features)
        gmm.fit(features, y)
    else:
        gmm.fit(features)
    return gmm


def estim_class_model_kmeans(features, nb_classes, init_type='k-means++', max_iter=99):
    """ Gaussians fitted on a k-means clustering (reference graph_cuts.py:252-285) """
    from sklearn import cluster, mixture
    if init_type == 'quantiles':
        init_perc = np.array(np.percentile(features, np.linspace(5, 95, nb_classes).tolist(), axis=0))
        kmeans = cluster.KMeans(nb_classes, init=init_perc, max_iter=2)
    else:
        kmeans = cluster.KMeans(nb_classes, init=init_type, max_iter=max_iter, n_init=max(1, int(np.sqrt(max_iter))))
    y = kmeans.fit_predict(features)
    gmm = mixture.GaussianMixture(n_components=nb_classes, covariance_type='full', max_iter=1)
    gmm.fit(features, y)
    return gmm, y


def device_gmm_applicable(nb_features, nb_classes, estim_model='GMM', pca_coef=None):
    return (USE_DEVICE_GMM and estim_model == 'GMM' and pca_coef is None and nb_features <= DEVICE_GMM_MAX_FEATURES
            and nb_classes <= DEVICE_GMM_MAX_CLASSES)


def sklearn_pipeline_from_device(params, nb_features, nb_classes, nb_samples, use_scaler=True, n_init=1, max_iter=99):
    """ wrap the parameters fitted by ``isb_gmm_fit_predict`` into the scikit-learn objects the reference returns
    (Pipeline[StandardScaler?, GaussianMixture]) so that ``predict_proba`` & co. keep working on the host """
    from sklearn import mixture, pipeline, preprocessing
    p = np.asarray(params, dtype=np.float64)
    D, K = int(nb_features), int(nb_classes)
    mean, scale = p[:D].copy(), p[D:2 * D].copy()
    o = 2 * D
    weights = p[o:o + K].copy()
    o += K
    means = p[o:o + K * D].reshape(K, D).copy()
    o += K * D
    covs = p[o:o + K * D * D].reshape(K, D, D).copy()
    o += K * D * D
    prec_chol = p[o:o + K * D * D].reshape(K, D, D).copy()
    o += K * D * D
    lower, n_iter, converged, ok = p[o:o + 4]
    if not ok:
        raise ValueError('Fitting the mixture model failed because some components have ill-defined empirical covariance '
                         '(for instance caused by singleton or collapsed samples). Try to decrease the number of components')
    steps = []
    if use_scaler:
        sc = preprocessing.StandardScaler()
        sc.mean_, sc.scale_, sc.var_ = mean, scale, scale ** 2
        sc.n_features_in_, sc.n_samples_seen_ = D, int(nb_samples)
        steps.append(('std_scaler', sc))
    mm = mixture.GaussianMixture(n_components=K, covariance_type='full', n_init=n_init, max_iter=max_iter)
    mm.weights_, mm.means_, mm.covariances_, mm.precisions_cholesky_ = weights, means, covs, prec_chol
    mm.precisions_ = np.array([u @ u.T for u in prec_chol])
    mm.converged_, mm.n_iter_, mm.lower_bound_, mm.n_features_in_ = bool(converged), int(n_iter), float(lower), D
    steps.append(('model', mm))
    return pipeline.Pipeline(steps)


def estim_class_model_device(features, nb_classes, use_scaler=True, max_iter=99, init_labels=None, seed=None):
    """ the default 'GMM' model fitted on the GPU; returns the same kind of object as :func:`estim_class_model` """
    features = np.ascontiguousarray(features, dtype=np.float64)
    eng = get_engine()
    n_init = max(1, int(np.sqrt(max_iter))) if init_labels is None else len(np.atleast_2d(init_labels))
    d_feat = eng.to_device(features, 'feat_in')
    _, params = eng.gmm_fit_predict(d_feat, nb_classes, n_init, max_iter, use_scaler, RANDOM_SEED if seed is None else seed,
                                    init_labels=None if init_labels is None else np.atleast_2d(init_labels))
    return sklearn_pipeline_from_device(eng.to_host(params), features.shape[1], nb_classes, len(features), use_scaler, n_init, max_iter)


def _mixture_and_scaler(model):
    """(StandardScaler or None, fitted mixture) of a model :class:`DeviceClassModel` can evaluate; ValueError naming the step it
    cannot take"""
    from sklearn import mixture, pipeline, preprocessing
    steps = list(model.steps) if isinstance(model, pipeline.Pipeline) else [('model', model)]
    for i, (name, step) in enumerate(steps[:-1]):
        if i > 0 or not isinstance(step, preprocessing.StandardScaler):
            raise ValueError('DeviceClassModel takes a mixture model behind at most one StandardScaler, not step %r (%s)'
                             % (name, type(step).__name__))
    name, mm = steps[-1]
    if not isinstance(mm, (mixture.GaussianMixture, mixture.BayesianGaussianMixture)):
        raise ValueError('DeviceClassModel evaluates a GaussianMixture or BayesianGaussianMixture, not step %r (%s)'
                         % (name, type(mm).__name__))
    if not hasattr(mm, 'precisions_cholesky_'):
        raise ValueError('DeviceClassModel needs a fitted model (step %r is not fitted)' % name)
    return (steps[0][1] if len(steps) > 1 else None), mm


def pack_class_model(model):
    """ the device vector of ``isb_gmm_predict`` for a fitted mixture model (optionally behind a StandardScaler):
    shift[D] | scale[D] | U[K, D, D] | b[K, D] | c[K], computed the way scikit-learn's ``_estimate_log_gaussian_prob``,
    ``_estimate_log_prob`` and ``_estimate_log_weights`` compute them (every covariance type expanded to a full triangular U_k)

    :return tuple(ndarray, int, int): the vector, D, K
    """
    from scipy.special import digamma
    from sklearn import mixture
    scaler, mm = _mixture_and_scaler(model)
    means = np.asarray(mm.means_, dtype=np.float64)
    K, D = means.shape
    if D > DEVICE_GMM_MAX_FEATURES or K > DEVICE_GMM_MAX_CLASSES:
        raise ValueError('DeviceClassModel handles up to %d features and %d classes (got D=%d, K=%d)'
                         % (DEVICE_GMM_MAX_FEATURES, DEVICE_GMM_MAX_CLASSES, D, K))
    shift, scale = np.zeros(D), np.ones(D)
    if scaler is not None:
        if getattr(scaler, 'n_features_in_', D) != D:
            raise ValueError('the StandardScaler has %d features, the mixture %d' % (scaler.n_features_in_, D))
        if scaler.with_mean:
            shift = np.asarray(scaler.mean_, dtype=np.float64)
        if scaler.with_std:
            scale = np.asarray(scaler.scale_, dtype=np.float64)
    pc = np.asarray(mm.precisions_cholesky_, dtype=np.float64)
    diag = np.arange(D)
    ct = mm.covariance_type
    U = np.zeros((K, D, D))
    if ct == 'full':
        U[:] = pc
        log_det = np.log(pc[:, diag, diag]).sum(axis=1)
    elif ct == 'tied':
        U[:] = pc[None]
        log_det = np.full(K, np.log(np.diag(pc)).sum())
    elif ct == 'diag':
        U[:, diag, diag] = pc
        log_det = np.log(pc).sum(axis=1)
    elif ct == 'spherical':
        U[:, diag, diag] = pc[:, None]
        log_det = D * np.log(pc)
    else:
        raise ValueError('unknown covariance_type %r' % ct)
    b = np.einsum('kd,kde->ke', means, U)
    if isinstance(mm, mixture.BayesianGaussianMixture):
        dof = np.broadcast_to(np.asarray(mm.degrees_of_freedom_, dtype=np.float64), (K,))
        log_lambda = D * np.log(2.0) + np.sum(digamma(0.5 * (dof - np.arange(D)[:, None])), 0)
        c = log_det - 0.5 * D * np.log(dof) + 0.5 * (log_lambda - D / np.asarray(mm.mean_precision_, dtype=np.float64))
        if mm.weight_concentration_prior_type == 'dirichlet_process':
            a, bb = (np.asarray(v, dtype=np.float64) for v in mm.weight_concentration_)
            dsum = digamma(a + bb)
            log_w = digamma(a) - dsum + np.hstack((0, np.cumsum(digamma(bb) - dsum)[:-1]))
        else:
            conc = np.asarray(mm.weight_concentration_, dtype=np.float64)
            log_w = digamma(conc) - digamma(np.sum(conc))
        c = c + log_w
    else:
        c = log_det + np.log(np.asarray(mm.weights_, dtype=np.float64))
    vec = np.concatenate([shift, scale, U.ravel(), b.ravel(), c]).astype(np.float64)
    return np.ascontiguousarray(vec), int(D), int(K)


class DeviceClassModel(object):
    """ a fitted class model whose ``predict_proba`` runs on the GPU (``isb_gmm_predict``): a GaussianMixture or
    BayesianGaussianMixture of any covariance type, bare or as the last step of a Pipeline whose only other step is a
    StandardScaler -- every model the reference's ``estim_class_model`` builds without PCA.  Packed once, at construction.

    Passed to ``segment_color2d_slic_features_model_graphcut``, ``segment_images_batch(model_pipeline=...)``,
    ``segment_resident`` or ``tiled.segment_color2d_slic_features_model_graphcut_tiled`` it keeps the whole path on the device
    (no feature download, no host model, CUDA-graph replays); a plain scikit-learn model keeps the host round trip.

    :param model: the fitted scikit-learn object, kept as ``.model``; ``classes_`` is passed through when it has one
    """

    def __init__(self, model):
        import hashlib
        import weakref
        self.model = model
        self.params, self.n_features, self.n_classes = pack_class_model(model)
        self.digest = hashlib.blake2b(self.params.tobytes(), digest_size=16).hexdigest()
        classes = getattr(model, 'classes_', None)
        if classes is not None:
            self.classes_ = classes
        self._on_device = weakref.WeakKeyDictionary()

    def device_params(self, eng):
        """the packed vector on ``eng``'s device (``Engine.const_device``: one tensor per engine and content, never overwritten);
        call it outside a CUDA-graph capture"""
        d = self._on_device.get(eng)
        if d is None:
            d = self._on_device[eng] = eng.const_device(self.params, 'class_model')
        return d

    def predict_proba(self, features):
        """ class probabilities [N, K] of host features [N, D] (NaN taken as 0), computed on the device """
        X = np.ascontiguousarray(features, dtype=np.float64)
        if X.ndim != 2 or X.shape[1] != self.n_features:
            raise ValueError('features of shape %r, the model takes %d columns' % (X.shape, self.n_features))
        if not len(X):
            return np.zeros((0, self.n_classes))
        eng = get_engine()
        d_feat = eng.to_device(X, 'feat_in')
        proba = eng.gmm_predict(d_feat, self.device_params(eng), self.n_classes)
        return eng.to_host(proba).copy()

    def __repr__(self):
        return 'DeviceClassModel(%r)' % (self.model, )


def estim_class_model(features, nb_classes, estim_model='GMM', pca_coef=None, use_scaler=True, max_iter=99):
    """ scikit-learn pipeline (scaler, PCA, mixture model) fitted on the features (reference graph_cuts.py:73-163)

    :param ndarray features: [nb_samples, nb_features]
    :param int nb_classes: number of classes
    :param str estim_model: 'GMM', 'GMM_kmeans', 'GMM_Otsu', 'kmeans', 'kmeans_quantiles', 'BGM', 'Otsu'
    :return: fitted sklearn Pipeline with ``predict_proba``
    """
    features = np.asarray(features)
    if device_gmm_applicable(features.shape[1], nb_classes, estim_model, pca_coef):
        import torch
        if torch.cuda.is_available():
            return estim_class_model_device(features, nb_classes, use_scaler, max_iter)
    from sklearn import cluster, decomposition, mixture, pipeline, preprocessing
    steps = []
    if use_scaler:
        steps.append(('std_scaler', preprocessing.StandardScaler()))
    if pca_coef is not None:
        steps.append(('reduce_dim', decomposition.PCA(pca_coef)))
    nb_inits = max(1, int(np.sqrt(max_iter)))
    mm = mixture.GaussianMixture(n_components=nb_classes, covariance_type='full', n_init=nb_inits, max_iter=max_iter)
    init_type = ''
    if '_' in estim_model:
        estim_model, init_type = estim_model.split('_')[0], estim_model.split('_')[-1]
    y = None
    if estim_model == 'GMM':
        if init_type == 'kmeans':
            mm.set_params(n_init=1)
            y = cluster.KMeans(n_clusters=nb_classes, init='k-means++').fit_predict(features)
        elif init_type == 'Otsu':
            mm.set_params(n_init=1)
            y = compute_multivarian_otsu(features)
    elif estim_model == 'kmeans':
        mm.set_params(max_iter=1)
        init_type = 'quantiles' if init_type == 'quantiles' else 'k-means++'
        _, y = estim_class_model_kmeans(features, nb_classes, init_type=init_type, max_iter=max_iter)
    elif estim_model == 'BGM':
        mm = mixture.BayesianGaussianMixture(n_components=nb_classes, covariance_type='full', n_init=nb_inits,
                                             max_iter=max_iter)
    elif estim_model == 'Otsu' and nb_classes == 2:
        mm.set_params(max_iter=1, n_init=1)
        y = compute_multivarian_otsu(features)
    steps.append(('model', mm))
    model = pipeline.Pipeline(steps)
    if y is not None:
        model.fit(features, y)
    else:
        model.fit(features)
    return model


# ---------------------------------------------------------------------------------------------------------------------
# graph + energies
# ---------------------------------------------------------------------------------------------------------------------

def get_vertexes_edges(segments):
    """ vertices and edges of the region adjacency graph, 2-D or 3-D (reference graph_cuts.py:288-300) """
    segments = np.asarray(segments)
    if segments.ndim == 3:
        return make_graph_segm_connect_grid3d_conn6(segments)
    if segments.ndim == 2:
        return make_graph_segm_connect_grid2d_conn4(segments)
    return None, None


def compute_spatial_dist(centres, edges, relative=False):
    """ Euclidean distance between the centres of connected segments (reference graph_cuts.py:303-336) """
    if np.max(edges) >= len(centres):
        raise ValueError('max vertex %i exceed size of centres %i' % (np.max(edges), len(centres)))
    ndim = np.max([len(c) for c in centres if c is not None])
    centres = [[np.nan] * ndim if (c is None or len(c) == 0) else c for c in centres]
    centres = np.nan_to_num(np.asarray(centres, dtype=float))
    edges = np.asarray(edges)
    diff = centres[edges[:, 0]] - centres[edges[:, 1]]
    dist = np.sqrt(np.einsum('ij,ij->i', diff, diff))
    if relative:
        dist = dist / np.mean(dist)
    return dist


def compute_edge_model(edges, proba, metric='l_T'):
    """ edge weight exp(-d / (2 std(d)^2)) from the class probabilities of the two vertices, d by ``metric``
    'l1' / 'l2' / 'lT' (reference graph_cuts.py:383-439) """
    edges, proba = np.asarray(edges), np.asarray(proba)
    if np.max(edges) >= len(proba):
        raise ValueError('max vertex %i exceed size of proba %r' % (np.max(edges), proba.shape))
    v1, v2 = proba[edges[:, 0]], proba[edges[:, 1]]
    if metric == 'l1':
        dist = np.abs(v1 - v2).sum(axis=1)
    elif metric == 'l2':
        d = v1 - v2
        dist = np.sqrt(np.einsum('ij,ij->i', d, d))
    elif metric == 'lT':
        dist = np.max((v1 - v2) ** 2, axis=1)
    else:
        logging.error('not implemented for: %s', metric)
        return np.ones(len(edges))
    return np.exp(-dist / (2 * np.std(dist) ** 2))


def create_pairwise_matrix_uniform(gc_reg, nb_classes):
    """ Potts matrix gc_reg * (1 - I) (reference graph_cuts.py:442-456) """
    return (np.ones(nb_classes) - np.eye(nb_classes)) * gc_reg


def create_pairwise_matrix_specif(pos_weights, nb_classes=None):
    """ Potts matrix with given symmetric entries (reference graph_cuts.py:459-482) """
    if not nb_classes:
        nb_classes = np.max([list(c) for c, _ in pos_weights]) + 1
    pairwise = np.ones(nb_classes) - np.eye(nb_classes)
    for (i, j), w in pos_weights:
        pairwise[i, j] = pairwise[j, i] = w
    return pairwise


def create_pairwise_matrix(gc_regul, nb_classes):
    """ uniform / listed / full-matrix pairwise term (reference graph_cuts.py:485-520) """
    if isinstance(gc_regul, np.ndarray):
        if not gc_regul.shape[0] == gc_regul.shape[1] == nb_classes:
            raise ValueError('GC regul matrix %r should match match number of classes (%i)' % (gc_regul.shape, nb_classes))
        return gc_regul - np.min(gc_regul)
    if isinstance(gc_regul, list):
        return create_pairwise_matrix_specif(gc_regul, nb_classes)
    return create_pairwise_matrix_uniform(gc_regul, nb_classes)


def compute_unary_cost(proba, min_prob=MIN_UNARY_PROB):
    """ |-log(clip(proba, min_prob, 1 - min_prob))| (reference graph_cuts.py:523-540) """
    proba = np.clip(np.asarray(proba, dtype=float), min_prob, 1 - min_prob)
    return np.abs(np.array(-np.log(proba), dtype=np.float64))


def compute_pairwise_cost(gc_regul, proba_shape, max_pairwise_cost=MAX_PAIRWISE_COST):
    """ pairwise matrix capped at ``max_pairwise_cost`` (reference graph_cuts.py:543-555) """
    cost = np.array(create_pairwise_matrix(gc_regul, proba_shape[1]), dtype=np.float64)
    cost[cost > max_pairwise_cost] = max_pairwise_cost
    return cost


def insert_gc_debug_images(debug_visual, segments, graph_labels, unary_cost, edges, edge_weights):
    """ raw intermediates for debugging (reference graph_cuts.py:558-571; the rendered figures of
    ``imsegm.utilities.drawing`` are out of scope, the arrays they are drawn from are kept) """
    if debug_visual is None:
        return
    debug_visual['segments'] = segments
    debug_visual['edges'] = edges
    debug_visual['edge_weights'] = edge_weights
    debug_visual['imgs_unary_cost'] = [np.asarray(unary_cost)[:, i][segments] for i in range(np.asarray(unary_cost).shape[1])]
    debug_visual['img_graph_edges'] = None
    debug_visual['img_graph_segm'] = np.asarray(graph_labels)[segments]


def _edge_mode(edge_type):
    if edge_type.startswith('model'):
        metric = edge_type.split('_')[-1] if '_' in edge_type else 'lT'
        key = 'model_' + metric
        if edge_type == 'model':
            return EDGE_MODES['model']
        if key not in EDGE_MODES:
            logging.error('not implemented for: %s', metric)
            return EDGE_MODES['']
        return EDGE_MODES[key]
    return EDGE_MODES.get(edge_type, EDGE_MODES[''])


def _device_graph(eng, segments):
    """label map -> (device labels, nb, device edges, E, device centres)"""
    segments = np.asarray(segments)
    nb = int(segments.max()) + 1
    d_seg = eng.to_device(segments.astype(np.int32, copy=False), 'seg_in')
    d_edges, E = device_adjacency(eng, d_seg, nb)
    return d_seg, nb, d_edges, E


def compute_edge_weights(segments, image=None, features=None, proba=None, edge_type=''):
    """ edges of the superpixel graph and their weights (reference graph_cuts.py:574-657)

    :param ndarray segments: superpixels
    :param str edge_type: '', 'spatial', 'model[_l1|_l2|_lT]', 'color', 'features'
    :return tuple(ndarray,ndarray): edges [E, 2] int32, weights [E] float64 clamped to [1e-3, 1e3]
    """
    segments = np.asarray(segments)
    eng = get_engine()
    if edge_type.startswith('model') and (proba is None or len(proba) == 0):
        raise ValueError('"proba" is required')
    if edge_type in ('color', 'features'):
        # these two compare host-side vectors (mean colour / standardised features): same kernel, different vectors
        _, edges = get_vertexes_edges(segments)
        edges = np.array(edges, dtype=np.int32)
        if edge_type == 'color':
            if image is None:
                raise RuntimeError('"image" is required')
            from .descriptors import compute_selected_features_img2d
            image_float = np.array(image, dtype=float)
            if np.max(image) > 1:
                image_float /= 255.
            vec, _ = compute_selected_features_img2d(image_float, segments, {'color': ['mean']})
            dist = np.abs(vec[edges[:, 0]] - vec[edges[:, 1]]).sum(axis=1)
        else:
            if features is None:
                raise RuntimeError('"features" is required')
            from sklearn import preprocessing
            vec = preprocessing.StandardScaler().fit_transform(features)
            d = vec[edges[:, 0]] - vec[edges[:, 1]]
            dist = np.sqrt(np.einsum('ij,ij->i', d, d))
        weights = np.exp(-(dist.astype(float) / (2 * np.std(dist) ** 2)))
        weights /= compute_spatial_dist(superpixel_centers(segments), edges, relative=True)
        weights[weights < 1. / MIN_MAX_EDGE_WEIGHT] = 1. / MIN_MAX_EDGE_WEIGHT
        weights[weights > MIN_MAX_EDGE_WEIGHT] = MIN_MAX_EDGE_WEIGHT
        return edges, weights
    if segments.ndim == 3:
        return _edge_weights_volume(eng, segments, proba, edge_type)
    mode = _edge_mode(edge_type)
    d_seg, nb, d_edges, E = _device_graph(eng, segments)
    K = 1 if proba is None else int(np.asarray(proba).shape[1])
    p = np.ones((nb, K)) if proba is None else np.ascontiguousarray(proba, dtype=np.float64)
    if len(p) < nb:
        raise ValueError('max vertex %i exceed size of proba %r' % (nb - 1, p.shape))
    d_proba = eng.to_device(p, 'proba')
    centres = None
    if mode[1]:
        _, centres, _ = eng.segment_stats(None, d_seg, nb, (), want_centres=True)
    _, edge_w, _, _, _ = eng.gc_energies(d_proba, d_edges, E, None, centres, mode, 1.0, np.zeros((K, K)))
    edges = eng.to_host(d_edges[:E]).copy() if E else np.zeros((0, 2), dtype=np.int32)
    weights = eng.to_host(edge_w[:E]).copy() if E else np.zeros(0)
    return edges, weights


def _edge_weights_volume(eng, segments, proba, edge_type):
    """edges and weights of a label VOLUME: the 6-connected pairs and the centres come from the device (isb_adjacency_edges_3d,
    isb_centroids_3d), the per-edge arithmetic -- a few thousand edges -- follows the reference on the host (graph_cuts.py:617-657)"""
    _edge_mode(edge_type)     # validates the name
    nb = int(segments.max()) + 1
    d_seg = eng.to_device(segments.astype(np.int32, copy=False), 'seg_in3d')
    d_edges, E = device_adjacency(eng, d_seg, nb)
    d_centres = eng.centroids3d(d_seg, nb)
    edges = eng.to_host(d_edges[:E]).copy() if E else np.zeros((0, 2), dtype=np.int32)
    if not E:
        return edges, np.zeros(0)
    if edge_type.startswith('model'):
        metric = edge_type.split('_')[-1] if '_' in edge_type else 'lT'
        weights = np.array(compute_edge_model(edges, proba, metric), dtype=float)
    else:
        weights = np.ones(len(edges))
    if edge_type in ('model', 'spatial'):
        weights = weights / compute_spatial_dist(eng.to_host(d_centres).copy(), edges, relative=True)
    weights[weights < 1. / MIN_MAX_EDGE_WEIGHT] = 1. / MIN_MAX_EDGE_WEIGHT
    weights[weights > MIN_MAX_EDGE_WEIGHT] = MIN_MAX_EDGE_WEIGHT
    return edges, weights


def segment_graph_cut_general(segments, proba, image=None, features=None, gc_regul=1., edge_type='model', edge_cost=1.,
                              debug_visual=None):
    """ GraphCut labelling of the superpixels (reference graph_cuts.py:660-747)

    :param ndarray segments: superpixel map
    :param ndarray proba: class probabilities per superpixel [N, K]
    :param gc_regul: regularisation (float, list of ((i, j), w) or full matrix)
    :param str edge_type: see :func:`compute_edge_weights`
    :return ndarray: label per superpixel, int32
    """
    segments = np.asarray(segments)
    proba = np.ascontiguousarray(proba, dtype=np.float64)
    pairwise_cost = compute_pairwise_cost(gc_regul, proba.shape)
    scalar_regul = not isinstance(gc_regul, (list, np.ndarray))
    if scalar_regul and gc_regul <= 0:
        unary_cost = compute_unary_cost(proba)
        graph_labels = np.argmin(unary_cost, axis=-1).astype(np.int32)
        if debug_visual is not None:
            edges, edge_weights = compute_edge_weights(segments, image, features, proba, edge_type)
            insert_gc_debug_images(debug_visual, segments, graph_labels, unary_cost, edges, edge_weights * edge_cost)
        return graph_labels
    eng = get_engine()
    if edge_type in ('color', 'features') or segments.ndim == 3:
        edges, edge_weights = compute_edge_weights(segments, image, features, proba, edge_type)
        edge_weights = edge_weights * edge_cost
        unary_cost = compute_unary_cost(proba)
        graph_labels = cut_general_graph(edges, edge_weights, unary_cost, pairwise_cost, n_iter=-1)
    else:
        mode = _edge_mode(edge_type)
        d_seg, nb, d_edges, E = _device_graph(eng, segments)
        if len(proba) < nb:
            raise ValueError('max vertex %i exceed size of proba %r' % (nb - 1, proba.shape))
        d_proba = eng.to_device(proba, 'proba')
        centres = None
        if mode[1]:
            _, centres, _ = eng.segment_stats(None, d_seg, nb, (), want_centres=True)
        labels, unary, edge_w = eng.graph_cut(d_proba, d_edges, E, None, centres, mode, float(edge_cost), pairwise_cost)
        graph_labels = eng.to_host(labels).copy()
        if debug_visual is not None:
            edges, edge_weights = eng.to_host(d_edges[:E]).copy(), eng.to_host(edge_w[:E]).copy()
            unary_cost = eng.to_host(unary).copy()
    if debug_visual is not None:
        insert_gc_debug_images(debug_visual, segments, graph_labels, unary_cost, edges, edge_weights)
    return graph_labels


def _canonical_int_edges(edges, w_i):
    """pairs as (a, b) with a < b, self loops dropped, parallel edges merged by adding their (already integer) weights -- the energy
    GCO builds when ``setNeighbors`` is called for both orders or twice for the same pair"""
    edges = np.asarray(edges, dtype=np.int64).reshape(-1, 2)
    lo, hi = edges.min(axis=1), edges.max(axis=1)
    keep = lo != hi
    lo, hi, w_i = lo[keep], hi[keep], np.asarray(w_i, dtype=np.int64)[keep]
    if not len(lo):
        return np.zeros((0, 2), np.int32), np.zeros(0, np.intc)
    key = lo * (int(hi.max()) + 1) + hi
    uniq, inverse = np.unique(key, return_inverse=True)
    if len(uniq) == len(key) and (edges[keep][:, 0] < edges[keep][:, 1]).all():
        return np.ascontiguousarray(edges[keep], dtype=np.int32), np.ascontiguousarray(w_i, dtype=np.intc)
    merged_w = np.bincount(inverse, weights=w_i.astype(np.float64), minlength=len(uniq))
    first = np.zeros(len(uniq), dtype=np.int64)
    first[inverse[::-1]] = np.arange(len(key))[::-1]                      # first occurrence of every pair
    order = np.argsort(first, kind='stable')
    out = np.stack([lo[first], hi[first]], axis=1)[order]
    return np.ascontiguousarray(out, dtype=np.int32), np.ascontiguousarray(np.minimum(merged_w[order], 2 ** 31 - 1), dtype=np.intc)


def cut_general_graph(edges, edge_weights, unary_cost, pairwise_cost, n_iter=-1, algorithm='expansion', init_labels=None,
                      down_weight_factor=None):
    """ drop-in for ``gco.cut_general_graph`` (pyGCO) as the reference calls it (graph_cuts.py:735-744,
    region_growing.py:148,1698): float energies are integerised like pyGCO does, alpha-expansion runs on the GPU.  Edges may come in
    either orientation and more than once (region_growing.py:1433-1444 lists an edge from both of its ends): parallel edges add up.

    :return ndarray: labels int32 [N]
    """
    if algorithm != 'expansion':
        raise NotImplementedError('only algorithm="expansion" is used by the reference hot path')
    eng = get_engine()
    w = np.asarray(edge_weights)
    un = np.asarray(unary_cost)
    pw = np.asarray(pairwise_cost)
    is_float = any(a.dtype.kind == 'f' for a in (w, un, pw))
    if is_float:
        if down_weight_factor is None:
            down_weight_factor = max(np.abs(un).max(), (np.abs(w).max() if w.size else 0.) * pw.max()) + 1e-10
        un_i = (un / down_weight_factor * 100000).astype(np.intc)
        w_i = (w / down_weight_factor * 1000).astype(np.intc)
        pw_i = (pw * 100).astype(np.intc)
    else:
        un_i, w_i, pw_i = un.astype(np.intc), w.astype(np.intc), pw.astype(np.intc)
    edges, w_i = _canonical_int_edges(edges, w_i)
    N, K = un_i.shape
    if len(edges) and int(edges.max()) >= N:
        raise ValueError('an edge refers to vertex %d, the unary table has %d rows' % (int(edges.max()), N))
    E = len(edges)
    d_edges = eng.to_device(edges if E else np.zeros((1, 2), np.int32), 'edges_in')
    d_w = eng.to_device(np.ascontiguousarray(w_i) if E else np.zeros(1, np.intc), 'edge_wi_in')
    d_un = eng.to_device(np.ascontiguousarray(un_i), 'unary_i_in')
    d_pw = eng.to_device(np.ascontiguousarray(pw_i), 'smooth_i_in')
    init = None
    if init_labels is not None:
        init = eng.to_device(np.ascontiguousarray(init_labels, dtype=np.int32), 'init_labels')
    labels, _, _ = eng.alpha_expansion(N, K, E, None, d_edges, d_w, d_un, d_pw, int(n_iter), init)
    return eng.to_host(labels).copy()


def cut_grid_graph(unary_cost, pairwise_cost, cost_v, cost_h, n_iter=-1, algorithm='expansion'):
    """ drop-in for ``gco.cut_grid_graph`` (pyGCO) as the reference calls it (region_growing.py:248): alpha-expansion over the
    4-connected pixel grid, ``cost_v[y, x]`` weighting the edge (y, x)-(y+1, x) and ``cost_h[y, x]`` the edge (y, x)-(y, x+1)

    :param ndarray unary_cost: [H, W, K]
    :return ndarray: labels int32 [H * W]
    """
    unary_cost = np.asarray(unary_cost)
    height, width, nb_labels = unary_cost.shape
    idx = np.arange(height * width).reshape(height, width)
    edges = np.concatenate([np.stack([idx[:-1].ravel(), idx[1:].ravel()], 1), np.stack([idx[:, :-1].ravel(), idx[:, 1:].ravel()], 1)])
    weights = np.concatenate([np.asarray(cost_v, dtype=float).ravel(), np.asarray(cost_h, dtype=float).ravel()])
    return cut_general_graph(edges, weights, unary_cost.reshape(-1, nb_labels), pairwise_cost, n_iter=n_iter, algorithm=algorithm,
                             down_weight_factor=1.0)


def count_label_transitions_connected_segments(dict_slics, dict_labels, nb_labels=None):
    """ label co-occurrence counts over connected segments (reference graph_cuts.py:750-793) """
    if not nb_labels:
        nb_labels = int(max(np.max(lbs) for lbs in dict_labels.values())) + 1
    transitions = np.zeros((nb_labels, nb_labels))
    for name in dict_slics:
        if (np.max(dict_slics[name]) + 1) != len(dict_labels[name]):
            raise ValueError('dims are not matching - max slic (%i) and label (%i)' %
                             (np.max(dict_slics[name]), len(dict_labels[name])))
        _, edges = get_vertexes_edges(dict_slics[name])
        pairs = np.asarray(dict_labels[name])[np.asarray(edges)]
        np.add.at(transitions, (pairs[:, 0], pairs[:, 1]), 1)
        np.add.at(transitions, (pairs[:, 1], pairs[:, 0]), 1)
    transitions[np.diag_indices(nb_labels)] /= 2
    return transitions


def compute_pairwise_cost_from_transitions(trans, min_prob=1e-9):
    """ pairwise cost log(1 / ratio) from the transition counts (reference graph_cuts.py:796-832) """
    trans = np.asarray(trans, dtype=float)
    ratio = trans / np.tile(np.sum(trans, axis=0), (len(trans), 1))
    ratio = np.maximum(ratio, ratio.T) if ratio.ndim == 2 else ratio
    ratio[ratio < min_prob] = min_prob
    return np.log(1. / ratio)
