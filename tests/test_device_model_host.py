"""Host side of graph_cuts.DeviceClassModel (no GPU): the packed vector of isb_gmm_predict, evaluated by a numpy restatement of the
kernel's arithmetic that reads nothing but that vector, reproduces scikit-learn's predict_proba for every model the reference's
estim_class_model builds without PCA -- GaussianMixture and BayesianGaussianMixture (both weight priors), all four covariance
types, with and without a StandardScaler -- at D = 3, 40 and 189; models the kernel cannot evaluate are refused.

Fitted models at large D classify their own training samples with probabilities of 0 or 1, which would hide a wrong per-component
constant.  The evaluation set therefore also holds points on the model's decision boundaries (between every two component means,
at log-odds -4 .. 4), so that a good share of the probabilities is far from 0 and 1 at every D."""
import functools
import warnings

import numpy as np
import pytest

KINDS = ('gm', 'bgm_process', 'bgm_distribution')
COVARIANCES = ('full', 'tied', 'diag', 'spherical')


def make_data(D, K=3, N=None, seed=0):
    """K classes in D dimensions with per-feature offsets and scales (the scaler has something to do); the noise grows with
    sqrt(D) so that the classes stay about equally far apart in Mahalanobis distance -- far enough for every mixture type to find
    all K of them (the probabilities between them come from boundary_points)"""
    rng = np.random.RandomState(seed + D)
    N = N or max(300, 5 * D)
    centres = rng.normal(0, 3, (K, D))
    y = rng.randint(0, K, N)
    return centres[y] + rng.normal(0, 0.35 * np.sqrt(D), (N, D)) * rng.uniform(0.5, 2, D) + rng.uniform(-5, 5, D)


@functools.lru_cache(maxsize=None)
def fitted_model(kind, covariance, scaler, D, K=3):
    from sklearn import mixture, pipeline, preprocessing
    common = dict(n_components=K, covariance_type=covariance, random_state=0, max_iter=30, reg_covar=1e-2)
    if kind == 'gm':
        mm = mixture.GaussianMixture(**common)
    else:
        mm = mixture.BayesianGaussianMixture(weight_concentration_prior_type='dirichlet_' + kind.split('_')[1],
                                             weight_concentration_prior=10., **common)   # keeps every component populated
    model = pipeline.Pipeline([('std_scaler', preprocessing.StandardScaler()), ('model', mm)]) if scaler else mm
    with warnings.catch_warnings():
        warnings.simplefilter('ignore')
        model.fit(make_data(D, K))
    return model


def boundary_points(model, n_targets=41):
    """points x = m_a + t (m_b - m_a) between every two component means (raw feature space) at which log p_a - log p_b takes the
    values linspace(-4, 4); found by bisection on t where the log-odds cross the target between the two means"""
    from sklearn import pipeline
    mm = model.steps[-1][1] if isinstance(model, pipeline.Pipeline) else model
    means = mm.means_
    if isinstance(model, pipeline.Pipeline):
        means = model.steps[0][1].inverse_transform(means)
    K = len(means)
    pairs = [(a, b) for a in range(K) for b in range(a + 1, K)]
    targets = np.linspace(-4, 4, n_targets)
    A = np.repeat([means[a] for a, _ in pairs], n_targets, 0)
    B = np.repeat([means[b] for _, b in pairs], n_targets, 0)
    ia = np.repeat([a for a, _ in pairs], n_targets)
    ib = np.repeat([b for _, b in pairs], n_targets)
    s = np.tile(targets, len(pairs))

    def f(t):
        p = np.maximum(model.predict_proba(A + t[:, None] * (B - A)), 1e-300)
        rows = np.arange(len(t))
        return np.log(p[rows, ia]) - np.log(p[rows, ib]) - s

    lo, hi = np.zeros(len(s)), np.ones(len(s))
    flo, fhi = f(lo), f(hi)
    ok = np.sign(flo) != np.sign(fhi)
    for _ in range(60):
        mid = 0.5 * (lo + hi)
        fm = f(mid)
        left = np.sign(fm) == np.sign(flo)
        lo, flo = np.where(left, mid, lo), np.where(left, fm, flo)
        hi = np.where(left, hi, mid)
    t = 0.5 * (lo + hi)
    return (A + t[:, None] * (B - A))[ok]


def evaluation_set(model, D, seed=1):
    """150 training-like rows (some entries NaN) + the boundary points"""
    rng = np.random.RandomState(seed)
    X = make_data(D)[:150].copy()
    X[rng.rand(*X.shape) < 0.02] = np.nan
    X[3] = np.nan
    return np.vstack([X, boundary_points(model)])


def kernel_restatement(vec, X, D, K):
    """isb_gmm_predict in numpy, from the packed vector alone: x = (nan -> 0 (f) - shift) / scale, q_k = |x U_k - b_k|^2,
    lw_k = -(D log 2 pi + q_k) / 2 + c_k, proba = softmax(lw)"""
    o = 2 * D
    U = vec[o:o + K * D * D].reshape(K, D, D)
    o += K * D * D
    b = vec[o:o + K * D].reshape(K, D)
    c = vec[o + K * D:o + K * D + K]
    assert len(vec) == o + K * D + K
    x = (np.where(np.isnan(X), 0., X) - vec[:D]) / vec[D:2 * D]
    q = np.stack([np.sum((x @ U[k] - b[k]) ** 2, axis=1) for k in range(K)], 1)
    lw = -0.5 * (D * 1.8378770664093453 + q) + c
    lse = lw.max(1, keepdims=True) + np.log(np.exp(lw - lw.max(1, keepdims=True)).sum(1, keepdims=True))
    return np.exp(lw - lse)


@pytest.mark.parametrize('D', [3, 40, 189])
@pytest.mark.parametrize('scaler', [False, True])
@pytest.mark.parametrize('covariance', COVARIANCES)
@pytest.mark.parametrize('kind', KINDS)
def test_packed_model_reproduces_sklearn(kind, covariance, scaler, D):
    from pyimsegm_b200.graph_cuts import pack_class_model
    model = fitted_model(kind, covariance, scaler, D)
    vec, d, k = pack_class_model(model)
    assert (d, k) == (D, 3) and len(vec) == 2 * D + k * D * D + k * D + k
    X = evaluation_set(model, D)
    want = model.predict_proba(np.nan_to_num(X))
    got = kernel_restatement(vec, X, d, k)
    unsaturated = np.mean((want > 0.05) & (want < 0.95))
    assert unsaturated >= 0.10, 'only %.3f of the probabilities lie in (0.05, 0.95)' % unsaturated
    np.testing.assert_allclose(got, want, rtol=0, atol=1e-12)


def test_scaler_without_mean_or_std():
    from sklearn import mixture, pipeline, preprocessing
    from pyimsegm_b200.graph_cuts import pack_class_model
    X = make_data(5)
    for with_mean, with_std in ((False, True), (True, False), (False, False)):
        model = pipeline.Pipeline([('s', preprocessing.StandardScaler(with_mean=with_mean, with_std=with_std)),
                                   ('m', mixture.GaussianMixture(3, random_state=0))]).fit(X)
        vec, D, K = pack_class_model(model)
        np.testing.assert_allclose(kernel_restatement(vec, X, D, K), model.predict_proba(X), rtol=0, atol=1e-12)


def test_unsupported_models_are_refused():
    from sklearn import decomposition, ensemble, mixture, pipeline, preprocessing
    from pyimsegm_b200.graph_cuts import DeviceClassModel
    X = make_data(4)
    y = (X[:, 0] > np.median(X[:, 0])).astype(int)
    pca = pipeline.Pipeline([('std_scaler', preprocessing.StandardScaler()), ('reduce_dim', decomposition.PCA(3)),
                             ('model', mixture.GaussianMixture(2, random_state=0))]).fit(X)
    with pytest.raises(ValueError, match='reduce_dim'):
        DeviceClassModel(pca)
    with pytest.raises(ValueError, match='RandomForestClassifier'):
        DeviceClassModel(ensemble.RandomForestClassifier(n_estimators=3, random_state=0).fit(X, y))
    with pytest.raises(ValueError, match='K=9'):
        DeviceClassModel(mixture.GaussianMixture(9, covariance_type='diag', random_state=0).fit(make_data(4, K=9, N=400)))
    with pytest.raises(ValueError, match='D=233'):
        DeviceClassModel(mixture.GaussianMixture(2, covariance_type='spherical', random_state=0, max_iter=2).fit(make_data(233, N=300)))
    with pytest.raises(ValueError, match='not fitted'):
        DeviceClassModel(mixture.GaussianMixture(2))


def test_device_class_model_passes_the_model_through():
    """construction needs no GPU; ``classes_`` is there exactly when the wrapped model has it, the digest follows the content"""
    from sklearn import mixture
    from pyimsegm_b200.graph_cuts import DeviceClassModel

    class WithClasses(object):
        pass

    model = fitted_model('gm', 'full', True, 3)
    dcm = DeviceClassModel(model)
    assert dcm.model is model and not hasattr(dcm, 'classes_')
    assert (dcm.n_features, dcm.n_classes) == (3, 3)
    assert DeviceClassModel(model).digest == dcm.digest
    assert DeviceClassModel(fitted_model('gm', 'diag', True, 3)).digest != dcm.digest
    mm = mixture.GaussianMixture(2, random_state=0).fit(make_data(3))
    mm.classes_ = np.array([4, 9])
    assert np.array_equal(DeviceClassModel(mm).classes_, [4, 9])
    with pytest.raises(ValueError, match='WithClasses'):      # any other object is not a mixture
        DeviceClassModel(WithClasses())
