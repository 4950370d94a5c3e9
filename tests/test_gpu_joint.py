"""
Joint posterior on the B200 (gpso_predict_f_cov_* / gpso_predict_f_samples_*) against the numpy oracle -- run with ``-m gpu``.

Tolerances: covariance entries |d| <= 1e-8 * max(|ref|, kernel variance) (the posterior-variance tolerance of
test_gpu_parity.py; 1e-7 for Matern12, see check_cov), exact symmetry, the mean bit-identical to predict_y's on the FP64 DMMA engine; samples checked against
the factor the call itself used (z = I returns it) and, statistically, against cov + jitter I.
"""
import numpy as np
import pytest

from oracle import gpr_oracle as go
from pygpso_b200 import backend, gpmodel
from tests.joint_oracle import predict_f_full_cov

pytestmark = pytest.mark.gpu

JITTER = gpmodel.SAMPLE_JITTER


@pytest.fixture(scope="module")
def cuda():
    return backend.default_backend()


def synthetic(N, d, seed=20240517):
    rng = np.random.default_rng(seed)
    X = rng.random((N, d))
    y = np.sin(3 * X.sum(1)) + 0.01 * rng.standard_normal(N)
    return X, y[:, None]


def candidates(X, M, seed=11):
    """M candidates, a quarter of them (up to N) copies of training points, where K** - A^T A cancels most."""
    k = min(X.shape[0], M // 4)
    rng = np.random.default_rng(seed)
    return np.ascontiguousarray(np.vstack([X[:k], rng.random((M - k, X.shape[1]))]))


def theta_of(h):
    t = list(np.atleast_1d(h.lengthscales)) + [h.variance, h.noise_variance]
    if h.has_mean:
        t.append(h.mean_c)
    return np.array(t)


def fitted(cuda, kernel, X, y, h, mode=None):
    s = cuda.open_session(kernel, h.lengthscales.size, h.has_mean)
    if mode is not None:
        s.set_predict_mode(*mode)
    s.set_data(X, y)
    s.factorize(theta_of(h))
    return s


def hyper(d, ard, has_mean):
    ls = list(0.25 + 0.1 * np.arange(d)) if ard else 0.3 * np.sqrt(d)
    return go.Hyper(ls, 1.3, 1e-3, 0.1 if has_mean else None)


def check_cov(s, kernel, X, y, h, Xnew):
    mean, cov = s.predict_f_cov(Xnew)
    mean_ref, cov_ref = predict_f_full_cov(kernel, X, y, h, Xnew)
    # Matern12 is not differentiable at r = 0: GPflow's |x|^2 + |x'|^2 - 2 x.x' distance leaves r ~ 1e-8 on the diagonal of
    # K** and between candidates that coincide with training points (k = variance * (1 - 1e-8) there), the kernels take
    # differences first and get r = 0 exactly -- the same 1e-7 allowance test_gpu_parity.py makes for this kernel
    tol = (1e-7 if kernel == "Matern12" else 1e-8) * np.maximum(np.abs(cov_ref), h.variance)
    assert np.all(np.abs(cov - cov_ref) <= tol), float(np.max(np.abs(cov - cov_ref) / tol))
    assert np.array_equal(cov, cov.T)
    np.testing.assert_allclose(mean, mean_ref[:, 0], rtol=0, atol=1e-8 * max(np.abs(y).max(), 1.0))
    _, var = s.predict_y(Xnew)
    var_f = var - h.noise_variance
    assert np.all(np.abs(np.diag(cov) - var_f) <= 1e-8 * np.maximum(np.abs(var_f), h.variance))
    return mean, cov


@pytest.mark.parametrize("N", [1, 6, 129, 700])
@pytest.mark.parametrize("M", [1, 2, 127, 128, 129, 1000])
def test_cov_shapes(cuda, N, M):
    X, y = synthetic(N, 2)
    h = hyper(2, False, True)
    s = fitted(cuda, "Matern52", X, y, h, mode=(1, 0))
    Xnew = candidates(X, M)
    mean, _ = check_cov(s, "Matern52", X, y, h, Xnew)
    mean_y, _ = s.predict_y(Xnew)
    assert np.array_equal(mean, mean_y)  # same cross-covariance kernel, same per-candidate operation sequence
    s.close()


@pytest.mark.parametrize("kernel", ["Matern52", "Matern32", "Matern12", "SquaredExponential"])
@pytest.mark.parametrize("ard,has_mean", [(False, True), (True, True), (False, False), (True, False)])
def test_cov_kernels(cuda, kernel, ard, has_mean):
    d = 3
    X, y = synthetic(300, d, seed=5)
    h = hyper(d, ard, has_mean)
    s = fitted(cuda, kernel, X, y, h, mode=(1, 0))
    Xnew = candidates(X, 257)
    mean, _ = check_cov(s, kernel, X, y, h, Xnew)
    assert np.array_equal(mean, s.predict_y(Xnew)[0])
    s.close()


@pytest.mark.parametrize("M", [129, 1000])
def test_cov_hybrid_factor(cuda, M):
    X, y = synthetic(4097, 2, seed=9)
    h = hyper(2, False, True)
    s = fitted(cuda, "Matern52", X, y, h)
    assert s.factor_info()["schedule"] == "hybrid"
    check_cov(s, "Matern52", X, y, h, candidates(X, M))
    s.close()


def test_cov_largest_batch(cuda):
    X, y = synthetic(300, 2, seed=12)
    h = hyper(2, False, True)
    s = fitted(cuda, "Matern52", X, y, h)
    check_cov(s, "Matern52", X, y, h, candidates(X, backend.MAX_JOINT))
    s.close()


def test_duplicates_are_bit_identical(cuda):
    bounds = np.array([[0.0, 1.0], [0.0, 1.0]])
    leaves = cuda.grow_leaves(bounds, 5)
    _, first, counts = np.unique(leaves, axis=0, return_index=True, return_counts=True)
    assert counts.max() > 1  # the centre child repeats its parent
    X, y = synthetic(200, 2, seed=3)
    s = fitted(cuda, "Matern52", X, y, hyper(2, False, True))
    mean, cov = s.predict_f_cov(leaves)
    for i in range(leaves.shape[0]):
        j = int(np.flatnonzero((leaves == leaves[i]).all(1))[0])
        assert np.array_equal(cov[i], cov[j]) and np.array_equal(cov[:, i], cov[:, j]) and mean[i] == mean[j]
    s.close()


def test_fitted_state_untouched(cuda):
    N = 4096
    X, y = synthetic(N, 3, seed=21)
    h = hyper(3, False, True)
    s = fitted(cuda, "Matern52", X, y, h, mode=(2, 0))
    s.set_screen_mode(1)
    s.factorize(theta_of(h))
    pool = np.random.default_rng(4).random((70000, 3))
    small = pool[:500]

    def state():
        return (s.ucb_argmax(pool, go.VARSIGMA_DEFAULT), s.predict_y(small), s.debug_fetch(1), s.debug_fetch(2), s.debug_fetch(3))

    before = state()
    assert s.screen_info()["path"] != "unscreened"
    s.predict_f_cov(small)
    s.predict_f_samples(small, np.random.default_rng(1).standard_normal((3, 500)), JITTER)
    after = state()
    assert before[0] == after[0]
    for a, b in zip(before[1:], after[1:]):
        for u, v in zip(a if isinstance(a, tuple) else (a,), b if isinstance(b, tuple) else (b,)):
            assert np.array_equal(u, v)
    s.close()


def test_independent_of_predict_mode(cuda):
    X, y = synthetic(700, 2, seed=8)
    h = hyper(2, False, True)
    Xnew = candidates(X, 300)
    z = np.random.default_rng(2).standard_normal((7, 300))
    out = []
    for mode in [(1, 0), (2, 0), (2, 6)]:
        s = fitted(cuda, "Matern52", X, y, h, mode=mode)
        out.append(s.predict_f_cov(Xnew) + (s.predict_f_samples(Xnew, z, JITTER),))
        s.close()
    for other in out[1:]:
        for a, b in zip(out[0], other):
            assert np.array_equal(a, b)


@pytest.mark.parametrize("N,M", [(129, 200), (700, 2048)])
def test_samples_identity_normals_return_the_factor(cuda, N, M):
    X, y = synthetic(N, 2, seed=13)
    h = hyper(2, False, True)
    s = fitted(cuda, "Matern52", X, y, h)
    rng = np.random.default_rng(5)
    Xnew = rng.random((M, 2))
    mean, cov = s.predict_f_cov(Xnew)
    out = s.predict_f_samples(Xnew, np.eye(M), JITTER)
    Lc = (out - mean[None, :]).T
    assert np.all(np.triu(Lc, 1) == 0.0)
    target = cov + JITTER * np.eye(M)
    assert np.max(np.abs(Lc @ Lc.T - target)) <= 1e-12 * h.variance
    z = rng.standard_normal((64, M))
    f = s.predict_f_samples(Xnew, z, JITTER)
    ref = mean[None, :] + z @ Lc.T
    assert np.max(np.abs(f - ref)) <= 1e-12 * np.sqrt(h.variance) * np.sqrt(M) * np.abs(z).max()
    s.close()


def test_samples_empirical_covariance(cuda):
    X, y = synthetic(50, 2, seed=17)
    h = hyper(2, False, True)
    s = fitted(cuda, "Matern52", X, y, h)
    Xnew = np.random.default_rng(6).random((8, 2))
    mean, cov = s.predict_f_cov(Xnew)
    S = 20000
    f = s.predict_f_samples(Xnew, np.random.default_rng(123).standard_normal((S, 8)), JITTER)
    target = cov + JITTER * np.eye(8)
    dev = f - mean[None, :]
    emp = dev.T @ dev / S
    se = np.sqrt((np.outer(np.diag(target), np.diag(target)) + target ** 2) / S)
    assert np.all(np.abs(emp - target) <= 5 * se)
    s.close()


def test_model_layer_on_device(cuda):
    X, y = synthetic(100, 2, seed=19)
    m = gpmodel.GPR((X, y), gpmodel.Matern52(variance=1.3, lengthscales=0.4), gpmodel.Constant(0.1), noise_variance=1e-3)
    Xnew = np.random.default_rng(3).random((50, 2))
    mean, cov = m.predict_f(Xnew, full_cov=True)
    assert mean.shape == (50, 1) and cov.shape == (1, 50, 50)
    f = m.predict_f_samples(Xnew, 4, seed=0)
    assert f.shape == (4, 50, 1)
    np.testing.assert_array_equal(f, m.predict_f_samples(Xnew, 4, seed=0))
    m.close()


def test_launch_count_is_constant(cuda):
    X, y = synthetic(129, 2, seed=23)
    s = fitted(cuda, "Matern52", X, y, hyper(2, False, True))
    steps = []
    for M in (128, backend.MAX_JOINT):
        Xnew = np.random.default_rng(M).random((M, 2))
        c0 = s.launch_count()
        s.predict_f_cov(Xnew)
        c1 = s.launch_count()
        s.predict_f_samples(Xnew, np.random.default_rng(1).standard_normal((1, M)), JITTER)
        steps.append((c1 - c0, s.launch_count() - c1))
    assert steps[0] == steps[1], steps
    s.close()
