"""
Joint posterior (GPR.predict_f(full_cov=True), GPR.predict_f_samples) without a GPU: the oracle's full covariance, the model
layer on the checker backend, and the argument checks of the four C entry points.
"""
import ctypes
import os

import numpy as np
import pytest

from oracle import gpr_oracle as go
from pygpso_b200 import backend, gpmodel
from tests.joint_oracle import JointOracleBackend, predict_f_full_cov, sample_mvn


def problem(N=40, d=2, seed=3):
    rng = np.random.default_rng(seed)
    X = rng.random((N, d))
    y = np.sin(3 * X.sum(1))[:, None] + 0.01 * rng.standard_normal((N, 1))
    return X, y


def test_oracle_full_cov_matches_predict_y():
    X, y = problem()
    h = go.Hyper(0.3, 1.4, 1e-4, 0.2)
    Xnew = np.vstack([np.random.default_rng(4).random((60, 2)), X[:5]])  # training points: largest cancellation
    mean, cov = predict_f_full_cov("Matern52", X, y, h, Xnew)
    mean_y, var_y = go.predict_y("Matern52", X, y, h, Xnew)
    var_f = var_y[:, 0] - h.noise_variance
    tol = 1e-12 * np.maximum(np.abs(var_f), h.variance)
    assert np.all(np.abs(np.diag(cov) - var_f) <= tol)
    np.testing.assert_allclose(mean, mean_y, rtol=0, atol=1e-12)
    assert np.max(np.abs(cov - cov.T)) <= 1e-12 * h.variance
    assert np.linalg.eigvalsh(0.5 * (cov + cov.T)).min() >= -1e-10 * h.variance


def test_sample_mvn_identity_normals_give_the_factor():
    cov = np.array([[2.0, 0.5], [0.5, 1.0]])
    out = sample_mvn(np.array([1.0, -1.0]), cov, np.eye(2), 0.0)
    np.testing.assert_allclose((out - [1.0, -1.0]).T, np.linalg.cholesky(cov), atol=1e-15)


@pytest.fixture
def model():
    X, y = problem()
    m = gpmodel.GPR((X, y), gpmodel.Matern52(variance=1.4, lengthscales=0.3), gpmodel.Constant(0.2), noise_variance=1e-4,
                    backend=JointOracleBackend())
    return m


def test_predict_f_default_is_unchanged(model):
    Xnew = np.random.default_rng(5).random((17, 2))
    mean, var = model.predict_f(Xnew)
    mean_y, var_y = model.predict_y(Xnew)
    np.testing.assert_array_equal(mean, mean_y)
    np.testing.assert_array_equal(var, var_y - 1e-4)
    assert mean.shape == var.shape == (17, 1)


def test_predict_f_full_cov_shapes(model):
    Xnew = np.random.default_rng(6).random((9, 2))
    mean, cov = model.predict_f(Xnew, full_cov=True)
    assert mean.numpy().shape == (9, 1)
    assert cov.numpy().shape == (1, 9, 9)
    _, var = model.predict_f(Xnew)
    np.testing.assert_allclose(np.diag(cov[0]), var[:, 0], rtol=0, atol=1e-12)
    mean2, cov2 = model.predict_f(Xnew, full_cov=True, full_output_cov=True)
    np.testing.assert_array_equal(cov, cov2)


def test_predict_f_samples_shapes_and_seed(model):
    Xnew = np.random.default_rng(7).random((11, 2))
    f = model.predict_f_samples(Xnew, 5, seed=1)
    assert f.numpy().shape == (5, 11, 1)
    assert model.predict_f_samples(Xnew, seed=1).numpy().shape == (11, 1)
    np.testing.assert_array_equal(f, model.predict_f_samples(Xnew, 5, seed=1))
    assert not np.array_equal(f, model.predict_f_samples(Xnew, 5, seed=2))
    # joint draws: mean + z chol(cov + jitter I)^T with the model's jitter constant
    z = np.random.default_rng(1).standard_normal((5, 11))
    mean, cov = model.predict_f(Xnew, full_cov=True)
    np.testing.assert_allclose(f[:, :, 0], sample_mvn(mean[:, 0], cov[0], z, gpmodel.SAMPLE_JITTER), rtol=0, atol=1e-12)


def test_predict_f_samples_diagonal_is_exact(model):
    Xnew = np.random.default_rng(8).random((13, 2))
    f = model.predict_f_samples(Xnew, 4, full_cov=False, seed=9)
    mean, var = model.predict_f(Xnew)
    z = np.random.default_rng(9).standard_normal((4, 13))
    np.testing.assert_array_equal(f[:, :, 0], mean[:, 0] + np.sqrt(var[:, 0]) * z)


@pytest.mark.parametrize("bad", [np.zeros(3), np.zeros((4, 3)), np.zeros((2, 2, 2))])
def test_bad_candidates_raise(model, bad):
    with pytest.raises(ValueError):
        model.predict_f(bad, full_cov=True)
    with pytest.raises(ValueError):
        model.predict_f_samples(bad, 2)


def test_bad_sample_count_raises(model):
    with pytest.raises(ValueError):
        model.predict_f_samples(np.zeros((3, 2)), 0)


# ---- C entry points: argument checks come before any CUDA call --------------------------------------------------------
@pytest.fixture(scope="module")
def lib():
    if not os.path.exists(backend.library_path()):
        pytest.skip("library not built")
    return backend.load_library()


def _buf(n=8):
    return (ctypes.c_double * n)()


def _cov(lib, h, M):
    b = _buf()
    return lib.gpso_predict_f_cov_host(h, b, M, b, b), lib.gpso_predict_f_cov_dev(h, ctypes.addressof(b), M, ctypes.addressof(b),
                                                                                    ctypes.addressof(b), None)


def _samples(lib, h, M, S, jitter):
    b = _buf()
    return (lib.gpso_predict_f_samples_host(h, b, M, S, jitter, b, b),
            lib.gpso_predict_f_samples_dev(h, ctypes.addressof(b), M, S, jitter, ctypes.addressof(b), ctypes.addressof(b), None))


@pytest.mark.parametrize("M,msg", [(0, b"M must"), (-3, b"M must"), (8193, b"M must"), (4, b"null")])
def test_cov_entry_points_reject_bad_arguments(lib, M, msg):
    for rc in _cov(lib, None, M):
        assert rc == -1  # GPSO_E_BADARG
    assert msg in lib.gpso_last_error()


@pytest.mark.parametrize("M,S,jitter,msg", [(0, 1, 0.0, b"M must"), (8193, 1, 0.0, b"M must"), (4, 0, 0.0, b"null"),
                                            (4, 1, 1e-6, b"null")])
def test_sample_entry_points_reject_bad_sizes_and_null(lib, M, S, jitter, msg):
    for rc in _samples(lib, None, M, S, jitter):
        assert rc == -1
    assert msg in lib.gpso_last_error()


@pytest.mark.parametrize("S,jitter,msg", [(0, 0.0, b"S must"), (-1, 0.0, b"S must"), (2, -1e-6, b"jitter"), (2, float("nan"), b"jitter")])
def test_sample_entry_points_reject_bad_count_and_jitter(lib, S, jitter, msg):
    # a non-null dummy handle: the size checks run before anything touches it
    fake = ctypes.c_void_p(1)
    for rc in _samples(lib, fake, 4, S, jitter):
        assert rc == -1
    assert msg in lib.gpso_last_error()
