"""
Linear mean function (gpflow.mean_functions.Linear, m(X) = X A + b) without a GPU: the oracle's closed-form gradient, the model
layer (packing A then b, names, shape checks, frozen A / b, persistence, an optimiser run through the checker backend) and the
C argument checks that need no device.
"""
import ctypes

import numpy as np
import pytest

from oracle import gpr_oracle as go
from pygpso_b200 import GPRSurrogate, backend, gpmodel
from tests import linear_mean_oracle as lo
from tests import rq_oracle as rq
from tests.test_oracle_goldens import make_optimiser, seeded_points


def synthetic(N, d, seed=5):
    rng = np.random.default_rng(seed)
    X = rng.random((N, d))
    return X, (np.sin(3 * X.sum(1)) + 0.7 * X[:, 0] - 0.4 * X[:, -1] + 0.01 * rng.standard_normal(N))[:, None]


def kernel_hyper(kernel, ls):
    return rq.RQHyper(1.7, ls, 1.2, 2e-3) if kernel == rq.KERNEL else go.Hyper(ls, 1.2, 2e-3)


# ---- oracle ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kernel", ["Matern52", "SquaredExponential", "RationalQuadratic"])
@pytest.mark.parametrize("ard", [False, True])
def test_oracle_gradient_matches_finite_differences(kernel, ard):
    N, d = 40, 3
    X, y = synthetic(N, d)
    h = lo.LinearHyper(kernel_hyper(kernel, [0.4, 0.6, 0.5] if ard else 0.5), [0.3, -0.8, 0.5], 0.15)
    u = h.pack()
    n_ls = d if ard else 1
    f, g = lo.neg_lml_and_grad(kernel, X, y, u, n_ls)
    assert f == pytest.approx(-lo.lml(kernel, X, y, h), rel=1e-12)
    assert g.size == u.size
    for i in range(u.size):
        step = 1e-5 * max(1.0, abs(u[i]))
        up, um = u.copy(), u.copy()
        up[i] += step
        um[i] -= step
        fd = (lo.neg_lml_and_grad(kernel, X, y, up, n_ls)[0] - lo.neg_lml_and_grad(kernel, X, y, um, n_ls)[0]) / (2 * step)
        assert abs(g[i] - fd) <= 1e-6 * max(abs(fd), 1.0), (i, g[i], fd)


@pytest.mark.parametrize("kernel", ["Matern52", "RationalQuadratic"])
def test_oracle_linear_zero_is_constant(kernel):
    """A = 0 is the Constant(b) model: same LML, kernel gradient and posterior as the shared oracles."""
    X, y = synthetic(30, 2)
    Xc = np.random.default_rng(2).random((15, 2))
    hk = kernel_hyper(kernel, 0.4)
    h = lo.LinearHyper(hk, [0.0, 0.0], 0.3)
    if kernel == rq.KERNEL:
        hc = rq.RQHyper(hk.alpha, 0.4, hk.variance, hk.noise_variance, 0.3)
        f_c, g_c = rq.neg_lml_and_grad(X, y, hc.pack(), 1, True)
        m_c, v_c = rq.predict_y(X, y, hc, Xc)
    else:
        hc = go.Hyper(0.4, hk.variance, hk.noise_variance, 0.3)
        f_c, g_c = go.neg_lml_and_grad(kernel, X, y, hc.pack(), 1, True)
        m_c, v_c = go.predict_y(kernel, X, y, hc, Xc)
    f, g = lo.neg_lml_and_grad(kernel, X, y, h.pack(), 1)
    assert f == pytest.approx(f_c, rel=1e-13)
    np.testing.assert_allclose(g[:-3], g_c[:-1], rtol=1e-10, atol=1e-12)
    assert g[-1] == pytest.approx(g_c[-1], rel=1e-10)
    m, v = lo.predict_y(kernel, X, y, h, Xc)
    np.testing.assert_allclose(m, m_c, rtol=1e-12, atol=1e-13)
    np.testing.assert_allclose(v, v_c, rtol=1e-12, atol=1e-15)


def test_oracle_extrapolates_linearly():
    """Far from the data the posterior mean is the linear mean itself."""
    X, y = synthetic(30, 2)
    h = lo.LinearHyper(go.Hyper(0.2, 1.0, 1e-3), [2.0, -1.0], 0.5)
    far = np.array([[40.0, -30.0], [-25.0, 12.0]])
    mean, var = lo.predict_y("Matern52", X, y, h, far)
    np.testing.assert_allclose(mean[:, 0], far @ [2.0, -1.0] + 0.5, rtol=1e-14)
    np.testing.assert_allclose(var[:, 0], 1.0 + 1e-3, rtol=1e-14)


# ---- model layer --------------------------------------------------------------------------------------------------------
def model(kernel=None, A=((0.3,), (-0.2,)), b=0.1, backend_obj=None):
    X, y = synthetic(12, 2)
    kernel = kernel or gpmodel.Matern52(variance=1.1, lengthscales=0.4)
    return gpmodel.GPR((X, y), kernel, gpmodel.Linear(np.array(A), np.array([b])), noise_variance=1e-3,
                       backend=backend_obj or lo.LinearOracleBackend())


def test_linear_class_and_defaults():
    assert gpmodel.mean_functions.Linear is gpmodel.Linear
    m = gpmodel.Linear()
    assert m.A.shape.as_list() == [1, 1] and m.A.numpy()[0, 0] == 1.0
    assert m.b.shape.as_list() == [1] and m.b.numpy()[0] == 0.0
    assert not m.A.positive and not m.b.positive
    with pytest.raises(ValueError):
        gpmodel.Linear(np.ones(3))               # not [d, 1]
    with pytest.raises(ValueError):
        gpmodel.Linear(np.ones((3, 2)))          # several outputs
    with pytest.raises(ValueError):
        gpmodel.Linear(np.ones((3, 1)), np.zeros(2))
    X, y = synthetic(10, 3)
    with pytest.raises(ValueError):             # GPflow's default A fits one input dimension only
        gpmodel.GPR((X, y), gpmodel.Matern52(), gpmodel.Linear(), backend=lo.LinearOracleBackend())
    m1 = gpmodel.GPR((X[:, :1], y), gpmodel.Matern52(), gpmodel.Linear(), backend=lo.LinearOracleBackend())
    assert np.array_equal(m1._theta(), [1.0, 1.0, 1.0, 1.0, 0.0])
    m3 = gpmodel.GPR((X, y), gpmodel.Matern52(), gpmodel.Linear(np.zeros((3, 1))), backend=lo.LinearOracleBackend())
    with pytest.raises(ValueError):             # the data setter checks A against new inputs too
        m3.data = (X[:, :2], y)


def test_packing_order_and_names():
    m = model()
    names = [p.name for p in m.trainable_variables]
    assert names == ["kernel.lengthscales", "kernel.variance", "likelihood.variance", "mean_function.A", "mean_function.b"]
    assert np.array_equal(m._theta(), [0.4, 1.1, 1e-3, 0.3, -0.2, 0.1])
    h = lo.LinearHyper(go.Hyper(0.4, 1.1, 1e-3), [0.3, -0.2], 0.1)
    np.testing.assert_allclose(m._pack(), h.pack(), rtol=1e-14)
    rqm = model(gpmodel.RationalQuadratic(lengthscales=[0.3, 0.7], alpha=2.0))
    assert np.array_equal(rqm._theta(), [2.0, 0.3, 0.7, 1.0, 1e-3, 0.3, -0.2, 0.1])
    assert m._session.has_mean == lo.MEAN_ID and type(m._session) is lo.LinearOracleSession
    params = gpmodel.parameter_dict(m)
    assert list(params) == [".kernel.lengthscales", ".kernel.variance", ".likelihood.variance", ".mean_function.A",
                            ".mean_function.b"]
    gpmodel.multiple_assign(m, {".mean_function.A": np.array([[1.5], [2.5]]), ".mean_function.b": np.array([-0.5])})
    assert np.array_equal(m._theta()[-3:], [1.5, 2.5, -0.5])
    summary = gpmodel.tabulate_module_summary(m)
    assert "GPR.mean_function.A" in summary and "GPR.mean_function.b" in summary


def test_training_loss_and_predict_are_the_oracle():
    m = model(gpmodel.RationalQuadratic(lengthscales=0.4, alpha=1.5))
    f_ref, g_ref = lo.neg_lml_and_grad("RationalQuadratic", *m.data, m._pack(), 1)
    f, g = m.neg_log_marginal_likelihood_and_grad(m._pack())
    assert f == f_ref and np.array_equal(g, g_ref)
    xc = np.random.default_rng(0).random((7, 2))
    mean, var = m.predict_y(xc)
    h = lo.LinearHyper(rq.RQHyper(1.5, 0.4, 1.0, 1e-3), [0.3, -0.2], 0.1)
    m_ref, v_ref = lo.predict_y("RationalQuadratic", *m.data, h, xc)
    assert np.array_equal(mean, m_ref) and np.array_equal(var, v_ref)
    mf, cov = m.predict_f(xc, full_cov=True)
    np.testing.assert_allclose(mf[:, 0], mean[:, 0], rtol=1e-12)
    np.testing.assert_allclose(np.diag(cov[0]), var[:, 0] - 1e-3, rtol=1e-10, atol=1e-14)


@pytest.mark.parametrize("frozen", ["A", "b"])
def test_frozen_mean_parameter_is_left_alone(frozen):
    m = model()
    p = getattr(m.mean_function, frozen)
    p.trainable = False
    before = p.numpy().copy()
    other = m.mean_function.b if frozen == "A" else m.mean_function.A
    other_before = other.numpy().copy()
    res = gpmodel.Scipy().minimize(m.training_loss, m.trainable_variables)
    assert res.success or res.nit > 0
    assert np.array_equal(p.numpy(), before)
    assert not np.array_equal(other.numpy(), other_before)   # the trainable one does move


def test_save_from_saved_round_trips_A_and_b(tmp_path):
    oracle = lo.LinearOracleBackend()
    surr = GPRSurrogate(gp_kernel=gpmodel.Matern52(lengthscales=0.25), gp_meanf=gpmodel.Linear(np.zeros((2, 1))),
                        points=seeded_points(), backend=oracle)
    x, y = surr.current_training_data
    surr._gp_train(x=x, y=y[:, np.newaxis])
    A, b = surr.gpflow_model.mean_function.A.numpy(), surr.gpflow_model.mean_function.b.numpy()
    assert np.any(A != 0.0) and b[0] != 0.0
    surr.save(str(tmp_path / "s"))
    loaded = GPRSurrogate.from_saved(str(tmp_path / "s"), backend=lo.LinearOracleBackend())
    mf = loaded.gpflow_model.mean_function
    assert type(mf) is gpmodel.Linear and mf.A.shape.as_list() == [2, 1]
    assert mf.A.numpy().tobytes() == A.tobytes() and mf.b.numpy().tobytes() == b.tobytes()
    assert loaded.gpflow_model._theta().tobytes() == surr.gpflow_model._theta().tobytes()
    p = surr.gpflow_model.predict_y(x)
    q = loaded.gpflow_model.predict_y(x)
    assert np.array_equal(p[0], q[0]) and np.array_equal(p[1], q[1])


def test_optimiser_runs_with_the_linear_checker_backend():
    from tests.conftest import paper_objective

    opt = make_optimiser(backend=lo.LinearOracleBackend(), depth=3, budget=50)
    opt.gp_surr.gp_meanf = gpmodel.Linear(np.zeros((2, 1)))
    best = opt.run(paper_objective)
    mf = opt.gp_surr.gpflow_model.mean_function
    assert type(mf) is gpmodel.Linear
    assert opt.n_eval_counter >= 50 and np.isfinite(best.score_mu)
    assert np.any(mf.A.numpy() != 0.0)


# ---- C argument checks that need no device ------------------------------------------------------------------------------
def test_create_rejects_unknown_mean_id():
    lib = backend.load_library()
    h = ctypes.c_void_p()
    assert lib.gpso_create(0, 2, 0, 3, ctypes.byref(h)) == -1   # GPSO_E_BADARG before any CUDA call
    assert b"mean" in lib.gpso_last_error()
    assert lib.gpso_create(0, 2, 0, -1, ctypes.byref(h)) == -1
    assert not h.value
