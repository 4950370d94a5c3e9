"""
RationalQuadratic kernel without a GPU: the oracle's closed-form gradient, the model layer (packing with alpha first, frozen
alpha, persistence, an optimiser run through the checker backend), the device's FP64 log1p and float32 screening covariance
emulated in numpy against their error contracts, the screening error bound of the C library for RQ fits, and the C argument
checks that need no device.
"""
import ctypes

import numpy as np
import pytest
import scipy.linalg as sl

from oracle import gpr_oracle as go
from pygpso_b200 import GPRSurrogate, backend, gpmodel
from tests import rq_oracle as rq
from tests.test_oracle_goldens import make_optimiser, seeded_points
from tests.test_screen_model import VARSIGMA, c_bound, digits_of


def synthetic(N, d, seed=3):
    rng = np.random.default_rng(seed)
    X = rng.random((N, d))
    return X, (np.sin(3 * X.sum(1)) + 0.01 * rng.standard_normal(N))[:, None]


# ---- oracle ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("ard,has_mean", [(False, True), (True, True), (False, False)])
@pytest.mark.parametrize("alpha", [0.3, 2.0, 40.0])
def test_oracle_gradient_matches_finite_differences(ard, has_mean, alpha):
    N, d = 40, 3
    X, y = synthetic(N, d)
    h = rq.RQHyper(alpha, [0.4, 0.6, 0.5] if ard else 0.5, 1.2, 2e-3, 0.15 if has_mean else None)
    u = h.pack()
    n_ls = d if ard else 1
    f, g = rq.neg_lml_and_grad(X, y, u, n_ls, has_mean)
    assert f == pytest.approx(-rq.lml(X, y, h), rel=1e-12)
    for i in range(u.size):
        step = 1e-5 * max(1.0, abs(u[i]))
        up, um = u.copy(), u.copy()
        up[i] += step
        um[i] -= step
        fd = (rq.neg_lml_and_grad(X, y, up, n_ls, has_mean)[0] - rq.neg_lml_and_grad(X, y, um, n_ls, has_mean)[0]) / (2 * step)
        assert abs(g[i] - fd) <= 1e-6 * max(abs(fd), 1.0), (i, g[i], fd)


def test_large_alpha_is_squared_exponential():
    X, _ = synthetic(30, 2)
    Xc = np.random.default_rng(1).random((20, 2))
    h = rq.RQHyper(1e8, 0.4, 1.7, 1e-3)
    k_rq = rq.kern(X, Xc, h)
    k_se = go.kern("SquaredExponential", X, Xc, h)
    assert np.max(np.abs(k_rq - k_se)) <= 1e-6 * h.variance


@pytest.mark.parametrize("u_alpha", [-800.0, -740.0, -720.0])
def test_alpha_underflow(u_alpha):
    """softplus(-800) is exactly 0: k = variance for every pair and a zero alpha entry.  softplus(-740), softplus(-720) are
    subnormal: 0.5 * r2 / alpha overflows for every distinct pair (k = 0 there, as pow(inf, -alpha) in GPflow), k = variance
    on the diagonal; the LML and the gradient stay finite."""
    X, y = synthetic(25, 2)
    h = rq.RQHyper(1.0, 0.4, 1.3, 1e-2, 0.1)
    u = h.pack()
    u[0] = u_alpha
    hz = rq.RQHyper.unpack(u, 1, True)
    K = rq.kern(X, None, hz)
    assert np.all(np.diag(K) == hz.variance)
    if u_alpha == -800.0:
        assert hz.alpha == 0.0 and np.all(K == hz.variance)
    else:
        assert 0.0 < hz.alpha < 2.0 ** -1000 and np.all(K[~np.eye(25, dtype=bool)] == 0.0)
    f, g = rq.neg_lml_and_grad(X, y, u, 1, True)
    assert np.isfinite(f) and np.all(np.isfinite(g))
    assert f == pytest.approx(-rq.lml(X, y, hz), rel=1e-12)
    if u_alpha == -800.0:
        assert g[0] == 0.0


@pytest.mark.parametrize("alpha", [float(go.softplus(-740.0)), float(go.softplus(-720.0)), 2.0 ** -1001, 2.0 ** -999, 1e-300,
                                   1e-3, 0.5, 2.0, 1e8])
def test_device_z_is_gpflows_quotient(alpha):
    """The device's z = (r2 * ia) * sc against GPflow's 0.5 * r2 / alpha: 0 at r2 = 0 for every alpha > 0, within two ulp
    where finite, and overflowing to inf at the same r2 (up to the last ulp of the boundary)."""
    r2 = np.concatenate([[0.0, 5e-324], np.geomspace(1e-300, 1e300, 6001)])
    z = rq.rq_z(r2, alpha)
    with np.errstate(over="ignore"):
        ref = 0.5 * r2 / alpha
    assert z[0] == 0.0
    fin = np.isfinite(ref) & np.isfinite(z) & (ref > 0)
    assert np.all(np.abs(z[fin] - ref[fin]) <= 2.0 * np.spacing(ref[fin]))
    assert np.count_nonzero(np.isinf(z) != np.isinf(ref)) <= 1


# ---- model layer --------------------------------------------------------------------------------------------------------
def model(kernel=None, mean=True, backend_obj=None):
    X, y = synthetic(12, 2)
    kernel = kernel or gpmodel.RationalQuadratic(variance=1.1, lengthscales=0.4, alpha=2.5)
    return gpmodel.GPR((X, y), kernel, gpmodel.Constant(0.2) if mean else None, noise_variance=1e-3,
                       backend=backend_obj or rq.RQOracleBackend())


def test_packing_puts_alpha_first():
    m = model()
    names = [p.name for p in m.trainable_variables]
    assert names == ["kernel.alpha", "kernel.lengthscales", "kernel.variance", "likelihood.variance", "mean_function.c"]
    assert np.array_equal(m._theta(), [2.5, 0.4, 1.1, 1e-3, 0.2])
    h = rq.RQHyper(2.5, 0.4, 1.1, 1e-3, 0.2)
    np.testing.assert_allclose(m._pack(), h.pack(), rtol=1e-14)
    ard = model(gpmodel.RationalQuadratic(lengthscales=[0.3, 0.7]), mean=False)
    assert np.array_equal(ard._theta(), [1.0, 0.3, 0.7, 1.0, 1e-3])
    assert gpmodel.kernels.RationalQuadratic is gpmodel.RationalQuadratic
    assert backend.KERNEL_IDS["RationalQuadratic"] == 4


def test_training_loss_is_the_oracle_objective():
    m = model()
    f_ref, _ = rq.neg_lml_and_grad(*m.data, m._pack(), 1, True)
    assert m.training_loss() == f_ref


def test_frozen_alpha_is_left_alone():
    m = model()
    m.kernel.alpha.trainable = False
    before = m.kernel.alpha.numpy()
    res = gpmodel.Scipy().minimize(m.training_loss, m.trainable_variables)
    assert res.success or res.nit > 0
    assert m.kernel.alpha.numpy() == before
    free = model()
    gpmodel.Scipy().minimize(free.training_loss, free.trainable_variables)
    assert free.kernel.alpha.numpy() != before        # alpha does move when it is trainable


def test_parameter_dict_and_multiple_assign():
    m = model()
    params = gpmodel.parameter_dict(m)
    assert list(params) == [".kernel.alpha", ".kernel.lengthscales", ".kernel.variance", ".likelihood.variance", ".mean_function.c"]
    gpmodel.multiple_assign(m, {".kernel.alpha": 0.7})
    assert m.kernel.alpha.numpy() == 0.7
    assert "GPR.kernel.alpha" in gpmodel.tabulate_module_summary(m)


def test_save_from_saved_round_trips_alpha(tmp_path):
    oracle = rq.RQOracleBackend()
    surr = GPRSurrogate(gp_kernel=gpmodel.RationalQuadratic(lengthscales=0.25, alpha=1.5), gp_meanf=gpmodel.Constant(),
                        points=seeded_points(), backend=oracle)
    x, y = surr.current_training_data
    surr._gp_train(x=x, y=y[:, np.newaxis])
    alpha = surr.gpflow_model.kernel.alpha.numpy()
    assert alpha != 1.5
    surr.save(str(tmp_path / "s"))
    loaded = GPRSurrogate.from_saved(str(tmp_path / "s"), backend=rq.RQOracleBackend())
    assert type(loaded.gpflow_model.kernel) is gpmodel.RationalQuadratic
    assert loaded.gpflow_model.kernel.alpha.numpy().tobytes() == alpha.tobytes()
    assert loaded.gpflow_model._theta().tobytes() == surr.gpflow_model._theta().tobytes()
    a = surr.gpflow_model.predict_y(x)
    b = loaded.gpflow_model.predict_y(x)
    assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1])


def rq_optimiser(backend_obj, depth=3, budget=50):
    opt = make_optimiser(backend=backend_obj, depth=depth, budget=budget)
    default = opt.gp_surr.gp_kernel   # Matern52 of GPRSurrogate.default: the same starting lengthscale and variance
    opt.gp_surr.gp_kernel = gpmodel.RationalQuadratic(lengthscales=default.lengthscales.numpy(), variance=1.0)
    return opt


def test_optimiser_runs_with_the_rq_checker_backend():
    from tests.conftest import paper_objective

    opt = rq_optimiser(rq.RQOracleBackend())
    best = opt.run(paper_objective)
    assert type(opt.gp_surr.gpflow_model.kernel) is gpmodel.RationalQuadratic
    assert opt.n_eval_counter >= 50 and np.isfinite(best.score_mu)
    assert opt.gp_surr.gpflow_model.kernel.alpha.numpy() != 1.0


# ---- device arithmetic, emulated ----------------------------------------------------------------------------------------
def test_log1p_emulation_relative_error():
    z = np.concatenate([[0.0, 5e-324, 1e-300, 1e-30, 1e-17, 2.0 ** -52, 1e-9], np.geomspace(1e-8, 1e300, 20001),
                        np.linspace(0.0, 3.0, 20001), [np.sqrt(2.0) - 1.0, np.nextafter(np.sqrt(2.0) - 1.0, 0.0), 1.0, np.inf]])
    got = rq.log1p_pos(z)
    ref = np.log1p(z)
    assert got[0] == 0.0 and got[-1] == np.inf
    assert np.isnan(rq.log1p_pos(np.array([np.nan])))[0]
    live = (ref > 0) & np.isfinite(ref)
    assert np.max(np.abs(got[live] - ref[live]) / ref[live]) <= 4.0 * np.finfo(np.float64).eps


@pytest.mark.parametrize("alpha", [1e-2, 0.1, 0.5, 1.0, 2.0, 25.0, 1e3, 1e4, 1e6])
def test_cov32_within_the_screen_contract(alpha):
    r2 = np.concatenate([[0.0], np.geomspace(1e-12, 1e3, 40001), np.linspace(0.0, 20.0, 40001)]).astype(np.float32)
    k32 = rq.cov32(r2, 1.7, alpha).astype(np.float64)
    k64 = rq.k_of_r2(r2.astype(np.float64), 1.7, alpha)
    assert k32[0] == np.float32(1.7)
    assert np.max(np.abs(k32 - k64)) <= 2e-6 * 1.7 / 2.0     # half the contract: MUFU.LG2 / EX2 are not emulated
    assert np.isnan(rq.cov32(np.array([np.nan], dtype=np.float32), 1.0, alpha))[0]


def emulate_screen(X, y, h, Xc, S, full):
    """test_screen_model.emulate_screen for the RationalQuadratic kernel."""
    N = X.shape[0]
    K = rq.kern(X, None, h) + h.noise_variance * np.eye(N)
    L = np.linalg.cholesky(K)
    Linv = sl.solve_triangular(L, np.eye(N), lower=True)
    alpha = sl.cho_solve((L, True), y[:, 0] - h.mean_c)
    rowscale = np.ldexp(1.0, np.frexp(np.abs(Linv).max(axis=1))[1])
    beta = np.ldexp(1.0, int(np.floor(np.log2(h.variance))) + 1)
    a = digits_of(np.rint(Linv * (2.0 ** (8 * S - 2) / rowscale)[:, None]), S)
    ls = np.atleast_1d(h.lengthscales)
    diff = (X / ls).astype(np.float32)[:, None, :] - (Xc / ls).astype(np.float32)[None, :, :]
    k32 = rq.cov32(np.einsum("ijk,ijk->ij", diff, diff, dtype=np.float32), h.variance, h.alpha)
    b = digits_of(np.rint(k32.astype(np.float64) * np.float32(2.0 ** (8 * S - 2) / beta)).astype(np.int64), S)
    acc = np.zeros((N, Xc.shape[0]))
    top = 2 * S - 2 if full else S - 1
    for p in range(S):
        for q in range(S if full else S - p):
            acc += (a[p] @ b[q]) * 256.0 ** (top - (p + q))
    gscale = beta * 2.0 ** (-2 * (8 * S - 2) + 8 * (S - 1) - 8 * (top - (S - 1)))
    v = (acc.astype(np.float32) * (rowscale * gscale).astype(np.float32)[:, None]).astype(np.float32)
    var_s = (h.variance - (v * v).astype(np.float32).sum(axis=0, dtype=np.float32).astype(np.float64)) + h.noise_variance
    mean_s = (k32.T @ alpha.astype(np.float32)).astype(np.float64) + h.mean_c
    Ks = rq.kern(X, Xc, h)
    V = Linv @ Ks
    var = (h.variance - (V * V).sum(0)) + h.noise_variance
    mean = Ks.T @ alpha + h.mean_c
    info = {"rho_max": float(rowscale.max()), "rho_l2sq": float((rowscale ** 2).sum()),
            "rowl2_max": float(np.sqrt((Linv ** 2).sum(axis=1)).max()), "frob2": float((Linv ** 2).sum()),
            "alpha_l2": float(np.linalg.norm(alpha)), "k32_err": float(np.abs(k32 - Ks).max())}
    return mean_s, var_s, mean, var, info


@pytest.mark.parametrize("alpha,N,d,ls,noise", [(0.5, 512, 4, 0.5, 1e-3), (2.0, 512, 5, 0.25 * np.sqrt(5), 1e-3),
                                                 (50.0, 640, 3, 0.4, 1e-3), (0.05, 512, 3, 0.3, 2e-6)])
@pytest.mark.parametrize("S,full", [(2, True), (3, False), (4, False)])
def test_screen_error_bound_holds_for_rq(alpha, N, d, ls, noise, S, full):
    rng = np.random.default_rng(20240517)
    X = rng.random((N, d))
    y = (np.sin(3.0 * X.sum(axis=1)) + 0.01 * rng.standard_normal(N))[:, None]
    h = rq.RQHyper(alpha, ls, 1.1, noise, 0.1)
    Xc = np.vstack([rng.random((1500, d)), X[:100] + 1e-5 * rng.standard_normal((100, d))])
    mean_s, var_s, mean, var, info = emulate_screen(X, y, h, Xc, S, full)
    E, e_var, e_mean = c_bound(N, h.variance, noise, info, S, VARSIGMA, full)
    assert info["k32_err"] <= 1.0e-6 * h.variance
    assert np.abs(var_s - var).max() <= e_var / 8.0
    assert np.abs(mean_s - mean).max() <= e_mean / 8.0
    assert np.abs((mean_s + VARSIGMA * var_s) - (mean + VARSIGMA * var)).max() <= E / 8.0


# ---- C argument checks that need no device ------------------------------------------------------------------------------
def test_create_rejects_unknown_kernel_id():
    lib = backend.load_library()
    h = ctypes.c_void_p()
    assert lib.gpso_create(0, 5, 0, 1, ctypes.byref(h)) == -1   # GPSO_E_BADARG before any CUDA call
    assert b"kernel" in lib.gpso_last_error()
    assert lib.gpso_create(0, -1, 0, 1, ctypes.byref(h)) == -1
    assert not h.value
