"""
Parity of the CUDA path (through the C ABI) against the oracle -- run on the B200 box with ``-m gpu``.

Tolerances (SURVEY.md 7.2 / BASELINE.json north_star):
  posterior mean : |d| <= 1e-8 * max(|ref|, max|y|)
  posterior var  : |d| <= 1e-8 * max(|ref|, kernel variance)
  LML            : |d| <= 1e-9 * max(|LML|, N)
  gradient       : |d| <= 1e-6 * max(|ref|, 1)   (it feeds L-BFGS-B, whose own gtol is 1e-5)
  selected candidate (argmax index) and leaf coordinates: identical
"""
import numpy as np
import pytest

from oracle import gpr_oracle as go
from oracle import grow_oracle
from pygpso_b200 import GPRSurrogate, GPSOptimiser, ParameterSpace, backend, gpmodel
from pygpso_b200.optimisation import CallbackTypes
from tests.conftest import paper_objective
from tests.test_oracle_goldens import KATS, TRACE, _Recorder, make_optimiser, seeded_points

pytestmark = pytest.mark.gpu

VARSIGMA = go.VARSIGMA_DEFAULT


def synthetic(N, d, seed=20240517):
    rng = np.random.default_rng(seed)
    X = rng.random((N, d))
    y = np.sin(3 * X.sum(1)) + 0.01 * rng.standard_normal(N)
    return X, y[:, None]


@pytest.fixture(scope="module")
def cuda():
    return backend.default_backend()


# engines of the variance product: FP64 DMMA, and the exact-integer int8 tcgen05 emulation (automatic / forced digits)
ENGINES = {"dmma": (1, 0), "int8": (2, 0), "int8x5": (2, 5), "int8x6": (2, 6), "int8x7": (2, 7), "int8x8": (2, 8)}


def open_session(cuda, kernel, X, y, n_ls=1, has_mean=True, engine=None):
    s = cuda.open_session(kernel, n_ls, has_mean)
    if engine is not None:
        s.set_predict_mode(*ENGINES[engine])
    s.set_data(X, y)
    return s


def theta_of(h):
    t = list(np.atleast_1d(h.lengthscales)) + [h.variance, h.noise_variance]
    if h.has_mean:
        t.append(h.mean_c)
    return np.array(t)


def assert_predict_close(mean, var, mean_ref, var_ref, y, variance, rel=1e-8):
    mtol = rel * np.maximum(np.abs(mean_ref), np.abs(y).max())
    vtol = rel * np.maximum(np.abs(var_ref), variance)
    assert np.all(np.abs(mean - mean_ref) <= mtol), float(np.max(np.abs(mean - mean_ref) / mtol))
    assert np.all(np.abs(var - var_ref) <= vtol), float(np.max(np.abs(var - var_ref) / vtol))


# ---------------------------------------------------------------------------------------------------------------------
# factorisation intermediates
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("N,d", [(1, 1), (6, 2), (127, 3), (128, 2), (129, 2), (300, 5), (700, 10)])
def test_factor_intermediates(cuda, N, d):
    X, y = synthetic(N, d)
    h = go.Hyper(0.25 * np.sqrt(d), 1.3, 1e-3, 0.1)
    s = open_session(cuda, "Matern52", X, y)
    s.factorize(theta_of(h))
    K = go.kern("Matern52", X, None, h) + h.noise_variance * np.eye(N)
    L_ref = np.linalg.cholesky(K)
    L = s.debug_fetch(1)
    np.testing.assert_allclose(L, L_ref, rtol=0, atol=1e-11)
    Linv = s.debug_fetch(2)
    np.testing.assert_allclose(Linv @ L_ref, np.eye(N), rtol=0, atol=1e-8)
    alpha = s.debug_fetch(3)
    alpha_ref = np.linalg.solve(K, y[:, 0] - h.mean_c)
    np.testing.assert_allclose(alpha, alpha_ref, rtol=0, atol=1e-8 * max(1.0, np.abs(alpha_ref).max()))
    lml_ref = go.lml("Matern52", X, y, h)
    assert abs(s.log_marginal_likelihood() - lml_ref) <= 1e-9 * max(abs(lml_ref), N)
    s.close()


# ---------------------------------------------------------------------------------------------------------------------
# LML + gradient (the L-BFGS-B closure)
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kernel", ["Matern52", "Matern32", "Matern12", "SquaredExponential"])
@pytest.mark.parametrize("ard,has_mean", [(False, True), (True, True), (False, False)])
def test_neg_lml_and_grad(cuda, kernel, ard, has_mean):
    N, d = 200, 4
    X, y = synthetic(N, d, seed=7)
    ls = [0.4, 0.6, 0.5, 0.8] if ard else 0.5
    h = go.Hyper(ls, 1.2, 2e-3, 0.15 if has_mean else None)
    u = h.pack() + 0.05
    n_ls = d if ard else 1
    f_ref, g_ref = go.neg_lml_and_grad(kernel, X, y, u, n_ls, has_mean)
    s = open_session(cuda, kernel, X, y, n_ls=n_ls, has_mean=has_mean)
    f, g = s.neg_lml_and_grad(u)
    # Matern12 is not differentiable at r = 0: GPflow's |x|^2+|x'|^2-2x.x' distance leaves ~1e-16 rounding noise on the
    # Gram diagonal, i.e. r ~ 1e-8 and k_ii = variance*(1 - 1e-8) there (the oracle reproduces that artefact), while the
    # CUDA kernels take differences first and get r_ii = 0 exactly.  Any two evaluations of GPflow's formula differ at
    # this level for Matern12, so its tolerance is 1e-7 relative instead of 1e-9; the smooth kernels keep 1e-9.
    ftol, gtol = (1e-7, 1e-4) if kernel == "Matern12" else (1e-9, 1e-6)
    assert abs(f - f_ref) <= ftol * max(abs(f_ref), N), (f, f_ref)
    assert g.shape == g_ref.shape
    assert np.all(np.abs(g - g_ref) <= gtol * np.maximum(np.abs(g_ref), 1.0)), (g, g_ref)
    s.close()


@pytest.mark.parametrize("N,d", [(1, 2), (5, 2), (130, 3), (1000, 10)])
def test_neg_lml_and_grad_sizes(cuda, N, d):
    X, y = synthetic(N, d, seed=11)
    h = go.Hyper(0.25 * np.sqrt(d), 1.0, 1e-3, 0.0)
    u = h.pack()
    f_ref, g_ref = go.neg_lml_and_grad("Matern52", X, y, u, 1, True)
    s = open_session(cuda, "Matern52", X, y)
    f, g = s.neg_lml_and_grad(u)
    assert abs(f - f_ref) <= 1e-9 * max(abs(f_ref), N), (f, f_ref)
    assert np.all(np.abs(g - g_ref) <= 1e-6 * np.maximum(np.abs(g_ref), 1.0)), (g, g_ref)
    kinv = s.debug_fetch(4)
    K = go.kern("Matern52", X, None, h) + h.noise_variance * np.eye(N)
    kinv_ref = np.tril(np.linalg.inv(K))
    np.testing.assert_allclose(kinv, kinv_ref, rtol=0, atol=1e-7 * np.abs(kinv_ref).max())
    s.close()


# ---------------------------------------------------------------------------------------------------------------------
# K_y^-1 = L^-T L^-1 of the gradient: FP64 DMMA tiles against the exact-integer int8 tcgen05 product
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("N,d,noise", [(130, 3, 1e-3), (700, 4, 1e-3), (1100, 5, 1e-3), (2100, 6, 2e-5), (4096, 10, 1e-3)])
def test_kinv_engines_agree(cuda, N, d, noise):
    """The int8 engine (7 digits: 54-bit fixed point per row of L^-T, integer accumulation exact) must reproduce the FP64
    DMMA tiles to the fp64 rounding level of K_y^-1, and the LML gradient must not notice the difference."""
    X, y = synthetic(N, d, seed=5)
    h = go.Hyper(0.25 * np.sqrt(d), 1.1, noise, 0.05)
    u = h.pack()
    out = {}
    for name, mode in (("dmma", 1), ("int8", 2)):
        s = open_session(cuda, "Matern52", X, y)
        s.set_kinv_mode(mode)
        f, g = s.neg_lml_and_grad(u)
        f2, g2 = s.neg_lml_and_grad(u)  # same buffers, second call: deterministic
        assert f2 == f and np.array_equal(g, g2)
        out[name] = (f, g, s.debug_fetch(4))
        s.close()
    (f1, g1, k1), (f2, g2, k2) = out["dmma"], out["int8"]
    assert f1 == f2  # the LML does not depend on K_y^-1
    scale = np.abs(k1).max()
    assert np.abs(k1 - k2).max() <= 2e-12 * scale, np.abs(k1 - k2).max() / scale
    assert np.all(np.abs(g1 - g2) <= 1e-7 * np.maximum(np.abs(g1), 1.0)), (g1, g2)
    if N <= 2100:
        f_ref, g_ref = go.neg_lml_and_grad("Matern52", X, y, u, 1, True)
        assert np.all(np.abs(g2 - g_ref) <= 1e-6 * np.maximum(np.abs(g_ref), 1.0)), (g2, g_ref)
        K = go.kern("Matern52", X, None, h) + h.noise_variance * np.eye(N)
        kinv_ref = np.tril(np.linalg.inv(K))
        np.testing.assert_allclose(k2, kinv_ref, rtol=0, atol=1e-7 * np.abs(kinv_ref).max())


# ---------------------------------------------------------------------------------------------------------------------
# recursive-doubling inverse factor: FP64 DMMA tile tasks against the exact-integer int8 tcgen05 products
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("N,d,noise,persistent", [(200, 2, 1e-3, True), (300, 3, 1e-3, True), (700, 4, 1e-3, False), (1100, 5, 1e-3, True),
                                                  (2100, 6, 2e-5, True), (4096, 10, 1e-3, True)])
def test_inverse_engines_agree(cuda, N, d, noise, persistent):
    """L^-1 from the int8 engine (8 digits: 62-bit fixed point per operand row, exact integer accumulation, two products
    per level) against the DMMA tile tasks: same inverse to fp64 rounding, same LML, same predictions."""
    X, y = synthetic(N, d, seed=3)
    h = go.Hyper(0.25 * np.sqrt(d), 1.2, noise, -0.1)
    theta = theta_of(h)
    Xc = np.random.default_rng(9).random((3000, d))
    out = {}
    for name, mode in (("dmma", 1), ("int8", 2)):
        s = open_session(cuda, "Matern52", X, y)
        s.set_factor_mode(persistent)
        s.set_inverse_mode(mode)
        s.factorize(theta)
        linv = s.debug_fetch(2)
        lml = s.log_marginal_likelihood()
        mean, var = s.predict_y(Xc)
        f, g = s.neg_lml_and_grad(h.pack())
        out[name] = (linv, lml, mean, var, f, g, s.debug_fetch(1))
        s.close()
    a, b = out["dmma"], out["int8"]
    np.testing.assert_array_equal(a[6], b[6])  # the Cholesky factor itself does not depend on the engine
    rowmax = np.abs(a[0]).max(axis=1, keepdims=True)
    assert np.all(np.abs(a[0] - b[0]) <= 1e-11 * rowmax), float((np.abs(a[0] - b[0]) / rowmax).max())
    np.testing.assert_allclose(b[0] @ a[6], np.eye(N), rtol=0, atol=1e-8)
    assert abs(a[1] - b[1]) <= 1e-10 * max(abs(a[1]), N)
    assert_predict_close(b[2], b[3], a[2], a[3], y, h.variance, rel=1e-9)
    assert abs(a[4] - b[4]) <= 1e-10 * max(abs(a[4]), N)
    assert np.all(np.abs(a[5] - b[5]) <= 1e-7 * np.maximum(np.abs(a[5]), 1.0)), (a[5], b[5])
    if N <= 1100:
        lml_ref = go.lml("Matern52", X, y, h)
        assert abs(b[1] - lml_ref) <= 1e-9 * max(abs(lml_ref), N)
        mean_ref, var_ref = go.predict_y("Matern52", X, y, h, Xc)
        assert_predict_close(b[2], b[3], mean_ref[:, 0], var_ref[:, 0], y, h.variance)


# ---------------------------------------------------------------------------------------------------------------------
# the two Cholesky schedules: persistent tile scheduler (default) and one launch per step
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("N,d", [(129, 2), (300, 3), (1100, 5), (2100, 6)])
def test_factor_schedules_agree(cuda, N, d):
    """Persistent dataflow kernel (unblocked updates below 48 panels, fused diagonal update) against the step-by-step
    launches: same factor up to summation order, same LML / gradient well inside the parity tolerances, both against the
    oracle."""
    X, y = synthetic(N, d, seed=3)
    h = go.Hyper(0.25 * np.sqrt(d), 1.1, 1e-3, 0.05)
    u = h.pack()
    out = {}
    for mode in (True, False):
        s = open_session(cuda, "Matern52", X, y)
        s.set_factor_mode(mode)
        f, g = s.neg_lml_and_grad(u)
        s.factorize(theta_of(h))
        out[mode] = (f, g, s.debug_fetch(1), s.debug_fetch(2), s.debug_fetch(3))
        s.close()
    (f1, g1, L1, Li1, a1), (f0, g0, L0, Li0, a0) = out[True], out[False]
    assert abs(f1 - f0) <= 1e-12 * max(abs(f0), N), (f1, f0)
    assert np.all(np.abs(g1 - g0) <= 1e-8 * np.maximum(np.abs(g0), 1.0)), (g1, g0)
    np.testing.assert_allclose(L1, L0, rtol=0, atol=1e-12)
    np.testing.assert_allclose(Li1, Li0, rtol=0, atol=1e-9 * np.abs(Li0).max())
    np.testing.assert_allclose(a1, a0, rtol=0, atol=1e-9 * np.abs(a0).max())
    f_ref, g_ref = go.neg_lml_and_grad("Matern52", X, y, u, 1, True)
    assert abs(f1 - f_ref) <= 1e-9 * max(abs(f_ref), N), (f1, f_ref)
    assert np.all(np.abs(g1 - g_ref) <= 1e-6 * np.maximum(np.abs(g_ref), 1.0)), (g1, g_ref)
    K = go.kern("Matern52", X, None, h) + h.noise_variance * np.eye(N)
    np.testing.assert_allclose(L1, np.linalg.cholesky(K), rtol=0, atol=1e-11)


def test_factor_wide_blocks_large_matrix(cuda):
    """49 panels: the scheduler groups panels in blocks of 4 (K = 512 wide updates, look-ahead across blocks).  LML against
    the oracle (1e-9 relative) and against the step-by-step schedule; L^-1 L = I on a sample of rows."""
    N, d = 6200, 8
    X, y = synthetic(N, d, seed=5)
    h = go.Hyper(0.25 * np.sqrt(d), 1.0, 1e-3, 0.0)
    vals = {}
    for mode in (True, False):
        s = open_session(cuda, "Matern52", X, y)
        s.set_factor_mode(mode)
        s.factorize(theta_of(h))
        vals[mode] = s.log_marginal_likelihood()
        if mode:
            L, Linv = s.debug_fetch(1), s.debug_fetch(2)
        s.close()
    lml_ref = go.lml("Matern52", X, y, h)
    assert abs(vals[True] - lml_ref) <= 1e-9 * max(abs(lml_ref), N), (vals[True], lml_ref)
    assert abs(vals[True] - vals[False]) <= 1e-11 * max(abs(lml_ref), N), vals
    rows = np.random.default_rng(0).integers(0, N, 64)
    np.testing.assert_allclose(Linv[rows] @ L, np.eye(N)[rows], rtol=0, atol=1e-8)


def test_not_positive_definite_under_the_scheduler(cuda):
    """A matrix that loses positive definiteness in a late panel: the persistent kernel must finish (NaNs flow through
    the remaining tasks, nothing waits forever) and report the LAPACK-style pivot."""
    N, d = 600, 2
    X, y = synthetic(N, d, seed=9)
    X[450:] = X[:150]  # 150 exact duplicates and a noise variance far below rounding: K is numerically singular
    s = open_session(cuda, "SquaredExponential", X, y)
    with pytest.raises(np.linalg.LinAlgError) as err:
        s.factorize(np.array([0.5, 1.0, 1.0e-18, 0.0]))
    assert "pivot" in str(err.value)
    s.close()


def test_not_positive_definite_reports_info(cuda):
    y = np.array([[0.0], [1.0], [0.3], [0.5]])
    s = open_session(cuda, "Matern52", np.full((4, 2), np.nan), y)
    with pytest.raises(np.linalg.LinAlgError):
        s.factorize(np.array([0.3, 1.0, 1e-3, 0.0]))
    with pytest.raises(backend.GpsoBackendError):
        s.factorize(np.array([0.3, -1.0, 1e-3, 0.0]))  # bad argument, not a numerical failure
    s.close()


# ---------------------------------------------------------------------------------------------------------------------
# predict_y / UCB argmax
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("N,d,M", [(1, 1, 1), (6, 2, 2), (52, 2, 121), (128, 3, 127), (129, 3, 129), (512, 2, 5000), (1100, 10, 3001)])
@pytest.mark.parametrize("kernel", ["Matern52", "SquaredExponential"])
@pytest.mark.parametrize("engine", ["dmma", "int8"])
def test_predict_y_and_argmax(cuda, engine, kernel, N, d, M):
    X, y = synthetic(N, d)
    h = go.Hyper(0.25 * np.sqrt(d), 1.0, 1e-3, 0.05)
    rng = np.random.default_rng(N + M)
    Xc = rng.random((M, d))
    mean_ref, var_ref = go.predict_y(kernel, X, y, h, Xc)
    s = open_session(cuda, kernel, X, y, engine=engine)
    s.factorize(theta_of(h))
    info = s.predict_info()
    assert info["engine"] == ("fp64-dmma" if engine == "dmma" else "int8-tcgen05")
    mean, var = s.predict_y(Xc)
    assert_predict_close(mean, var, mean_ref[:, 0], var_ref[:, 0], y, h.variance)
    idx_ref, m_ref, v_ref, u_ref = go.ucb_argmax(mean_ref, var_ref, VARSIGMA)
    idx, m, v, u = s.ucb_argmax(Xc, VARSIGMA)
    assert idx == idx_ref
    # the fused argmax path returns exactly what predict_y returns for that candidate
    assert m == mean[idx] and v == var[idx] and u == mean[idx] + VARSIGMA * var[idx]
    s.close()


@pytest.mark.parametrize("engine", ["dmma", "int8"])
def test_ucb_topk_equals_stable_sort_of_predict_y(cuda, engine):
    """gpso_ucb_topk: the k best in arg-max order (descending UCB, lowest index on ties -- duplicated rows included), over
    several windows, with k larger than a window's share and than M."""
    N, d, M = 300, 3, 5000
    X, y = synthetic(N, d, seed=13)
    h = go.Hyper(0.4, 1.1, 1e-3, 0.1)
    s = open_session(cuda, "Matern52", X, y, engine=engine)
    s.factorize(theta_of(h))
    Xc = np.random.default_rng(8).random((M, d))
    Xc[4000:4100] = Xc[100:200]          # exact duplicates in a later window
    s.set_window(1024)                    # several windows even at this size
    mean, var = s.predict_y(Xc)
    ucb = mean + VARSIGMA * var
    for k in (1, 5, 64):
        top = s.ucb_topk(Xc, VARSIGMA, k)
        order = np.lexsort((np.arange(M), -ucb))[:k]
        assert top.shape == (k, 4)
        assert np.array_equal(top[:, 0].astype(int), order)
        assert np.array_equal(top[:, 1], mean[order]) and np.array_equal(top[:, 2], var[order]) and np.array_equal(top[:, 3], ucb[order])
    assert tuple(s.ucb_topk(Xc, VARSIGMA, 1)[0]) == tuple(float(v) for v in s.ucb_argmax(Xc, VARSIGMA))
    few = s.ucb_topk(Xc[:3], VARSIGMA, 8)
    assert few.shape == (3, 4) and sorted(few[:, 0].astype(int)) == [0, 1, 2]
    s.close()


@pytest.mark.parametrize("engine", ["dmma", "int8"])
@pytest.mark.parametrize("d", [1, 20, 33, 64])
def test_predict_input_dimensions(cuda, engine, d):
    """Smallest and largest supported input dimension (the cross-covariance kernels stage d x 128 training coordinates per
    slab in shared memory: 170 KB at d = 64) and an odd one."""
    N, M = 520, 1500
    X, y = synthetic(N, d, seed=21)
    h = go.Hyper(0.3 * np.sqrt(d), 0.9, 1e-3, 0.2)
    s = open_session(cuda, "Matern52", X, y, engine=engine)
    s.factorize(theta_of(h))
    Xc = np.random.default_rng(5).random((M, d))
    mean, var = s.predict_y(Xc)
    mean_ref, var_ref = go.predict_y("Matern52", X, y, h, Xc)
    assert_predict_close(mean, var, mean_ref[:, 0], var_ref[:, 0], y, h.variance)
    assert s.ucb_argmax(Xc, VARSIGMA)[0] == go.ucb_argmax(mean_ref, var_ref, VARSIGMA)[0]
    s.close()


@pytest.mark.parametrize("kernel", ["Matern32", "Matern12"])
def test_predict_other_kernels_ard(cuda, kernel):
    N, d, M = 150, 3, 700
    X, y = synthetic(N, d, seed=5)
    h = go.Hyper([0.3, 0.6, 0.9], 2.0, 5e-3, None)
    Xc = np.random.default_rng(2).random((M, d))
    mean_ref, var_ref = go.predict_y(kernel, X, y, h, Xc)
    s = open_session(cuda, kernel, X, y, n_ls=3, has_mean=False)
    s.factorize(theta_of(h))
    mean, var = s.predict_y(Xc)
    # Matern12 is not differentiable at r = 0: GPflow's |x|^2+|x'|^2-2x.x' distance (restated by the oracle) leaves
    # ~1e-16 rounding noise on the Gram diagonal, i.e. r_ii ~ 1e-8 and k_ii = variance*(1 - 1e-8), while the CUDA kernels
    # take coordinate differences first and get r_ii = 0 exactly.  Two evaluations of GPflow's own formula differ at
    # this level for Matern12 (same note as in test_neg_lml_and_grad); the smooth kernels keep 1e-8.
    assert_predict_close(mean, var, mean_ref[:, 0], var_ref[:, 0], y, h.variance, rel=1e-7 if kernel == "Matern12" else 1e-8)
    s.close()


def test_predict_ill_conditioned_fit(cuda):
    """Fitted hyper-parameters of the README run (noise at its 1e-6 floor, variance ~3): the cancellation case."""
    opt = make_optimiser(backend=None, depth=5, budget=50)  # backend None = CUDA
    opt.run(paper_objective)
    surr = opt.gp_surr
    X, yv = surr.current_training_data
    m = surr.gpflow_model
    h = go.Hyper(float(m.kernel.lengthscales), float(m.kernel.variance), float(m.likelihood.variance), float(m.mean_function.c))
    Xc = grow_oracle.grow_by_level([(0, 1 / 3), (0, 1)], 5)
    mean, var = m.predict_y(Xc)
    mean_ref, var_ref = go.predict_y("Matern52", X, yv[:, None], h, Xc)
    mean_ld, var_ld = go.predict_y_longdouble("Matern52", X, yv[:, None], h, Xc)
    # both implementations against the extended-precision truth, and against each other with the documented tolerance
    err_gpu = np.abs(var.numpy()[:, 0] - var_ld[:, 0].astype(float)).max()
    err_ref = np.abs(var_ref[:, 0] - var_ld[:, 0].astype(float)).max()
    assert err_gpu <= max(10 * err_ref, 1e-9)
    assert_predict_close(mean.numpy()[:, 0], var.numpy()[:, 0], mean_ref[:, 0], var_ref[:, 0], yv, h.variance)


@pytest.mark.parametrize("engine", ["int8x5", "int8x6", "int8x7", "int8x8"])
def test_int8_engine_digit_counts(cuda, engine):
    """Every digit count of the int8 engine against the FP64 DMMA engine on the same factor: the error must shrink with
    the digit count and stay within the estimate reported by the library."""
    N, d, M = 700, 4, 2000
    X, y = synthetic(N, d, seed=3)
    h = go.Hyper(0.5, 1.5, 1e-4, 0.1)
    Xc = np.random.default_rng(9).random((M, d))
    Xc[:50] = X[:50]  # cancellation: variance collapses to ~noise at training points
    ref = open_session(cuda, "Matern52", X, y, engine="dmma")
    ref.factorize(theta_of(h))
    mean_r, var_r = ref.predict_y(Xc)
    s = open_session(cuda, "Matern52", X, y, engine=engine)
    s.factorize(theta_of(h))
    info = s.predict_info()
    assert info["engine"] == "int8-tcgen05" and info["slices"] == ENGINES[engine][1]
    mean, var = s.predict_y(Xc)
    # the mean never goes through the integer product (fp64 FMA in both engines, different summation trees)
    np.testing.assert_allclose(mean, mean_r, rtol=0, atol=1e-12 * max(1.0, np.abs(y).max()))
    err = np.abs(var - var_r).max() / (1e-8 * h.variance)
    assert err <= max(10 * info["error_estimate_over_tol"], 1e-3), (err, info)
    mean_o, var_o = go.predict_y("Matern52", X, y, h, Xc)
    if engine != "int8x5":
        assert_predict_close(mean, var, mean_o[:, 0], var_o[:, 0], y, h.variance)
    ref.close()
    s.close()


def test_int8_engine_automatic_digit_choice(cuda):
    """Well-conditioned factor -> 6 digits; noise at the 1e-6 floor (rows of L^-1 up to ~1e3) -> more digits."""
    N, d = 600, 3
    X, y = synthetic(N, d, seed=4)
    s = open_session(cuda, "Matern52", X, y, engine="int8")
    s.factorize(np.array([0.5, 1.0, 1e-3, 0.0]))
    a = s.predict_info()
    s.factorize(np.array([1.5, 4.0, 1.0e-6 + 5e-8, 0.0]))
    b = s.predict_info()
    assert a["engine"] == b["engine"] == "int8-tcgen05"
    assert 5 <= a["slices"] <= b["slices"] <= 8 and b["slices"] > a["slices"]
    assert a["error_estimate_over_tol"] <= 0.02 and b["error_estimate_over_tol"] <= 0.02
    # the ill-conditioned factor still meets the parity tolerance against the oracle and the long-double truth
    h = go.Hyper(1.5, 4.0, 1.0e-6 + 5e-8, 0.0)
    Xc = np.random.default_rng(5).random((500, d))
    mean, var = s.predict_y(Xc)
    mean_ld, var_ld = go.predict_y_longdouble("Matern52", X, y, h, Xc)
    mean_ref, var_ref = go.predict_y("Matern52", X, y, h, Xc)
    err_gpu = np.abs(var - var_ld[:, 0].astype(float)).max()
    err_ref = np.abs(var_ref[:, 0] - var_ld[:, 0].astype(float)).max()
    assert err_gpu <= max(10 * err_ref, 1e-9 * h.variance), (err_gpu, err_ref)
    s.close()


@pytest.mark.parametrize("engine", ["dmma", "int8"])
def test_duplicates_are_bit_identical_and_first_wins(cuda, engine):
    """Appendix C: exact duplicate rows must give bit-identical UCBs wherever they sit (tiles, windows, shards)."""
    N, d = 300, 3
    X, y = synthetic(N, d)
    h = go.Hyper(0.4, 1.0, 1e-3, 0.0)
    rng = np.random.default_rng(0)
    base = rng.random((40, d))
    Xc = base[rng.integers(0, 40, size=5000)]
    s = open_session(cuda, "Matern52", X, y, engine=engine)
    s.factorize(theta_of(h))
    mean, var = s.predict_y(Xc)
    for b in range(40):
        rows = np.flatnonzero(np.all(Xc == base[b], axis=1))
        assert np.all(mean[rows] == mean[rows[0]]) and np.all(var[rows] == var[rows[0]])
    ucb = mean + VARSIGMA * var
    idx, m, v, u = s.ucb_argmax(Xc, VARSIGMA)
    assert idx == int(np.argmax(ucb)) and u == ucb[idx]
    # window size must not change a single bit
    s.set_window(1024)
    mean2, var2 = s.predict_y(Xc)
    assert np.array_equal(mean, mean2) and np.array_equal(var, var2)
    assert s.ucb_argmax(Xc, VARSIGMA) == (idx, m, v, u)
    # candidates equal to training points: variance collapses to ~noise, mean ~ y
    mt, vt = s.predict_y(X[:50])
    assert np.all(vt < 3 * h.noise_variance) and np.all(vt > 0)
    assert np.abs(mt - y[:50, 0]).max() < 0.05
    s.close()


def test_argmax_numpy_semantics_with_nan(cuda):
    N, d = 20, 2
    X, y = synthetic(N, d)
    s = open_session(cuda, "Matern52", X, y)
    s.factorize(np.array([0.5, 1.0, 1e-3, 0.0]))
    Xc = np.random.default_rng(1).random((300, d))
    Xc[137, 0] = np.nan
    Xc[250, 1] = np.nan
    idx, m, v, u = s.ucb_argmax(Xc, VARSIGMA)
    assert idx == 137 and np.isnan(u)  # np.argmax returns the first NaN
    s.close()


# ---------------------------------------------------------------------------------------------------------------------
# leaf generator
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("d,depth", [(1, 1), (2, 5), (3, 7), (10, 8), (33, 6), (64, 7)])
def test_grow_leaves_bit_exact_small(cuda, d, depth):
    space = ParameterSpace(parameter_bounds=[[0, 1]] * d, parameter_names=[f"p{i}" for i in range(d)])
    child = space.ternary_split()[0]
    got = child.grow(depth)
    assert child.children == ()
    want = grow_oracle.grow_literal(child.norm_bounds, depth)
    assert got.shape == want.shape == ((3 ** depth - 1) // 2, d)
    assert np.array_equal(got, want)


def test_grow_leaves_bit_exact_depth12(cuda):
    space = ParameterSpace(parameter_bounds=[[-5.12, 5.12]] * 10, parameter_names=[f"p{i}" for i in range(10)])
    child = space.ternary_split()[0]
    got = child.grow(12)
    want = grow_oracle.grow_by_level(child.norm_bounds, 12)
    assert got.shape == (265720, 10)
    assert np.array_equal(got, want)


def test_grow_ucb_argmax_equals_two_step_path(cuda):
    N, d = 60, 2
    X, y = synthetic(N, d)
    s = open_session(cuda, "Matern52", X, y)
    s.factorize(np.array([0.25, 1.0, 1e-3, 0.0]))
    bounds = np.array([[1 / 3, 2 / 3], [0.0, 1 / 3]])
    fused = s.grow_ucb_argmax(bounds, 6, VARSIGMA)
    leaves = grow_oracle.grow_by_level(bounds, 6)
    assert fused == s.ucb_argmax(leaves, VARSIGMA)
    mean_ref, var_ref = go.predict_y("Matern52", X, y, go.Hyper(0.25, 1.0, 1e-3, 0.0), leaves)
    assert fused[0] == go.ucb_argmax(mean_ref, var_ref, VARSIGMA)[0]
    s.close()


# ---------------------------------------------------------------------------------------------------------------------
# reference KATs end to end on the GPU
# ---------------------------------------------------------------------------------------------------------------------
def test_fit_predict_kat_on_gpu():
    kat = KATS["fit_predict"]
    surr = GPRSurrogate(gp_kernel=gpmodel.Matern52(), gp_meanf=gpmodel.Constant(), points=seeded_points())
    x, y = surr.current_training_data
    surr._gp_train(x=x, y=y[:, np.newaxis])
    mean, var = surr.gpflow_model.predict_y(np.array(kat["predict_at"]))
    assert float(np.around(mean.numpy(), 8)[0, 0]) == kat["mean_8dp"]
    assert float(np.around(var.numpy(), 8)[0, 0]) == kat["var_8dp"]
    best = surr.gp_eval_best_ucb(np.array(kat["ucb_candidates"]))
    assert float(np.around(best[2], 8)) == np.around(kat["mean_8dp"] + surr.gp_varsigma * kat["var_8dp"], 8)


def test_save_load_predictions_bit_equal(tmp_path):
    surr = GPRSurrogate(gp_kernel=gpmodel.Matern52(), gp_meanf=gpmodel.Constant(), points=seeded_points())
    x, y = surr.current_training_data
    surr._gp_train(x=x, y=y[:, np.newaxis])
    surr.save(str(tmp_path / "s"))
    loaded = GPRSurrogate.from_saved(str(tmp_path / "s"))
    a = surr.gpflow_model.predict_y(x)
    b = loaded.gpflow_model.predict_y(x)
    assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1])
    assert surr.gp_varsigma == loaded.gp_varsigma and surr.gp_lik_sigma == loaded.gp_lik_sigma
    assert list(surr.points) == list(loaded.points)


def test_end_to_end_depth3_on_gpu():
    kat = KATS["end_to_end_depth3"]
    opt = make_optimiser(backend=None, depth=3, budget=50)
    best = opt.run(paper_objective)
    np.testing.assert_almost_equal(np.array(kat["best_coords_7dp"]), best.normed_coord)
    assert np.around(best.score_mu, decimals=8) == kat["best_score_8dp"]
    assert opt.iterations == 13 and opt.n_eval_counter == 55


def test_notebook_trace_depth5_on_gpu():
    iters, fits = [], []
    opt = make_optimiser(backend=None, depth=5, budget=50,
                         callbacks=[_Recorder(CallbackTypes.post_iteration, iters), _Recorder(CallbackTypes.post_update, fits)])
    best = opt.run(paper_objective)
    assert [(i[0], i[1]) for i in iters] == [(w["evaluations"], w["highest_score"]) for w in TRACE["iterations"]]
    for got, want in zip(iters, TRACE["iterations"]):
        assert got[2] == pytest.approx(want["highest_ucb"], abs=5e-9)
    assert best.score_mu == TRACE["best_point"]["score_mu"]
    for got, want in zip(fits, TRACE["hyperparameters_per_update"]):
        for key, value in want.items():
            last_digit = 10.0 ** (np.floor(np.log10(abs(value))) - 5)
            assert abs(got[key] - value) <= 1.0 * last_digit, (key, got[key], value)


def test_end_to_end_sample_method_runs_on_gpu():
    space = ParameterSpace(parameter_names=["x", "y"], parameter_bounds=[[-3, 5], [-3, 3]])
    opt = GPSOptimiser(parameter_space=space, exploration_method="sample", exploration_depth=5, budget=30, n_workers=1)
    best = opt.run(paper_objective, seed=42)
    # only the first sampled child consumes the seed (reference optimisation.py:384), the later sample batches are drawn
    # from fresh entropy: assert what holds for every draw
    evaluated = [p for p in opt.gp_surr.points if p.label.name == "evaluated"]
    assert opt.n_eval_counter >= 30 and len(evaluated) == opt.n_eval_counter
    assert best.score_mu == max(p.score_mu for p in evaluated) >= max(p.score_mu for p in evaluated[:5])
    assert all(np.isfinite(p.score_ucb) for p in opt.gp_surr.points)


def rastrigin_max(point):
    """Config C5 objective: Rastrigin turned into a maximisation problem (domain shifted so that the optimum is not the
    centre of the box, which is always the first point evaluated)."""
    x = np.asarray(point, dtype=np.float64)
    return -(10.0 * x.size + np.sum(x * x - 10.0 * np.cos(2.0 * np.pi * x)))


def _rastrigin_run(backend_obj, d, depth, budget):
    space = ParameterSpace(parameter_names=[f"p{i}" for i in range(d)], parameter_bounds=[[-4.1, 5.12]] * d)
    opt = GPSOptimiser(parameter_space=space, gp_surrogate=GPRSurrogate.default(backend=backend_obj), exploration_method="tree",
                       exploration_depth=depth, budget=budget, stopping_condition="evaluations", update_cycle=1, n_workers=1)
    best = opt.run(rastrigin_max)
    evaluated = [(tuple(np.round(pt.normed_coord, 12)), pt.score_mu) for pt in opt.gp_surr.points if pt.label.name == "evaluated"]
    return opt, best, evaluated


def test_c5_rastrigin_10d_same_decisions_as_oracle_run():
    """Config C5 (10-D Rastrigin, ternary tree) at reduced depth/budget: the optimiser driven by the CUDA library must take
    the same decisions (same evaluated points in the same order, same best point) as the same loop driven by the oracle."""
    from tests.oracle_backend import OracleBackend

    d, depth, budget = 10, 6, 60
    opt_g, best_g, ev_g = _rastrigin_run(None, d, depth, budget)
    opt_o, best_o, ev_o = _rastrigin_run(OracleBackend(), d, depth, budget)
    assert opt_g.n_eval_counter == opt_o.n_eval_counter and opt_g.iterations == opt_o.iterations
    assert [e[0] for e in ev_g] == [e[0] for e in ev_o]
    assert [e[1] for e in ev_g] == [e[1] for e in ev_o]
    np.testing.assert_array_equal(best_g.normed_coord, best_o.normed_coord)
    assert best_g.score_mu == best_o.score_mu


# ---------------------------------------------------------------------------------------------------------------------
# full-size configuration (BASELINE config C3 shape): size-independent properties
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("engine", ["dmma", "int8"])
def test_c3_shape_properties(cuda, engine):
    N, d, M = 4096, 10, 200_000
    X, y = synthetic(N, d)
    theta = np.array([0.25 * np.sqrt(d), 1.0, 1e-3, 0.0])
    s = open_session(cuda, "Matern52", X, y, engine=engine)
    s.factorize(theta)
    Xc = np.random.default_rng([20240517, 0]).random((M, d))
    idx, m, v, u = s.ucb_argmax(Xc, VARSIGMA)
    # (1) shard independence: best over shards (lowest index on ties) equals the global answer bit for bit
    parts = [s.ucb_argmax(Xc[a:a + 50_000], VARSIGMA) for a in range(0, M, 50_000)]
    cand = [(p[3], -(a + p[0]), p) for a, p in zip(range(0, M, 50_000), parts)]
    best = max(cand)
    assert (-best[1], best[2][1:]) == (idx, (m, v, u))
    # (2) permutation: the same candidate wins wherever it sits
    perm = np.random.default_rng(1).permutation(M)
    idx_p, m_p, v_p, u_p = s.ucb_argmax(Xc[perm], VARSIGMA)
    assert perm[idx_p] == idx and (m_p, v_p, u_p) == (m, v, u)
    # (3) the winner agrees with the oracle on a sample that contains it (oracle at full N, 3000 candidates)
    sample = np.unique(np.concatenate([[idx], np.random.default_rng(2).integers(0, M, 2999)]))
    h = go.Hyper(theta[0], theta[1], theta[2], theta[3])
    mean_ref, var_ref = go.predict_y("Matern52", X, y, h, Xc[sample])
    mean_g, var_g = s.predict_y(Xc[sample])
    assert_predict_close(mean_g, var_g, mean_ref[:, 0], var_ref[:, 0], y, theta[1])
    assert sample[go.ucb_argmax(mean_ref, var_ref, VARSIGMA)[0]] == idx
    # (4) variance bounds: noise <= var <= variance + noise
    assert np.all(var_g >= theta[2] * 0.999) and np.all(var_g <= theta[1] + theta[2])
    s.close()
