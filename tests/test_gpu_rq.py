"""
RationalQuadratic kernel on the B200 against the RQ oracle (tests/rq_oracle.py) -- run with ``-m gpu``.

Tolerances are those of test_gpu_parity.py and test_gpu_joint.py: LML 1e-9 * max(|LML|, N), gradient 1e-6 * max(|g|, 1),
posterior mean / variance and joint covariance 1e-8; the screened arg-max is bit-identical to the unscreened one.
"""
import numpy as np
import pytest

from oracle import gpr_oracle as go
from pygpso_b200 import GPRSurrogate, backend, gpmodel
from tests import rq_oracle as rq
from tests.test_gpu_parity import ENGINES, assert_predict_close
from tests.test_oracle_goldens import seeded_points
from tests.test_rq_kernel import rq_optimiser

pytestmark = pytest.mark.gpu

VARSIGMA = go.VARSIGMA_DEFAULT
KERNEL = "RationalQuadratic"
JITTER = gpmodel.SAMPLE_JITTER


@pytest.fixture(scope="module")
def cuda():
    return backend.default_backend()


def synthetic(N, d, seed=20240517):
    rng = np.random.default_rng(seed)
    X = rng.random((N, d))
    return X, (np.sin(3 * X.sum(1)) + 0.01 * rng.standard_normal(N))[:, None]


def session(cuda, X, y, h, engine=None, factorize=True):
    s = cuda.open_session(KERNEL, h.lengthscales.size, h.has_mean)
    if engine is not None:
        s.set_predict_mode(*ENGINES[engine])
    s.set_data(X, y)
    if factorize:
        s.factorize(h.theta())
    return s


def check_lml_grad(cuda, X, y, h, u):
    n_ls = h.lengthscales.size
    f_ref, g_ref = rq.neg_lml_and_grad(X, y, u, n_ls, h.has_mean)
    s = session(cuda, X, y, h, factorize=False)
    f, g = s.neg_lml_and_grad(u)
    s.close()
    assert abs(f - f_ref) <= 1e-9 * max(abs(f_ref), X.shape[0]), (f, f_ref)
    assert g.shape == g_ref.shape
    assert np.all(np.abs(g - g_ref) <= 1e-6 * np.maximum(np.abs(g_ref), 1.0)), (g, g_ref)
    return f, g


# ---- LML + gradient ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("alpha", [0.3, 1.0, 25.0, 1e4])
@pytest.mark.parametrize("ard,has_mean", [(False, True), (True, True), (False, False)])
def test_neg_lml_and_grad(cuda, alpha, ard, has_mean):
    X, y = synthetic(200, 4, seed=7)
    h = rq.RQHyper(alpha, [0.4, 0.6, 0.5, 0.8] if ard else 0.5, 1.2, 2e-3, 0.15 if has_mean else None)
    check_lml_grad(cuda, X, y, h, h.pack() + 0.05)


@pytest.mark.parametrize("N,d", [(1, 2), (5, 2), (129, 3), (1100, 5), (4200, 6)])
def test_neg_lml_and_grad_sizes(cuda, N, d):
    """1100 rows: the int8 K_y^-1 engine; 4200 rows: the hybrid factorisation."""
    X, y = synthetic(N, d, seed=11)
    h = rq.RQHyper(2.0, 0.3 * np.sqrt(d), 1.1, 1e-3, 0.1)
    check_lml_grad(cuda, X, y, h, h.pack())


@pytest.mark.parametrize("u_alpha", [-800.0, -740.0, -720.0])
def test_alpha_underflow(cuda, u_alpha):
    """alpha = softplus(u_alpha) exactly 0 (-800) or subnormal (-740, -720, where 0.5 / alpha overflows): finite LML and
    gradient equal to the oracle's, and the same posterior."""
    X, y = synthetic(150, 3, seed=5)
    h = rq.RQHyper(1.0, 0.4, 1.3, 1e-2, 0.1)
    u = h.pack()
    u[0] = u_alpha
    f, g = check_lml_grad(cuda, X, y, h, u)
    assert np.isfinite(f) and np.all(np.isfinite(g))
    if u_alpha == -800.0:
        assert g[0] == 0.0
        return
    hz = rq.RQHyper.unpack(u, 1, True)
    s = session(cuda, X, y, hz)
    Xc = np.vstack([X[:20], np.random.default_rng(6).random((300, 3))])
    mean, var = s.predict_y(Xc)
    mean_ref, var_ref = rq.predict_y(X, y, hz, Xc)
    assert_predict_close(mean, var, mean_ref[:, 0], var_ref[:, 0], y, hz.variance)
    _, cov = s.predict_f_cov(Xc[20:])
    assert np.all(np.diag(cov) == hz.variance)   # far from every training point: k(x, x) = variance, k(X, x) = 0
    s.close()


@pytest.mark.parametrize("engine", ["dmma", "int8"])
@pytest.mark.parametrize("alpha", [0.5, 2.0, 25.0, 1e4, 1e8])
def test_device_covariance_relative_accuracy(cuda, engine, alpha):
    """k(x, x') of the device against exp(-alpha log1p(z)) in extended precision, from the same fp64 z: the scalar form
    (crosscov_kernel, FP64 engine) and the W-wide form (crosscov_slices_kernel, int8 engine).  One training point at the
    origin: the posterior mean is k(0, c) * alpha_0 with a single rounding, so the error of log1p_pos (a few ulp relative),
    of E = alpha * log1p and of exp_neg shows directly: |dk / k| <= eps (4 E + 8)."""
    X = np.zeros((1, 1))
    y = np.ones((1, 1))
    h = rq.RQHyper(alpha, 1.0, 1.0, 1e-3, None)
    c = np.concatenate([np.geomspace(1e-6, 1.0, 400), np.linspace(1.0, 60.0, 600)])[:, None]
    s = session(cuda, X, y, h, engine)
    mean, _ = s.predict_y(c)
    a0 = s.debug_fetch(3)[0]
    s.close()
    k = mean / a0
    z = rq.rq_z(np.square(c[:, 0]), alpha)              # the device's r2 and z, bit for bit
    E = np.longdouble(alpha) * np.log1p(z.astype(np.longdouble))
    k_ref = np.exp(-E)
    live = k_ref > 1e-290
    rel = np.abs((k[live] - k_ref[live]) / k_ref[live]).astype(np.float64)
    tol = np.finfo(np.float64).eps * (4.0 * E[live].astype(np.float64) + 8.0)
    assert np.all(rel <= tol), float(np.max(rel / tol))


def test_wrong_parameter_count_is_rejected(cuda):
    X, y = synthetic(20, 2)
    h = rq.RQHyper(1.0, 0.4, 1.0, 1e-3, 0.0)
    s = session(cuda, X, y, h, factorize=False)
    for p in (3, 4):  # n_ls + 2 and n_ls + 2 + 1: the counts of the other kernels
        with pytest.raises(backend.GpsoBackendError, match="hyper-parameters"):
            s.neg_lml_and_grad(np.zeros(p))
        with pytest.raises(backend.GpsoBackendError, match="hyper-parameters"):
            s.factorize(np.ones(p))
    s.close()


# ---- predict_y ------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("N,d,M", [(1, 1, 1), (6, 2, 2), (52, 2, 121), (128, 3, 127), (129, 3, 129), (512, 2, 5000), (1100, 10, 3001)])
@pytest.mark.parametrize("engine", ["dmma", "int8"])
def test_predict_y(cuda, engine, N, d, M):
    X, y = synthetic(N, d)
    h = rq.RQHyper(0.7, 0.25 * np.sqrt(d), 1.0, 1e-3, 0.05)
    Xc = np.random.default_rng(N + M).random((M, d))
    mean_ref, var_ref = rq.predict_y(X, y, h, Xc)
    s = session(cuda, X, y, h, engine)
    mean, var = s.predict_y(Xc)
    assert_predict_close(mean, var, mean_ref[:, 0], var_ref[:, 0], y, h.variance)
    idx, m, v, u = s.ucb_argmax(Xc, VARSIGMA)
    assert idx == go.ucb_argmax(mean_ref, var_ref, VARSIGMA)[0]
    assert m == mean[idx] and v == var[idx] and u == mean[idx] + VARSIGMA * var[idx]
    s.close()


@pytest.mark.parametrize("engine", ["dmma", "int8"])
def test_predict_y_ard_d20(cuda, engine):
    N, d, M = 700, 20, 3000
    X, y = synthetic(N, d, seed=4)
    h = rq.RQHyper(3.0, list(0.6 + 0.05 * np.arange(d)), 1.4, 1e-3, 0.0)
    Xc = np.random.default_rng(9).random((M, d))
    mean_ref, var_ref = rq.predict_y(X, y, h, Xc)
    s = session(cuda, X, y, h, engine)
    mean, var = s.predict_y(Xc)
    assert_predict_close(mean, var, mean_ref[:, 0], var_ref[:, 0], y, h.variance)
    s.close()


# ---- fused arg-max with the screen ----------------------------------------------------------------------------------------
@pytest.mark.parametrize("alpha", [0.5, 2.0, 50.0])
def test_screened_argmax_bit_identical(cuda, alpha):
    N, d, M = 1100, 4, 70_000  # padded N >= 512 and M >= 65 536: the screen takes the call (test_gpu_screen.py's problem)
    X, y = synthetic(N, d, seed=N)
    h = rq.RQHyper(alpha, 0.25 * np.sqrt(d), 1.0, 1e-3, 0.05)
    Xc = np.random.default_rng(M).random((M, d))
    bounds = np.array([[0.0, 1.0]] * d)
    depth = 11                 # grow(11) = 88 573 leaves
    s = session(cuda, X, y, h)
    s.set_screen_mode(0)
    s.factorize(h.theta())
    ref = s.ucb_argmax(Xc, VARSIGMA)
    ref_top = s.ucb_topk(Xc, VARSIGMA, 8)
    ref_grow = s.grow_ucb_argmax(bounds, depth, VARSIGMA)
    dup = np.vstack([Xc, Xc[ref[0]][None, :], Xc[:1000]])
    for mode in (1, 5, 6):
        s.set_screen_mode(mode)
        s.factorize(h.theta())
        assert s.ucb_argmax(Xc, VARSIGMA) == ref, mode
        info = s.screen_info()
        if info["path"] in ("screened", "mean-bound"):
            assert info["max_observed_deviation"] <= info["error_bound"] / 4.0, info
        if mode == 1:             # the ladder needs no full pass here (the forced 2-digit screen of mode 6 may)
            assert info["path"] == "screened", info
        assert np.array_equal(s.ucb_topk(Xc, VARSIGMA, 8), ref_top), mode
        assert s.grow_ucb_argmax(bounds, depth, VARSIGMA) == ref_grow, mode
        assert s.ucb_argmax(dup, VARSIGMA) == ref, mode   # a later duplicate of the winner does not displace it
    s.close()


# ---- joint posterior ------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("N,M,ard,has_mean", [(1, 1, False, True), (129, 300, False, True), (700, 1000, True, False)])
def test_predict_f_full_cov(cuda, N, M, ard, has_mean):
    d = 3
    X, y = synthetic(N, d, seed=N)
    h = rq.RQHyper(1.5, [0.3, 0.5, 0.4] if ard else 0.4, 1.3, 1e-3, 0.1 if has_mean else None)
    k = min(N, M // 4)
    Xc = np.vstack([X[:k], np.random.default_rng(M).random((M - k, d))])
    s = session(cuda, X, y, h)
    mean, cov = s.predict_f_cov(Xc)
    mean_ref, cov_ref = rq.predict_f_full_cov(X, y, h, Xc)
    assert np.all(np.abs(cov - cov_ref) <= 1e-8 * np.maximum(np.abs(cov_ref), h.variance))
    assert np.array_equal(cov, cov.T)
    np.testing.assert_allclose(mean, mean_ref, rtol=0, atol=1e-8 * max(np.abs(y).max(), 1.0))
    s.close()


def test_joint_diagonal_duplicates_and_factor(cuda):
    N, d = 300, 2
    X, y = synthetic(N, d, seed=31)
    h = rq.RQHyper(2.0, 0.3, 1.7, 1e-3, 0.0)
    rng = np.random.default_rng(32)
    far = 1e4 + rng.random((3, d))            # k(X, far) ~ 1e-17: V^T V vanishes below the variance's last bit
    Xc = np.vstack([rng.random((200, d)), far])
    Xc[150:160] = Xc[10:20]
    s = session(cuda, X, y, h)
    mean, cov = s.predict_f_cov(Xc)
    assert np.all(np.diag(cov)[-3:] == h.variance)   # the prior diagonal k(x, x) is exactly the variance
    assert np.array_equal(cov[150:160], cov[10:20]) and np.array_equal(cov[:, 150:160], cov[:, 10:20])
    assert np.array_equal(mean[150:160], mean[10:20])
    M = 120
    Lf = s.predict_f_samples(Xc[:M], np.eye(M), JITTER) - mean[:M][None, :]
    Lc = np.linalg.cholesky(cov[:M, :M] + JITTER * np.eye(M))
    np.testing.assert_allclose(Lf.T, Lc, rtol=0, atol=1e-9)
    s.close()


# ---- multi-GPU state ------------------------------------------------------------------------------------------------------
def test_state_export_import(cuda):
    import torch

    N, d = 900, 4
    X, y = synthetic(N, d, seed=41)
    h = rq.RQHyper(0.8, 0.4, 1.2, 1e-3, 0.1)
    a = session(cuda, X, y, h)
    nbytes = a.state_bytes()
    buf = torch.empty(nbytes, dtype=torch.uint8, device=f"cuda:{cuda.device}")
    a.export_state_dev(buf.data_ptr(), nbytes)
    torch.cuda.synchronize()
    b = cuda.open_session(KERNEL, 1, True)
    b.import_state_dev(buf.data_ptr(), nbytes, N, d)
    Xc = np.random.default_rng(42).random((5000, d))
    assert b.ucb_argmax(Xc, VARSIGMA) == a.ucb_argmax(Xc, VARSIGMA)
    ma, va = a.predict_y(Xc)
    mb, vb = b.predict_y(Xc)
    assert np.array_equal(ma, mb) and np.array_equal(va, vb)
    header = buf[: 16 * 8].cpu().numpy().view(np.float64)
    assert header[8] == h.alpha and header[6] == 4
    mean_b, cov_b = b.predict_f_cov(Xc[:64])   # the joint epilogue reads alpha from the imported header
    mean_a, cov_a = a.predict_f_cov(Xc[:64])
    assert np.array_equal(cov_a, cov_b) and np.array_equal(mean_a, mean_b)
    m52 = cuda.open_session("Matern52", 1, True)
    with pytest.raises(backend.GpsoBackendError, match="kernel mismatch"):
        m52.import_state_dev(buf.data_ptr(), nbytes, N, d)
    for s in (a, b, m52):
        s.close()


# ---- end to end -----------------------------------------------------------------------------------------------------------
def test_surrogate_fit_predict_matches_checker(cuda):
    results = []
    for be in (None, rq.RQOracleBackend()):
        surr = GPRSurrogate(gp_kernel=gpmodel.RationalQuadratic(lengthscales=0.25), gp_meanf=gpmodel.Constant(),
                            points=seeded_points(), backend=be)
        x, y = surr.current_training_data
        surr._gp_train(x=x, y=y[:, np.newaxis])
        results.append((surr.gpflow_model._theta(), surr.gpflow_model.predict_y(np.array([[0.3, 0.7], [0.9, 0.1]]))))
    (tg, (mg, vg)), (to, (mo, vo)) = results
    assert np.all(np.abs(tg - to) <= 1e-6 * np.maximum(np.abs(to), 1.0)), (tg, to)
    np.testing.assert_allclose(mg, mo, rtol=0, atol=1e-8)
    np.testing.assert_allclose(vg, vo, rtol=0, atol=1e-8)


def test_optimiser_same_decisions_as_checker_run():
    from tests.conftest import paper_objective

    runs = []
    for be in (None, rq.RQOracleBackend(rowwise=True)):
        opt = rq_optimiser(be)
        best = opt.run(paper_objective)
        evaluated = [(tuple(np.round(p.normed_coord, 12)), p.score_mu) for p in opt.gp_surr.points if p.label.name == "evaluated"]
        runs.append((opt, best, evaluated))
    (og, bg, eg), (oo, bo, eo) = runs
    assert og.n_eval_counter == oo.n_eval_counter and og.iterations == oo.iterations
    assert [e[0] for e in eg] == [e[0] for e in eo]
    np.testing.assert_array_equal(bg.normed_coord, bo.normed_coord)
    assert bg.score_mu == bo.score_mu
