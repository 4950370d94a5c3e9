"""
Linear mean function (GPSO_MEAN_LINEAR, m(x) = x . A + b) on the B200 against the linear-mean oracle
(tests/linear_mean_oracle.py) -- run with ``-m gpu``.

Tolerances are those of test_gpu_parity.py: LML 1e-9 * max(|LML|, N), gradient 1e-6 * max(|g|, 1), posterior mean / variance
and joint covariance 1e-8.  Screened, windowed, sharded and imported calls return records bit-identical to the plain call, and
Linear(A = 0, b = c) gives the bytes of Constant(c).
"""
import numpy as np
import pytest

from oracle import gpr_oracle as go
from pygpso_b200 import GPRSurrogate, backend, gpmodel
from tests import linear_mean_oracle as lo
from tests import rq_oracle as rq
from tests.test_gpu_parity import ENGINES, assert_predict_close
from tests.test_gpu_screen import same_record
from tests.test_oracle_goldens import seeded_points

pytestmark = pytest.mark.gpu

VARSIGMA = go.VARSIGMA_DEFAULT
JITTER = gpmodel.SAMPLE_JITTER


@pytest.fixture(scope="module")
def cuda():
    return backend.default_backend()


def synthetic(N, d, seed=20240517):
    rng = np.random.default_rng(seed)
    X = rng.random((N, d))
    return X, (np.sin(3 * X.sum(1)) + 0.8 * X[:, 0] - 0.5 * X[:, -1] + 0.01 * rng.standard_normal(N))[:, None]


def hyper(kernel, d, ard=False, A=None, b=0.1, ls=None):
    ls = ls if ls is not None else (list(0.3 + 0.1 * np.arange(d)) if ard else 0.25 * np.sqrt(d))
    hk = rq.RQHyper(1.5, ls, 1.1, 1e-3) if kernel == rq.KERNEL else go.Hyper(ls, 1.1, 1e-3)
    return lo.LinearHyper(hk, np.linspace(0.6, -0.4, d) if A is None else A, b)


def session(cuda, kernel, X, y, h, engine=None, factorize=True):
    s = cuda.open_session(kernel, h.k.lengthscales.size, lo.MEAN_ID)
    if engine is not None:
        s.set_predict_mode(*ENGINES[engine])
    s.set_data(X, y)
    if factorize:
        s.factorize(h.theta())
    return s


def check_lml_grad(cuda, kernel, X, y, h, u):
    n_ls = h.k.lengthscales.size
    f_ref, g_ref = lo.neg_lml_and_grad(kernel, X, y, u, n_ls)
    s = session(cuda, kernel, X, y, h, factorize=False)
    f, g = s.neg_lml_and_grad(u)
    s.close()
    assert abs(f - f_ref) <= 1e-9 * max(abs(f_ref), X.shape[0]), (f, f_ref)
    assert g.shape == g_ref.shape
    assert np.all(np.abs(g - g_ref) <= 1e-6 * np.maximum(np.abs(g_ref), 1.0)), (g, g_ref)


# ---- LML + gradient ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kernel", ["Matern52", "SquaredExponential", "RationalQuadratic"])
@pytest.mark.parametrize("ard", [False, True])
def test_neg_lml_and_grad(cuda, kernel, ard):
    X, y = synthetic(300, 4, seed=7)
    h = hyper(kernel, 4, ard)
    check_lml_grad(cuda, kernel, X, y, h, h.pack() + 0.05)


@pytest.mark.parametrize("kernel,N,d", [("Matern52", 1, 2), ("SquaredExponential", 129, 3), ("Matern52", 1100, 5),
                                        ("RationalQuadratic", 1100, 5), ("Matern52", 4200, 6), ("RationalQuadratic", 4200, 3)])
def test_neg_lml_and_grad_sizes(cuda, kernel, N, d):
    """1100 rows: the int8 K_y^-1 engine; 4200 rows: the hybrid factorisation."""
    X, y = synthetic(N, d, seed=11)
    h = hyper(kernel, d, ard=(d == 3))
    check_lml_grad(cuda, kernel, X, y, h, h.pack())


def test_wrong_parameter_count_is_rejected(cuda):
    X, y = synthetic(20, 2)
    h = hyper("Matern52", 2)
    s = session(cuda, "Matern52", X, y, h, factorize=False)
    for p in (3, 4, 5, 7):  # 1 + 2 + d + 1 = 6; 4 is the Constant count
        with pytest.raises(backend.GpsoBackendError, match="hyper-parameters"):
            s.neg_lml_and_grad(np.zeros(p))
        with pytest.raises(backend.GpsoBackendError, match="hyper-parameters"):
            s.factorize(np.ones(p))
    s.close()


# ---- predict_y ------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kernel,N,d,M", [("Matern52", 1, 1, 1), ("Matern52", 129, 3, 129), ("SquaredExponential", 512, 2, 5000),
                                          ("RationalQuadratic", 1100, 6, 3001)])
@pytest.mark.parametrize("engine", ["dmma", "int8"])
def test_predict_y(cuda, engine, kernel, N, d, M):
    X, y = synthetic(N, d)
    h = hyper(kernel, d)
    rng = np.random.default_rng(N + M)
    far = 30.0 * (rng.random((3, d)) - 0.5) + 20.0   # far outside the box: the linear mean itself
    Xc = np.vstack([rng.random((M, d)), far])
    mean_ref, var_ref = lo.predict_y(kernel, X, y, h, Xc)
    s = session(cuda, kernel, X, y, h, engine)
    mean, var = s.predict_y(Xc)
    assert_predict_close(mean, var, mean_ref[:, 0], var_ref[:, 0], y, h.k.variance)
    if kernel != rq.KERNEL:   # RationalQuadratic's polynomial tail still reaches that far
        np.testing.assert_allclose(mean[-3:], far @ h.A + h.b, rtol=1e-12)
    idx, m, v, u = s.ucb_argmax(Xc, VARSIGMA)
    assert idx == go.ucb_argmax(mean_ref, var_ref, VARSIGMA)[0]
    assert m == mean[idx] and v == var[idx] and u == mean[idx] + VARSIGMA * var[idx]
    s.close()


# ---- Linear(A = 0, b = c) is Constant(c), byte for byte ---------------------------------------------------------------------
@pytest.mark.parametrize("kernel", ["Matern52", "RationalQuadratic"])
def test_zero_slope_is_the_constant_mean(cuda, kernel):
    N, d, M = 1100, 4, 70_000
    X, y = synthetic(N, d, seed=3)
    h = hyper(kernel, d, A=np.zeros(d), b=0.2)
    hk = h.k
    theta_c = np.concatenate([h.theta()[:-(d + 1)], [h.b]])
    u_lin = h.pack() + 0.03
    u_con = np.concatenate([u_lin[:-(d + 1)], u_lin[-1:]])
    u_lin[-(d + 1):-1] = 0.0
    lin = session(cuda, kernel, X, y, h, factorize=False)
    con = cuda.open_session(kernel, hk.lengthscales.size, True)
    con.set_data(X, y)
    f_l, g_l = lin.neg_lml_and_grad(u_lin)
    f_c, g_c = con.neg_lml_and_grad(u_con)
    assert np.array([f_l]).tobytes() == np.array([f_c]).tobytes()
    assert g_l[:-(d + 1)].tobytes() == g_c[:-1].tobytes() and g_l[-1] == g_c[-1]
    lin.factorize(h.theta())
    con.factorize(theta_c)
    Xc = np.random.default_rng(4).random((M, d))
    for a, b in zip(lin.predict_y(Xc), con.predict_y(Xc)):
        assert a.tobytes() == b.tobytes()
    assert same_record(lin.ucb_argmax(Xc, VARSIGMA), con.ucb_argmax(Xc, VARSIGMA))
    for a, b in zip(lin.predict_f_cov(Xc[:300]), con.predict_f_cov(Xc[:300])):
        assert a.tobytes() == b.tobytes()
    lin.close()
    con.close()


# ---- screened arg-max, windows, top-k, grow ---------------------------------------------------------------------------------
@pytest.mark.parametrize("steep", [False, True])
@pytest.mark.parametrize("host", [True, False])
def test_screened_argmax_bit_identical(cuda, host, steep):
    """Screen modes 0-6 with windows of 16384 candidates: the record of mode 0.  The candidates reach past the training data,
    where the mean function takes over; steep: the slope decides the winner (the constant-mean model with the same kernel
    picks another candidate)."""
    import torch

    N, d, M = 1100, 4, 70_000
    X, y = synthetic(N, d, seed=N)
    A = np.array([3.0, -2.0, 1.5, 1.0]) if steep else np.array([0.2, -0.1, 0.05, 0.0])
    h = hyper("Matern52", d, A=A, b=0.05)
    Xc = 1.6 * np.random.default_rng(M).random((M, d)) - 0.3
    xd = torch.from_numpy(Xc).cuda() if not host else None

    def argmax(s):
        if host:
            return s.ucb_argmax(Xc, VARSIGMA)
        return s.ucb_argmax_dev(xd.data_ptr(), M, VARSIGMA, torch.cuda.current_stream().cuda_stream)

    s = session(cuda, "Matern52", X, y, h)
    s.set_screen_mode(0)
    s.factorize(h.theta())
    ref = argmax(s)
    assert ref == s.ucb_argmax(Xc, VARSIGMA)
    top = s.ucb_topk(Xc, VARSIGMA, 8)
    assert same_record(ref, (int(top[0, 0]), *top[0, 1:]))
    if steep:
        con = cuda.open_session("Matern52", 1, True)
        con.set_data(X, y)
        con.factorize(np.concatenate([h.theta()[:-(d + 1)], [h.b]]))
        assert con.ucb_argmax(Xc, VARSIGMA)[0] != ref[0]
        con.close()
    s.set_window(16_384)
    screened = 0
    for mode in range(7):
        s.set_screen_mode(mode)
        s.factorize(h.theta())
        got = argmax(s)
        info = s.screen_info()
        assert same_record(ref, got), (mode, ref, got, info)
        screened += info["path"] in ("screened", "mean-bound")
        if info["path"] in ("screened", "mean-bound"):
            assert info["max_observed_deviation"] <= info["error_bound"] / 4.0, info
    assert screened >= 3
    s.close()


def test_grow_whole_and_by_range(cuda):
    N, d, depth = 1100, 3, 11          # grow(11) = 88 573 leaves
    X, y = synthetic(N, d, seed=21)
    h = hyper("Matern52", d, A=np.array([1.0, -2.0, 0.5]), b=-0.3)
    bounds = np.array([[0.0, 1.0]] * d)
    s = session(cuda, "Matern52", X, y, h)
    whole = s.grow_ucb_argmax(bounds, depth, VARSIGMA)
    total = cuda.grow_count(depth)
    cut = 40_001
    parts = [s.grow_ucb_argmax(bounds, depth, VARSIGMA, rows=(0, cut)), s.grow_ucb_argmax(bounds, depth, VARSIGMA, rows=(cut, total))]
    best = max(parts, key=lambda r: (r[3], -r[0]))
    assert same_record(whole, best)
    leaves = cuda.grow_leaves(bounds, depth)
    mean, var = s.predict_y(leaves)
    assert whole[0] == int(np.argmax(mean + VARSIGMA * var))
    assert whole[1] == mean[whole[0]] and whole[2] == var[whole[0]]
    s.set_screen_mode(0)
    s.factorize(h.theta())
    assert same_record(s.grow_ucb_argmax(bounds, depth, VARSIGMA), whole)
    s.close()


# ---- joint posterior ------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kernel,N,M,ard", [("Matern52", 1, 1, False), ("Matern52", 129, 300, True), ("RationalQuadratic", 700, 1000, False)])
def test_predict_f_full_cov(cuda, kernel, N, M, ard):
    d = 3
    X, y = synthetic(N, d, seed=N)
    h = hyper(kernel, d, ard)
    k = min(N, M // 4)
    Xc = np.vstack([X[:k], np.random.default_rng(M).random((M - k, d))])
    s = session(cuda, kernel, X, y, h, "dmma")
    mean, cov = s.predict_f_cov(Xc)
    mean_ref, cov_ref = lo.predict_f_full_cov(kernel, X, y, h, Xc)
    assert np.all(np.abs(cov - cov_ref) <= 1e-8 * np.maximum(np.abs(cov_ref), h.k.variance))
    assert np.array_equal(cov, cov.T)
    np.testing.assert_allclose(mean, mean_ref, rtol=0, atol=1e-8 * max(np.abs(y).max(), 1.0))
    my, _ = s.predict_y(Xc)
    assert mean.tobytes() == my.tobytes()                         # the DMMA engine's predict_y mean, bit for bit
    draw = s.predict_f_samples(Xc, np.zeros((1, M)), JITTER)[0]
    assert draw.tobytes() == mean.tobytes()
    s.close()


def test_joint_duplicates(cuda):
    N, d = 300, 2
    X, y = synthetic(N, d, seed=31)
    h = hyper("Matern52", d, A=np.array([1.5, -0.7]), b=0.2)
    Xc = np.random.default_rng(32).random((200, d))
    Xc[150:160] = Xc[10:20]
    s = session(cuda, "Matern52", X, y, h)
    mean, cov = s.predict_f_cov(Xc)
    assert np.array_equal(cov[150:160], cov[10:20]) and np.array_equal(cov[:, 150:160], cov[:, 10:20])
    assert mean[150:160].tobytes() == mean[10:20].tobytes()
    f = s.predict_f_samples(Xc, np.random.default_rng(5).standard_normal((3, 200)), JITTER)
    assert np.all(np.isfinite(f))
    s.close()


# ---- multi-GPU state ------------------------------------------------------------------------------------------------------
def test_state_export_import(cuda):
    import torch

    N, d = 900, 4
    X, y = synthetic(N, d, seed=41)
    h = hyper("Matern52", d, A=np.array([0.7, -1.1, 0.3, 0.9]), b=0.1)
    a = session(cuda, "Matern52", X, y, h)
    nbytes = a.state_bytes()
    con = cuda.open_session("Matern52", 1, True)
    con.set_data(X, y)
    con.factorize(np.concatenate([h.theta()[:-(d + 1)], [h.b]]))
    assert nbytes == con.state_bytes() + 8 * d
    buf = torch.empty(nbytes, dtype=torch.uint8, device=f"cuda:{cuda.device}")
    a.export_state_dev(buf.data_ptr(), nbytes)
    torch.cuda.synchronize()
    header = buf[: 16 * 8].cpu().numpy().view(np.float64)
    assert header[9] == lo.MEAN_ID and header[4] == h.b
    b = cuda.open_session("Matern52", 1, lo.MEAN_ID)
    b.import_state_dev(buf.data_ptr(), nbytes, N, d)
    Xc = np.random.default_rng(42).random((70_000, d))
    assert same_record(b.ucb_argmax(Xc, VARSIGMA), a.ucb_argmax(Xc, VARSIGMA))
    ma, va = a.predict_y(Xc)
    mb, vb = b.predict_y(Xc)
    assert np.array_equal(ma, mb) and np.array_equal(va, vb)
    for p, q in zip(a.predict_f_cov(Xc[:64]), b.predict_f_cov(Xc[:64])):
        assert p.tobytes() == q.tobytes()
    # a linear state into a constant-mean handle and the other way round: refused
    with pytest.raises(backend.GpsoBackendError, match="linear mean"):
        cuda.open_session("Matern52", 1, True).import_state_dev(buf.data_ptr(), nbytes, N, d)
    cbytes = con.state_bytes()
    cbuf = torch.empty(nbytes, dtype=torch.uint8, device=f"cuda:{cuda.device}")
    con.export_state_dev(cbuf.data_ptr(), cbytes)
    torch.cuda.synchronize()
    with pytest.raises(backend.GpsoBackendError, match="linear mean"):
        cuda.open_session("Matern52", 1, lo.MEAN_ID).import_state_dev(cbuf.data_ptr(), nbytes, N, d)
    for s in (a, b, con):
        s.close()


# ---- launches ---------------------------------------------------------------------------------------------------------------
def test_launch_count_is_a_fixed_number_more(cuda):
    """Linear: one more launch per fit evaluation for the residual and one for X^T alpha, one per factorisation, one per
    candidate window of every pass, one per joint call; nothing else differs from Constant."""
    N, d, M = 700, 3, 50_000
    X, y = synthetic(N, d, seed=51)
    h = hyper("Matern52", d)
    lin = session(cuda, "Matern52", X, y, h, factorize=False)
    con = cuda.open_session("Matern52", 1, True)
    con.set_data(X, y)
    theta_c = np.concatenate([h.theta()[:-(d + 1)], [h.b]])
    u = h.pack()
    Xc = np.random.default_rng(52).random((M, d))

    def counted(s, call):
        c0 = s.launch_count()
        call(s)
        return s.launch_count() - c0

    assert counted(lin, lambda s: s.neg_lml_and_grad(u)) == counted(con, lambda s: s.neg_lml_and_grad(np.concatenate([u[:-(d + 1)], u[-1:]]))) + 2
    assert counted(lin, lambda s: s.factorize(h.theta())) == counted(con, lambda s: s.factorize(theta_c)) + 1
    for s in (lin, con):
        s.set_window(8192)
    for call in (lambda s: s.predict_y(Xc), lambda s: s.ucb_argmax(Xc, VARSIGMA), lambda s: s.ucb_topk(Xc, VARSIGMA, 4)):
        n_lin = counted(lin, call)
        windows = lin.last_windows()
        n_con = counted(con, call)
        assert con.last_windows() == windows and n_lin == n_con + windows, (n_lin, n_con, windows)
    assert counted(lin, lambda s: s.predict_f_cov(Xc[:500])) == counted(con, lambda s: s.predict_f_cov(Xc[:500])) + 1
    lin.close()
    con.close()


# ---- end to end -----------------------------------------------------------------------------------------------------------
def test_surrogate_fit_predict_matches_checker(cuda):
    results = []
    for be in (None, lo.LinearOracleBackend()):
        surr = GPRSurrogate(gp_kernel=gpmodel.Matern52(lengthscales=0.25), gp_meanf=gpmodel.Linear(np.zeros((2, 1))),
                            points=seeded_points(), backend=be)
        x, y = surr.current_training_data
        surr._gp_train(x=x, y=y[:, np.newaxis])
        results.append((surr.gpflow_model._theta(), surr.gpflow_model.predict_y(np.array([[0.3, 0.7], [0.9, 0.1], [3.0, -2.0]]))))
    (tg, (mg, vg)), (to, (mo, vo)) = results
    assert np.all(np.abs(tg - to) <= 1e-6 * np.maximum(np.abs(to), 1.0)), (tg, to)
    np.testing.assert_allclose(mg, mo, rtol=0, atol=1e-6)
    np.testing.assert_allclose(vg, vo, rtol=0, atol=1e-6)
