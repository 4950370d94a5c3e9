"""
gpflow.kernels.Linear, bare and as a term of a sum, on the B200 against the oracle (tests/linear_kernel_oracle.py) -- run with
``-m gpu``.

Tolerances are those of test_gpu_parity.py: LML 1e-9 * max(|LML|, N), gradient 1e-6 * max(|g|, 1), posterior variance 1e-8 of
the candidate's own prior variance k(x, x) (which varies by orders of magnitude here), mean 1e-8 of the largest of |mean|, |y| and
1.  A handle with a Linear term scores on the FP64 engines only: screen mode 1 returns the unscreened record bit for bit and the
int8 and screening modes are refused.
"""
import numpy as np
import pytest

from oracle import gpr_oracle as go
from pygpso_b200 import backend
from tests import linear_kernel_oracle as lo
from tests import periodic_oracle as pe
from tests import sum_oracle as so
from tests.joint_oracle import sample_mvn
from tests.test_gpu_screen import same_record

pytestmark = pytest.mark.gpu

VARSIGMA = go.VARSIGMA_DEFAULT
JITTER = 1.0e-6
D = 5


@pytest.fixture(scope="module")
def cuda():
    return backend.default_backend()


def synthetic(N, d=D, seed=20240517):
    rng = np.random.default_rng(seed)
    X = rng.random((N, d))
    return X, (np.sin(3 * X.sum(1)) + 0.3 * np.sin(25 * X[:, 0]) + 0.01 * rng.standard_normal(N))[:, None]


# (session kernel, n_lengthscales, components, leaf hypers, column map or None)
CASES = {
    "bare": ("Linear", 1, None, [lo.LinearHyper(0.7)], None),
    "bare_ard": ("Linear", D, None, [lo.LinearHyper([0.5, 0.9, 1.3, 0.4, 0.8])], None),
    "plus_m52": ("Sum", 0, [("Linear", 1), ("Matern52", 1)], [lo.LinearHyper(0.6), so.Comp("Matern52", 0.4, 0.9)], None),
    "three_terms": ("Sum", 0, [("Linear", 1), ("Matern52", 4), ("Periodic", 1, "SquaredExponential", 1)],
                    [lo.LinearHyper(1.1), so.Comp("Matern52", [0.4, 0.5, 0.7, 0.6], 0.8),
                     pe.PeriodicHyper("SquaredExponential", 0.6, 0.7, 0.8, 1.0)], [[0], [1, 2, 3, 4], [D - 1]]),
}


def specs(case):
    kernel, n_ls, components, _, _ = CASES[case]
    return lo.leaves_of(kernel, n_ls, components)


def dims(case, d=D):
    cols = CASES[case][4]
    return cols if cols is not None else [list(range(d))] * len(CASES[case][3])


def hyper(case, mean_id, d=D):
    mean = {0: None, 1: 0.1, 2: (np.linspace(0.5, -0.3, d), 0.05)}[mean_id]
    return lo.Hyper("Sum", CASES[case][3], 2e-3, mean)


def session(cuda, case, X, y, mean_id=1, factorize=True):
    kernel, n_ls, components, _, cols = CASES[case]
    s = cuda.open_session(kernel, n_ls, mean_id, components=components)
    if cols is not None:
        s.set_active_dims(cols)
    s.set_data(X, y)
    if factorize:
        s.factorize(hyper(case, mean_id, X.shape[1]).theta())
    return s


def far_candidates(M, seed):
    """Candidates far outside [0, 1]^d: the prior variance of a Linear term spans orders of magnitude."""
    rng = np.random.default_rng(seed)
    return (rng.random((M, D)) - 0.5) * 10.0 ** rng.integers(-1, 3, size=(M, 1))


def assert_predict_close(h, case, X, y, Xc, mean, var):
    mean_ref, var_ref = lo.predict_y(h, dims(case), X, y, Xc)
    kss = lo.kern_diag(h, dims(case), Xc)
    scale = max(np.abs(mean_ref).max(), np.abs(y).max(), 1.0)
    assert np.all(np.abs(mean - mean_ref[:, 0]) <= 1e-8 * scale)
    assert np.all(np.abs(var - var_ref[:, 0]) <= 1e-8 * np.maximum(kss, 1.0))
    assert np.all(var >= h.noise_variance - 1e-8 * np.maximum(kss, 1.0))
    return mean_ref, var_ref


# ---- LML + gradient ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("N", [1, 129, 1100, 4200])
@pytest.mark.parametrize("case", sorted(CASES))
@pytest.mark.parametrize("mean_id", [0, 1, 2])
def test_neg_lml_and_grad(cuda, case, N, mean_id):
    """1100 rows: the int8 K_y^-1 engine; 4200 rows: the hybrid factorisation."""
    X, y = synthetic(N, seed=N + 3)
    u = hyper(case, mean_id).pack() + 0.03
    kind, sp = specs(case)
    f_ref, g_ref = lo.neg_lml_and_grad(kind, sp, dims(case), X, y, u, mean_id)
    s = session(cuda, case, X, y, mean_id, factorize=False)
    f, g = s.neg_lml_and_grad(u)
    s.close()
    assert abs(f - f_ref) <= 1e-9 * max(abs(f_ref), N), (f, f_ref)
    assert g.shape == g_ref.shape
    assert np.all(np.abs(g - g_ref) <= 1e-6 * np.maximum(np.abs(g_ref), 1.0)), (g, g_ref)


# ---- predict_y, arg-max, top-k, grow --------------------------------------------------------------------------------------
@pytest.mark.parametrize("case", sorted(CASES))
@pytest.mark.parametrize("N,M", [(129, 1000), (1100, 5001)])
def test_predict_y_far_candidates(cuda, case, N, M):
    X, y = synthetic(N)
    h = hyper(case, 1)
    Xc = far_candidates(M, N + M)
    s = session(cuda, case, X, y)
    assert s.predict_info()["engine"] == "fp64-dmma"
    mean, var = s.predict_y(Xc)
    mean_ref, var_ref = assert_predict_close(h, case, X, y, Xc, mean, var)
    idx, m, v, u = s.ucb_argmax(Xc, VARSIGMA)
    assert idx == go.ucb_argmax(mean_ref, var_ref, VARSIGMA)[0]
    assert m == mean[idx] and v == var[idx] and u == mean[idx] + VARSIGMA * var[idx]
    s.close()


@pytest.mark.parametrize("case", ["bare_ard", "three_terms"])
@pytest.mark.parametrize("host", [True, False])
def test_argmax_windows_topk_and_screen_modes(cuda, case, host):
    """Several windows on host and device candidates: the oracle's arg-max, values to 1e-8; top-k in arg-max order; screen mode 1
    is the unscreened record bit for bit with no screen run; modes 2..6 and the int8 predict mode are refused."""
    import torch

    N, M = 1100, 70_000
    X, y = synthetic(N, seed=N)
    h = hyper(case, 1)
    Xc = far_candidates(M, 7)
    xd = torch.from_numpy(Xc).cuda() if not host else None

    def argmax(s):
        if host:
            return s.ucb_argmax(Xc, VARSIGMA)
        return s.ucb_argmax_dev(xd.data_ptr(), M, VARSIGMA, torch.cuda.current_stream().cuda_stream)

    s = session(cuda, case, X, y)
    s.set_window(16_384)
    s.set_screen_mode(0)
    s.factorize(h.theta())
    ref = argmax(s)
    assert s.last_windows() == 5
    mean_ref, var_ref = lo.predict_y(h, dims(case), X, y, Xc)
    ucb_ref = mean_ref[:, 0] + VARSIGMA * var_ref[:, 0]
    assert ref[0] == int(np.argmax(ucb_ref))
    assert abs(ref[3] - ucb_ref[ref[0]]) <= 1e-8 * max(abs(ucb_ref[ref[0]]), 1.0)
    top = s.ucb_topk(Xc, VARSIGMA, 8)
    assert same_record(ref, (int(top[0, 0]), *top[0, 1:]))
    assert list(top[:, 0].astype(int)) == list(np.argsort(-ucb_ref, kind="stable")[:8])
    s.set_screen_mode(1)
    s.factorize(h.theta())
    got = argmax(s)
    assert same_record(ref, got) and s.screen_info()["path"] == "unscreened"
    for mode in range(2, 7):
        with pytest.raises(backend.GpsoBackendError, match="Linear term"):
            s.set_screen_mode(mode)
    with pytest.raises(backend.GpsoBackendError, match="Linear term"):
        s.set_predict_mode(2)
    s.close()


def test_grow_whole_and_by_range(cuda):
    N, depth = 1100, 8
    X, y = synthetic(N, seed=21)
    bounds = np.array([[-3.0, 4.0]] * D)
    s = session(cuda, "three_terms", X, y)
    whole = s.grow_ucb_argmax(bounds, depth, VARSIGMA)
    total = cuda.grow_count(depth)
    cut = total // 3 + 1
    parts = [s.grow_ucb_argmax(bounds, depth, VARSIGMA, rows=(0, cut)), s.grow_ucb_argmax(bounds, depth, VARSIGMA, rows=(cut, total))]
    assert same_record(whole, max(parts, key=lambda r: (r[3], -r[0])))
    leaves = cuda.grow_leaves(bounds, depth)
    mean, var = s.predict_y(leaves)
    assert whole[0] == int(np.argmax(mean + VARSIGMA * var))
    assert whole[1] == mean[whole[0]] and whole[2] == var[whole[0]]
    s.close()


# ---- joint posterior ------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("case,N,M", [("bare", 1, 1), ("bare_ard", 129, 300), ("plus_m52", 700, 1000), ("three_terms", 300, 500)])
def test_predict_f_full_cov(cuda, case, N, M):
    X, y = synthetic(N, seed=N)
    h = hyper(case, 1)
    k = min(N, M // 4)
    Xc = np.vstack([X[:k], far_candidates(M - k, M)])
    s = session(cuda, case, X, y)
    mean, cov = s.predict_f_cov(Xc)
    mean_ref, cov_ref = lo.predict_f_full_cov(h, dims(case), X, y, Xc)
    kss = lo.kern_diag(h, dims(case), Xc)
    bound = 1e-8 * np.maximum(np.sqrt(np.outer(kss, kss)), 1.0)
    assert np.all(np.abs(cov - cov_ref) <= bound)
    assert np.array_equal(cov, cov.T)
    # the diagonal is each candidate's own prior variance minus the explained part: predict_y's variance without the noise
    _, var = s.predict_y(Xc)
    assert np.all(np.abs(np.diag(cov) + h.noise_variance - var) <= 1e-8 * np.maximum(kss, 1.0))
    np.testing.assert_allclose(mean, mean_ref, rtol=0, atol=1e-8 * max(np.abs(mean_ref).max(), np.abs(y).max(), 1.0))
    ms = min(M, 200)
    z = np.random.default_rng(5).standard_normal((3, ms))
    Xs = np.vstack([X[:min(N, ms // 4)], np.random.default_rng(M).random((ms - min(N, ms // 4), D))])
    f = s.predict_f_samples(Xs, z, JITTER)
    f_ref = sample_mvn(*lo.predict_f_full_cov(h, dims(case), X, y, Xs), z, JITTER)
    np.testing.assert_allclose(f, f_ref, rtol=0, atol=1e-5 * max(np.abs(f_ref).max(), 1.0))
    s.close()


# ---- multi-GPU state ------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("case,others", [("bare", [("Matern52", 1, None), ("Linear", D, None)]),
                                         ("plus_m52", [("Sum", 0, [("Matern52", 1), ("Matern52", 1)]),
                                                       ("Sum", 0, [("Linear", D), ("Matern52", 1)])])])
def test_state_export_import(cuda, case, others):
    import torch

    N = 900
    X, y = synthetic(N, seed=41)
    a = session(cuda, case, X, y)
    nbytes = a.state_bytes()
    buf = torch.empty(nbytes, dtype=torch.uint8, device=f"cuda:{cuda.device}")
    a.export_state_dev(buf.data_ptr(), nbytes)
    torch.cuda.synchronize()
    kernel, n_ls, components, _, _ = CASES[case]
    b = cuda.open_session(kernel, n_ls, 1, components=components)
    b.import_state_dev(buf.data_ptr(), nbytes, N, D)
    Xc = far_candidates(20_000, 42)
    assert same_record(b.ucb_argmax(Xc, VARSIGMA), a.ucb_argmax(Xc, VARSIGMA))
    for p, q in zip(a.predict_y(Xc), b.predict_y(Xc)):
        assert p.tobytes() == q.tobytes()
    for p, q in zip(a.predict_f_cov(Xc[:64]), b.predict_f_cov(Xc[:64])):
        assert p.tobytes() == q.tobytes()
    for kernel, n_ls, components in others:   # a non-Linear handle, another variance count: GPSO_E_BADARG either way (a
        other = cuda.open_session(kernel, n_ls, 1, components=components)   # larger layout is refused by its size first)
        with pytest.raises(backend.GpsoBackendError, match=r"status -1\): gpso_import_state_dev: (.*mismatch|source too small)"):
            other.import_state_dev(buf.data_ptr(), nbytes, N, D)
        other.close()
    a.close()
    b.close()


# ---- a Linear leaf alone at d = 1 on the noise floor --------------------------------------------------------------------
def test_rank_one_gram_on_the_noise_floor(cuda):
    """The rank-1 Gram v x x^T plus 1e-6 I: factorises, or fails with the pivot as LinAlgError, as numpy's Cholesky does."""
    X, y = synthetic(200, d=1, seed=3)
    theta = np.array([0.8, go.NOISE_FLOOR, 0.0])
    K = 0.8 * X @ X.T + go.NOISE_FLOOR * np.eye(200)
    try:
        np.linalg.cholesky(K)
        expect_ok = True
    except np.linalg.LinAlgError:
        expect_ok = False
    s = cuda.open_session("Linear", 1, 1)
    s.set_data(X, y)
    if expect_ok:
        s.factorize(theta)
        h = lo.Hyper("Sum", [lo.LinearHyper(0.8)], go.NOISE_FLOOR, 0.0)
        assert s.log_marginal_likelihood() == pytest.approx(lo.lml(h, [[0]], X, y), rel=1e-8)
    else:
        with pytest.raises(np.linalg.LinAlgError):
            s.factorize(theta)
    s.close()
