"""
Kernels on a subset of the inputs (gpso_set_active_dims) on the B200 against the active-dims oracle (tests/active_dims_oracle.py)
-- run with ``-m gpu``.

Tolerances are those of test_gpu_product_kernel.py: LML 1e-9 * max(|LML|, N), gradient 1e-6 * max(|g|, 1), posterior mean /
variance and joint covariance 1e-8.  Screened, windowed and imported calls return records bit-identical to the plain call, every
screened value lies within E/4 of the exact UCB, candidates that differ only in inactive columns get the same bits, and an
explicit identity map gives the bytes of the handle without a map (the gradient to rounding, see test_identity_map_is_no_map).
"""
import ctypes

import numpy as np
import pytest

from oracle import gpr_oracle as go
from pygpso_b200 import backend
from tests import active_dims_oracle as ad
from tests import periodic_oracle as pe
from tests import rq_oracle as rq
from tests import sum_oracle as so
from tests.test_gpu_parity import ENGINES, assert_predict_close
from tests.test_gpu_screen import same_record

pytestmark = pytest.mark.gpu

VARSIGMA = go.VARSIGMA_DEFAULT
JITTER = 1.0e-6


@pytest.fixture(scope="module")
def cuda():
    return backend.default_backend()


def synthetic(N, d, seed=20240517):
    rng = np.random.default_rng(seed)
    X = rng.random((N, d))
    return X, (np.sin(3 * X.sum(1)) + 0.3 * np.sin(25 * X[:, 0]) + 0.01 * rng.standard_normal(N))[:, None]


def PH(base, ls, var, p, alpha=None):
    return pe.PeriodicHyper(base, ls, var, p, 1.0, alpha=alpha)


# (session kernel, n_lengthscales, components, leaf specs' hypers, column map) on d = 5 inputs
CASES = {
    "m52_subset": ("Matern52", 1, None, [so.Comp("Matern52", 0.4, 0.9)], [[0, 2, 4]]),
    "rq_ard_permuted": (rq.KERNEL, 2, None, [so.Comp(rq.KERNEL, [0.3, 0.6], 0.7, alpha=1.4)], [[3, 0]]),
    "periodic": ("Periodic", 1, [("SquaredExponential", 1)], [PH("SquaredExponential", 0.5, 0.8, 0.7)], [[2]]),
    "periodic_ard": ("Periodic", 1, [("SquaredExponential", 2)], [PH("SquaredExponential", 0.5, 0.8, [0.6, 0.9])], [[1, 3]]),
    "additive": ("Sum", 0, [("Matern52", 2), ("Periodic", 1, rq.KERNEL, 1), ("Matern32", 1)],
                 [so.Comp("Matern52", [0.4, 0.5], 0.6), PH(rq.KERNEL, 0.7, 0.5, 0.8, alpha=1.3), so.Comp("Matern32", 0.5, 0.3)],
                 [[0, 1], [2], [3, 4]]),
    "phase_product": ("Product", 0, [("Matern52", 1), ("Periodic", 1, "SquaredExponential", 1)],
                      [so.Comp("Matern52", 0.5, 0.9), PH("SquaredExponential", 0.6, 1.2, 0.7)], [[0, 1, 2], [3]]),
    "overlap_repeat": ("Product", 0, [("SquaredExponential", 3), ("Periodic", 2, "SquaredExponential", 1)],
                       [so.Comp("SquaredExponential", [0.4, 0.8, 0.5], 0.9), PH("SquaredExponential", [0.6, 0.7], 1.1, 0.9)],
                       [[1, 1, 2], [2, 0]]),
}
D = 5


def hyper(case, mean_id, d=D):
    kernel, n_ls, components, comps, _ = CASES[case]
    kind, _ = ad.leaves_of(kernel, n_ls, components or [(c.family, c.n_ls) for c in comps])
    mean = {0: None, 1: 0.1, 2: (np.linspace(0.5, -0.3, d), 0.05)}[mean_id]
    return pe.CompositeHyper(kind, comps, 2e-3, mean)


def specs(case):
    kernel, n_ls, components, comps, _ = CASES[case]
    return ad.leaves_of(kernel, n_ls, components or [(c.family, c.n_ls) for c in comps])


def open_session(cuda, case, mean_id, dims=None):
    kernel, n_ls, components, comps, cols = CASES[case]
    s = cuda.open_session(kernel, n_ls, mean_id, components=components)
    s.set_active_dims(cols if dims is None else dims)
    return s


def session(cuda, case, X, y, mean_id=1, engine=None, factorize=True):
    s = open_session(cuda, case, mean_id)
    if engine is not None:
        s.set_predict_mode(*ENGINES[engine])
    s.set_data(X, y)
    if factorize:
        s.factorize(hyper(case, mean_id, X.shape[1]).theta())
    return s


# ---- LML + gradient ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("N", [1, 129, 300, 1100, 4200])
@pytest.mark.parametrize("case", sorted(CASES))
def test_neg_lml_and_grad(cuda, case, N):
    """1100 rows: the int8 K_y^-1 engine; 4200 rows: the hybrid factorisation."""
    mean_id = N % 3
    X, y = synthetic(N, D, seed=N + 3)
    h = hyper(case, mean_id)
    u = h.pack() + 0.03
    kind, sp = specs(case)
    f_ref, g_ref = ad.neg_lml_and_grad(kind, sp, CASES[case][4], X, y, u, mean_id)
    s = session(cuda, case, X, y, mean_id, factorize=False)
    f, g = s.neg_lml_and_grad(u)
    s.close()
    assert abs(f - f_ref) <= 1e-9 * max(abs(f_ref), N), (f, f_ref)
    assert g.shape == g_ref.shape
    assert np.all(np.abs(g - g_ref) <= 1e-6 * np.maximum(np.abs(g_ref), 1.0)), (g, g_ref)


# ---- predict_y ------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("case,N,M", [("m52_subset", 129, 129), ("periodic_ard", 512, 5000), ("additive", 1100, 3001),
                                      ("phase_product", 700, 4000), ("overlap_repeat", 300, 1000)])
@pytest.mark.parametrize("engine", ["dmma", "int8"])
def test_predict_y(cuda, engine, case, N, M):
    X, y = synthetic(N, D)
    h = hyper(case, 1)
    Xc = np.random.default_rng(N + M).random((M, D))
    mean_ref, var_ref = ad.predict_y(h, CASES[case][4], X, y, Xc)
    s = session(cuda, case, X, y, engine=engine)
    assert s.predict_info()["engine"] == ("fp64-dmma" if engine == "dmma" else "int8-tcgen05")
    mean, var = s.predict_y(Xc)
    assert_predict_close(mean, var, mean_ref[:, 0], var_ref[:, 0], y, h.prior_variance, rel=1e-8)
    idx, m, v, u = s.ucb_argmax(Xc, VARSIGMA)
    assert idx == go.ucb_argmax(mean_ref, var_ref, VARSIGMA)[0]
    assert m == mean[idx] and v == var[idx] and u == mean[idx] + VARSIGMA * var[idx]
    s.close()


# ---- an explicit identity map is no map ------------------------------------------------------------------------------------
@pytest.mark.parametrize("case", ["m52_subset", "rq_ard_permuted", "periodic_ard", "additive", "phase_product"])
def test_identity_map_is_no_map(cuda, case):
    """The map 0..d-1 on every leaf against the same handle without a map.  A bare kernel with a map runs as a one-component
    sum (composite row layout), so its gradient sums the same terms in another order where the layouts' reductions differ (the
    ARD and periodic gradients): rounding apart, 1e-9 relative.  The LML, the records of screen modes 0, 1 and 5 and predict_y
    are the same bytes."""
    N, d, M = 1100, 2, 70_000
    X, y = synthetic(N, d, seed=5)
    kernel, n_ls, components, comps, cols = CASES[case]
    h = hyper(case, 1, d)
    ident = [list(range(d))] * len(cols)
    mapped = cuda.open_session(kernel, n_ls, 1, components=components)
    mapped.set_active_dims(ident)
    plain = cuda.open_session(kernel, n_ls, 1, components=components)
    for s in (mapped, plain):
        s.set_data(X, y)
    u = h.pack() + 0.02
    (f1, g1), (f0, g0) = mapped.neg_lml_and_grad(u), plain.neg_lml_and_grad(u)
    assert np.array([f1]).tobytes() == np.array([f0]).tobytes()
    assert np.all(np.abs(g1 - g0) <= 1e-9 * np.maximum(np.abs(g0), 1.0)), (g1 - g0, g0)
    Xc = np.random.default_rng(4).random((M, d))
    for s in (mapped, plain):
        s.set_window(16_384)
    for mode in (0, 1, 5):
        for s in (mapped, plain):
            s.set_screen_mode(mode)
            s.factorize(h.theta())
        assert same_record(mapped.ucb_argmax(Xc, VARSIGMA), plain.ucb_argmax(Xc, VARSIGMA)), mode
    for a, b in zip(mapped.predict_y(Xc), plain.predict_y(Xc)):
        assert a.tobytes() == b.tobytes()
    mapped.close()
    plain.close()


# ---- inactive columns ------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("case", ["m52_subset", "periodic", "phase_product"])
def test_inactive_columns_are_ignored(cuda, case):
    """Candidates that differ only in columns no leaf reads: the same bits in predict_y, in the screened values and in the joint
    covariance."""
    N, M = 1100, 70_000
    X, y = synthetic(N, D, seed=8)
    cols = CASES[case][4]
    inactive = [j for j in range(D) if all(j not in c for c in cols)]
    assert inactive
    Xc = np.random.default_rng(9).random((M, D))
    Xd = Xc.copy()
    Xd[:, inactive] = np.random.default_rng(10).random((M, len(inactive)))
    s = session(cuda, case, X, y)
    for a, b in zip(s.predict_y(Xc), s.predict_y(Xd)):
        assert a.tobytes() == b.tobytes()
    for mode in (1, 5):   # the automatic screen and the mean-bound level
        s.set_screen_mode(mode)
        s.factorize(hyper(case, 1).theta())
        ra = s.ucb_argmax(Xc, VARSIGMA)
        info = s.screen_info()
        va = s.screened_values(M) if info["path"] in ("screened", "mean-bound") else None
        assert same_record(ra, s.ucb_argmax(Xd, VARSIGMA)), mode
        # the automatic mode adapts to the previous call, so the second call may take another path
        if va is not None and s.screen_info()["path"] == info["path"]:
            assert va.tobytes() == s.screened_values(M).tobytes(), mode
    for a, b in zip(s.predict_f_cov(Xc[:500]), s.predict_f_cov(Xd[:500])):
        assert a.tobytes() == b.tobytes()
    s.close()


# ---- screened arg-max, top-k, grow ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("case", ["rq_ard_permuted", "periodic", "additive", "phase_product"])
@pytest.mark.parametrize("host", [True, False])
def test_screened_argmax_bit_identical(cuda, host, case):
    """Screen modes 0-6 with windows of 16384 candidates: the record of mode 0, top-k record 0 is the arg-max, and every screened
    value lies within E / 4 of the exact UCB (of the exact mean on the mean-bound level).  On these inputs the screens of the
    two bare leaves keep too many survivors and fall back to the full pass, so only their records are compared."""
    import torch

    N, M = 1100, 70_000
    X, y = synthetic(N, D, seed=N)
    h = hyper(case, 1)
    Xc = np.random.default_rng(M).random((M, D))
    xd = torch.from_numpy(Xc).cuda() if not host else None

    def argmax(s):
        if host:
            return s.ucb_argmax(Xc, VARSIGMA)
        return s.ucb_argmax_dev(xd.data_ptr(), M, VARSIGMA, torch.cuda.current_stream().cuda_stream)

    s = session(cuda, case, X, y)
    s.set_screen_mode(0)
    s.factorize(h.theta())
    ref = argmax(s)
    mean, var = s.predict_y(Xc)
    assert ref[0] == int(np.argmax(mean + VARSIGMA * var))
    top = s.ucb_topk(Xc, VARSIGMA, 8)
    assert same_record(ref, (int(top[0, 0]), *top[0, 1:]))
    s.set_window(16_384)
    screened = 0
    for mode in range(7):
        s.set_screen_mode(mode)
        s.factorize(h.theta())
        got = argmax(s)
        info = s.screen_info()
        assert same_record(ref, got), (mode, ref, got, info)
        if info["path"] in ("screened", "mean-bound"):
            screened += 1
            exact = mean if info["path"] == "mean-bound" else mean + VARSIGMA * var
            u = s.screened_values(M)
            assert float(np.max(np.abs(u - exact))) <= info["error_bound"] / 4.0, (mode, info)
        t = s.ucb_topk(Xc, VARSIGMA, 4)
        assert same_record(ref, (int(t[0, 0]), *t[0, 1:]))
    assert screened >= (3 if case in ("additive", "phase_product") else 0)
    s.close()


@pytest.mark.parametrize("case", ["additive", "phase_product"])
def test_grow_whole_and_by_range(cuda, case):
    N, depth = 1100, 8
    X, y = synthetic(N, D, seed=21)
    bounds = np.array([[0.0, 1.0]] * D)
    s = session(cuda, case, X, y)
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
@pytest.mark.parametrize("case,N,M", [("m52_subset", 1, 1), ("periodic_ard", 129, 300), ("additive", 700, 1000),
                                      ("overlap_repeat", 300, 500)])
def test_predict_f_full_cov(cuda, case, N, M):
    X, y = synthetic(N, D, seed=N)
    h = hyper(case, 1)
    k = min(N, M // 4)
    Xc = np.vstack([X[:k], np.random.default_rng(M).random((M - k, D))])
    s = session(cuda, case, X, y, engine="dmma")
    mean, cov = s.predict_f_cov(Xc)
    mean_ref, cov_ref = ad.predict_f_full_cov(h, CASES[case][4], X, y, Xc)
    assert np.all(np.abs(cov - cov_ref) <= 1e-8 * np.maximum(np.abs(cov_ref), h.prior_variance))
    assert np.array_equal(cov, cov.T)
    np.testing.assert_allclose(mean, mean_ref, rtol=0, atol=1e-8 * max(np.abs(y).max(), 1.0))
    assert mean.tobytes() == s.predict_y(Xc)[0].tobytes()
    ms = min(M, 200)
    z = np.random.default_rng(5).standard_normal((3, ms))
    f = s.predict_f_samples(Xc[:ms], z, JITTER)
    f_ref = so.sample_mvn(*ad.predict_f_full_cov(h, CASES[case][4], X, y, Xc[:ms]), z, JITTER)
    np.testing.assert_allclose(f, f_ref, rtol=0, atol=1e-5 * max(np.abs(f_ref).max(), 1.0))
    s.close()


def test_joint_diagonal_is_the_prior_variance_far_from_the_data(cuda):
    """Far from the data in the Matern factor's columns the product vanishes whatever the phase: the posterior covariance is the
    prior's, whose diagonal is var_prod exactly, and the mean is the constant."""
    X, y = synthetic(300, D, seed=9)
    s = session(cuda, "phase_product", X, y)
    far = np.full((2, D), 0.3)
    far[0, :3] = 1e100
    far[1, :3] = -1e100
    mean, cov = s.predict_f_cov(far)
    h = hyper("phase_product", 1)
    assert cov[0, 0] == h.prior_variance and cov[1, 1] == h.prior_variance
    assert np.all(mean == 0.1)
    s.close()


# ---- multi-GPU state ------------------------------------------------------------------------------------------------------
def test_state_export_import(cuda):
    import torch

    N = 900
    X, y = synthetic(N, D, seed=41)
    case = "phase_product"
    a = session(cuda, case, X, y)
    nbytes = a.state_bytes()
    buf = torch.empty(nbytes, dtype=torch.uint8, device=f"cuda:{cuda.device}")
    a.export_state_dev(buf.data_ptr(), nbytes)
    torch.cuda.synchronize()
    b = open_session(cuda, case, 1)
    b.import_state_dev(buf.data_ptr(), nbytes, N, D)
    Xc = np.random.default_rng(42).random((70_000, D))
    assert same_record(b.ucb_argmax(Xc, VARSIGMA), a.ucb_argmax(Xc, VARSIGMA))
    for p, q in zip(a.predict_y(Xc), b.predict_y(Xc)):
        assert p.tobytes() == q.tobytes()
    for p, q in zip(a.predict_f_cov(Xc[:64]), b.predict_f_cov(Xc[:64])):
        assert p.tobytes() == q.tobytes()
    kernel, n_ls, components, _, cols = CASES[case]
    for other in ([[0, 1, 2], [4]], [[0, 1, 3], [3]]):   # another map
        with pytest.raises(backend.GpsoBackendError, match="active dims mismatch"):
            open_session(cuda, case, 1, dims=other).import_state_dev(buf.data_ptr(), nbytes, N, D)
    with pytest.raises(backend.GpsoBackendError, match="active dims mismatch"):   # no map
        cuda.open_session(kernel, n_ls, 1, components=components).import_state_dev(buf.data_ptr(), nbytes, N, D)
    plain = cuda.open_session(kernel, n_ls, 1, components=components)   # a state without a map into a handle with one
    plain.set_data(X, y)
    plain.factorize(hyper(case, 1).theta())
    pbytes = plain.state_bytes()
    pbuf = torch.empty(pbytes, dtype=torch.uint8, device=f"cuda:{cuda.device}")
    plain.export_state_dev(pbuf.data_ptr(), pbytes)
    torch.cuda.synchronize()
    with pytest.raises(backend.GpsoBackendError, match="active dims mismatch"):
        open_session(cuda, case, 1).import_state_dev(pbuf.data_ptr(), pbytes, N, D)
    for s in (a, b, plain):
        s.close()


# ---- C argument checks ---------------------------------------------------------------------------------------------------
def test_set_active_dims_argument_checks(cuda):
    lib = backend.load_library()
    X, y = synthetic(50, 3)
    s = cuda.open_session("Sum", 0, 1, components=[("Matern52", 1), ("Matern32", 1)])
    h = s._h

    def call(n, counts, dims):
        c = (ctypes.c_int * max(len(counts), 1))(*counts)
        d = (ctypes.c_int * max(len(dims), 1))(*dims)
        return lib.gpso_set_active_dims(h, n, c, d)

    assert call(5, [1] * 5, [0] * 5) == -1 and b"0..4" in lib.gpso_last_error()
    assert call(-1, [], []) == -1
    assert call(2, [1, 0], [0]) == -1 and b"columns" in lib.gpso_last_error()
    assert call(2, [1, 1], [0, -2]) == -1 and b"negative" in lib.gpso_last_error()
    assert lib.gpso_set_active_dims(h, 1, None, None) == -1 and b"null" in lib.gpso_last_error()
    # checked at gpso_set_data: the leaf count, the columns against d and the 64 rows
    for counts, dims, what in (([1], [0], "leaf count"), ([1, 1], [0, 3], "below the input dimension")):
        assert call(len(counts), counts, dims) == 0
        with pytest.raises(backend.GpsoBackendError, match=what):
            s.set_data(X, y)
    wide = cuda.open_session("Sum", 0, 1, components=[("Matern52", 1), ("Periodic", 1, "SquaredExponential", 1)])
    wide.set_active_dims([[0] * 33, [1] * 16])
    with pytest.raises(backend.GpsoBackendError, match="64"):
        wide.set_data(X, y)
    # the map drops the data: no fit call until gpso_set_data
    assert call(2, [1, 2], [0, 1, 2]) == 0
    s.set_data(X, y)
    u = np.zeros(2 * 2 + 2)
    s.neg_lml_and_grad(u)
    s.set_active_dims([[0], [1]])
    with pytest.raises(backend.GpsoBackendError, match="set_data"):
        s.neg_lml_and_grad(u)
    s.set_active_dims(None)   # cleared: every column again
    s.set_data(X, y)
    assert np.isfinite(s.neg_lml_and_grad(u)[0])
    for q in (s, wide):
        q.close()
