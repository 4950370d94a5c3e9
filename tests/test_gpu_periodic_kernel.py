"""
Periodic kernel (gpso_create_periodic: gpflow.kernels.Periodic with a SquaredExponential or RationalQuadratic base) on the B200
against the periodic oracle (tests/periodic_oracle.py) -- run with ``-m gpu``.

Tolerances are those of test_gpu_parity.py: LML 1e-9 * max(|LML|, N), gradient 1e-6 * max(|g|, 1), posterior mean / variance and
joint covariance 1e-8.  Screened, windowed, top-k, grow and imported calls return records bit-identical to the plain call, every
screened value lies within E/4 of the exact UCB, NaN and infinite candidates are scored NaN and never discarded, duplicated
candidates give identical joint rows, and states are not imported across periodic and non-periodic kernels or across bases.
"""
import numpy as np
import pytest

from oracle import gpr_oracle as go
from pygpso_b200 import backend
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
    return X, (np.sin(6 * np.pi * X[:, 0]) + 0.5 * np.sin(3 * X.sum(1)) + 0.01 * rng.standard_normal(N))[:, None]


def hyper(base, d, ard_ls=False, ard_p=False, mean_id=1, noise=1e-3):
    ls = list(0.4 + 0.1 * np.arange(d)) if ard_ls else 0.5
    p = list(0.35 + 0.2 * np.arange(d)) if ard_p else 0.6
    mean = {0: None, 1: 0.1, 2: (np.linspace(0.5, -0.3, d), 0.05)}[mean_id]
    return pe.PeriodicHyper(base, ls, 1.2, p, noise, alpha=1.6 if base == rq.KERNEL else None, mean=mean)


def session(cuda, h, X, y, mean_id=1, engine=None, factorize=True):
    s = cuda.open_session("Periodic", h.lengthscales.size, mean_id, components=[(h.base, h.period.size)])
    if engine is not None:
        s.set_predict_mode(*ENGINES[engine])
    s.set_data(X, y)
    if factorize:
        s.factorize(h.theta())
    return s


# ---- LML + gradient ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("base", pe.BASES)
@pytest.mark.parametrize("N,d,ard_ls,ard_p,mean_id", [(1, 2, False, False, 1), (129, 3, True, False, 0), (300, 4, False, True, 2),
                                                      (300, 3, True, True, 1), (1100, 5, True, True, 2), (1100, 12, False, True, 0),
                                                      (4200, 3, True, True, 1), (700, 32, True, True, 1)])
def test_neg_lml_and_grad(cuda, base, N, d, ard_ls, ard_p, mean_id):
    """1100 rows: the int8 K_y^-1 engine; 4200 rows: the hybrid factorisation; d = 12 and 32: every warp of the gradient's
    second pass takes more than one dimension, and d = 32 is the largest input dimension (64 embedded rows)."""
    X, y = synthetic(N, d, seed=N + d)
    h = hyper(base, d, ard_ls, ard_p, mean_id)
    u = h.pack() + 0.03
    f_ref, g_ref = pe.neg_lml_and_grad(base, h.lengthscales.size, h.period.size, X, y, u, mean_id)
    s = session(cuda, h, X, y, mean_id, factorize=False)
    f, g = s.neg_lml_and_grad(u)
    s.close()
    assert abs(f - f_ref) <= 1e-9 * max(abs(f_ref), N), (f, f_ref)
    assert g.shape == g_ref.shape
    assert np.all(np.abs(g - g_ref) <= 1e-6 * np.maximum(np.abs(g_ref), 1.0)), (g, g_ref)


def test_bad_parameters_and_shapes_are_rejected(cuda):
    X, y = synthetic(20, 2)
    h = hyper(rq.KERNEL, 2, ard_p=True)
    s = session(cuda, h, X, y, factorize=False)
    n = h.theta().size   # alpha, ls, var, 2 periods, noise, c = 7
    for p in (n - 2, n - 1, n + 1):
        with pytest.raises(backend.GpsoBackendError, match="hyper-parameters"):
            s.neg_lml_and_grad(np.zeros(p))
        with pytest.raises(backend.GpsoBackendError, match="hyper-parameters"):
            s.factorize(np.ones(p))
    theta = h.theta()
    theta[4] = -1.0   # the second period
    with pytest.raises(backend.GpsoBackendError, match="period"):
        s.factorize(theta)
    s.close()
    wide = hyper("SquaredExponential", 33)
    with pytest.raises(backend.GpsoBackendError, match="32"):
        session(cuda, wide, *synthetic(10, 33), factorize=False)
    with pytest.raises(backend.GpsoBackendError, match="32"):
        cuda.open_session("Periodic", 1, 1, components=[("SquaredExponential", 1)]).state_bytes(10, 33)


# ---- predict_y ------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("base,N,d,M,ard", [("SquaredExponential", 1, 1, 1, False), (rq.KERNEL, 129, 3, 129, True),
                                            ("SquaredExponential", 512, 2, 5000, True), (rq.KERNEL, 1100, 6, 3001, False)])
@pytest.mark.parametrize("engine", sorted(ENGINES))
def test_predict_y(cuda, engine, base, N, d, M, ard):
    X, y = synthetic(N, d)
    h = hyper(base, d, ard, ard)
    Xc = np.random.default_rng(N + M).random((M, d))
    mean_ref, var_ref = pe.predict_y(h, X, y, Xc)
    s = session(cuda, h, X, y, engine=engine)
    mean, var = s.predict_y(Xc)
    assert_predict_close(mean, var, mean_ref[:, 0], var_ref[:, 0], y, h.variance)
    idx, m, v, u = s.ucb_argmax(Xc, VARSIGMA)
    assert idx == go.ucb_argmax(mean_ref, var_ref, VARSIGMA)[0]
    assert m == mean[idx] and v == var[idx] and u == mean[idx] + VARSIGMA * var[idx]
    s.close()


# ---- screened arg-max, windows, top-k, grow ---------------------------------------------------------------------------------
@pytest.mark.parametrize("base", pe.BASES)
@pytest.mark.parametrize("host", [True, False])
def test_screened_argmax_bit_identical(cuda, host, base):
    """Screen modes 0-6 with windows of 16384 candidates: the record of mode 0, top-k record 0 is the arg-max, every screened
    value within E/4 of the exact UCB, NaN / infinite candidates NaN in the screen and never winning silently."""
    import torch

    N, d, M = 1100, 3, 70_000
    X, y = synthetic(N, d, seed=N)
    h = hyper(base, d, True, True)
    Xc = np.random.default_rng(M).random((M, d))
    Xc[50_000:50_100] = Xc[100:200]   # duplicated candidates: bit-identical values wherever they sit
    Xc[60_000:60_100] += 3 * h.period  # shifted by whole periods: the same covariance
    xd = torch.from_numpy(Xc).cuda() if not host else None

    def argmax(s):
        if host:
            return s.ucb_argmax(Xc, VARSIGMA)
        return s.ucb_argmax_dev(xd.data_ptr(), M, VARSIGMA, torch.cuda.current_stream().cuda_stream)

    s = session(cuda, h, X, y)
    s.set_screen_mode(0)
    s.factorize(h.theta())
    ref = argmax(s)
    assert ref == s.ucb_argmax(Xc, VARSIGMA)
    top = s.ucb_topk(Xc, VARSIGMA, 8)
    assert same_record(ref, (int(top[0, 0]), *top[0, 1:]))
    mean, var = s.predict_y(Xc)
    assert mean[50_000:50_100].tobytes() == mean[100:200].tobytes() and var[50_000:50_100].tobytes() == var[100:200].tobytes()
    mref, _ = pe.predict_y(h, X, y, Xc[60_000:60_100])
    np.testing.assert_allclose(mean[60_000:60_100], mref[:, 0], rtol=0, atol=1e-8 * max(np.abs(y).max(), 1.0))
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
            assert info["max_observed_deviation"] <= info["error_bound"] / 4.0, info
            u = s.screened_values(M)
            exact = mean if info["path"] == "mean-bound" else mean + VARSIGMA * var
            assert np.max(np.abs(u - exact)) <= info["error_bound"] / 4.0, (mode, info)
        t = s.ucb_topk(Xc, VARSIGMA, 4)
        assert same_record(ref, (int(t[0, 0]), *t[0, 1:]))
    assert screened >= 3
    # NaN and infinite coordinates: NaN screened values, and the NaN candidate wins as in numpy
    bad = Xc.copy()
    bad[123, 1] = np.nan
    bad[4567, 0] = np.inf
    s.set_screen_mode(2)
    s.factorize(h.theta())
    rec = s.ucb_argmax(bad, VARSIGMA)
    assert rec[0] == 123 and np.isnan(rec[3])
    if s.screen_info()["path"] == "screened":
        u = s.screened_values(M)
        assert np.isnan(u[123]) and np.isnan(u[4567]) and np.isfinite(np.delete(u, [123, 4567])).all()
    s.close()


def test_grow_whole_and_by_range(cuda):
    N, d, depth = 1100, 3, 11          # grow(11) = 88 573 leaves
    X, y = synthetic(N, d, seed=21)
    h = hyper("SquaredExponential", d, True, True)
    bounds = np.array([[0.0, 1.0]] * d)
    s = session(cuda, h, X, y)
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
# The joint path forms V = L^-1 Ks^T with the fp64 L^-1 whatever gpso_set_predict_mode selects for predict_y (the header says so):
# under every other engine the joint mean, covariance and samples are the dmma session's bytes.  The samples pass through the
# Cholesky factor of cov + jitter I, whose smallest eigenvalues are near the jitter: it amplifies the 1e-8 agreement of cov with
# the oracle, so they are held to 1e-5 against the oracle's own draws, and to 1e-8 against the oracle's sampler applied to the
# device's joint mean and covariance; the zero draw is the mean's bytes.
@pytest.mark.parametrize("engine", sorted(ENGINES))
@pytest.mark.parametrize("base,N,M", [("SquaredExponential", 1, 1), (rq.KERNEL, 129, 300), ("SquaredExponential", 700, 1000)])
def test_predict_f_full_cov(cuda, base, N, M, engine):
    d = 3
    X, y = synthetic(N, d, seed=N)
    h = hyper(base, d, True, True)
    k = min(N, M // 4)
    Xc = np.vstack([X[:k], np.random.default_rng(M).random((M - k, d))])
    if M > 10:
        Xc[-5:] = Xc[:5]   # duplicated candidates: identical joint rows and columns
    s = session(cuda, h, X, y, engine=engine)
    mean, cov = s.predict_f_cov(Xc)
    mean_ref, cov_ref = pe.predict_f_full_cov(h, X, y, Xc)
    assert np.all(np.abs(cov - cov_ref) <= 1e-8 * np.maximum(np.abs(cov_ref), h.variance))
    assert np.array_equal(cov, cov.T)
    if M > 10:
        assert cov[-5:].tobytes() == cov[:5].tobytes() and mean[-5:].tobytes() == mean[:5].tobytes()
    np.testing.assert_allclose(mean, mean_ref, rtol=0, atol=1e-8 * max(np.abs(y).max(), 1.0))
    my, _ = s.predict_y(Xc)
    if engine == "dmma":
        assert mean.tobytes() == my.tobytes()
    else:
        np.testing.assert_allclose(my, mean, rtol=0, atol=1e-8 * max(np.abs(y).max(), 1.0))
    draw = s.predict_f_samples(Xc, np.zeros((1, M)), JITTER)[0]
    assert draw.tobytes() == mean.tobytes()
    ms = min(M, 200)
    z = np.random.default_rng(5).standard_normal((3, ms))
    f = s.predict_f_samples(Xc[:ms], z, JITTER)
    f_ref = so.sample_mvn(*pe.predict_f_full_cov(h, X, y, Xc[:ms]), z, JITTER)
    np.testing.assert_allclose(f, f_ref, rtol=0, atol=1e-5 * max(np.abs(f_ref).max(), 1.0))
    f_own = so.sample_mvn(*s.predict_f_cov(Xc[:ms]), z, JITTER)
    np.testing.assert_allclose(f, f_own, rtol=0, atol=1e-8 * max(np.abs(f_own).max(), 1.0))
    if engine != "dmma":
        r = session(cuda, h, X, y, engine="dmma")
        mean_d, cov_d = r.predict_f_cov(Xc)
        assert mean_d.tobytes() == mean.tobytes() and cov_d.tobytes() == cov.tobytes()
        assert r.predict_f_samples(Xc[:ms], z, JITTER).tobytes() == f.tobytes()
        r.close()
    s.close()


# ---- multi-GPU state ------------------------------------------------------------------------------------------------------
def test_state_export_import(cuda):
    import torch

    N, d = 900, 4
    X, y = synthetic(N, d, seed=41)
    h = hyper(rq.KERNEL, d, True, True)
    a = session(cuda, h, X, y)
    nbytes = a.state_bytes()
    assert nbytes == 8 * (128 + 2 * d * 1024 + 1024 + 1024 * 1024)
    buf = torch.empty(nbytes, dtype=torch.uint8, device=f"cuda:{cuda.device}")
    a.export_state_dev(buf.data_ptr(), nbytes)
    torch.cuda.synchronize()
    header = buf[: 128 * 8].cpu().numpy().view(np.float64)
    assert header[6] == 4 and header[10] == 1.0 and header[11] == 1.0 and np.array_equal(header[80:80 + d], h.period)
    b = cuda.open_session("Periodic", d, 1, components=[(rq.KERNEL, d)])
    b.import_state_dev(buf.data_ptr(), nbytes, N, d)
    Xc = np.random.default_rng(42).random((70_000, d))
    assert same_record(b.ucb_argmax(Xc, VARSIGMA), a.ucb_argmax(Xc, VARSIGMA))
    ma, va = a.predict_y(Xc)
    mb, vb = b.predict_y(Xc)
    assert np.array_equal(ma, mb) and np.array_equal(va, vb)
    for p, q in zip(a.predict_f_cov(Xc[:64]), b.predict_f_cov(Xc[:64])):
        assert p.tobytes() == q.tobytes()
    # another base, another ARD flag of the period or the lengthscales, the bare base kernel: refused
    for kind, n_ls, comps in (("Periodic", d, [("SquaredExponential", d)]), ("Periodic", d, [(rq.KERNEL, 1)]),
                              ("Periodic", 1, [(rq.KERNEL, d)])):
        with pytest.raises(backend.GpsoBackendError, match="mismatch|too small"):
            cuda.open_session(kind, n_ls, 1, components=comps).import_state_dev(buf.data_ptr(), nbytes, N, d)
    with pytest.raises(backend.GpsoBackendError, match="mismatch|too small"):
        cuda.open_session(rq.KERNEL, d, True).import_state_dev(buf.data_ptr(), nbytes, N, d)
    # and a bare SquaredExponential state (half the input rows) is not taken by a periodic handle
    se = cuda.open_session("SquaredExponential", 1, True)
    se.set_data(X, y)
    se.factorize(np.array([0.5, 1.0, 1e-3, 0.1]))
    sb = torch.empty(se.state_bytes(), dtype=torch.uint8, device=f"cuda:{cuda.device}")
    se.export_state_dev(sb.data_ptr(), se.state_bytes())
    torch.cuda.synchronize()
    padded = torch.zeros(nbytes, dtype=torch.uint8, device=f"cuda:{cuda.device}")
    padded[: se.state_bytes()] = sb
    for src, n, why in ((sb, se.state_bytes(), "too small"), (padded, nbytes, "periodic kernel mismatch")):
        with pytest.raises(backend.GpsoBackendError, match=why):
            cuda.open_session("Periodic", 1, 1, components=[("SquaredExponential", 1)]).import_state_dev(src.data_ptr(), n, N, d)
    for s in (a, b, se):
        s.close()


# ---- periodic terms inside sums and products ----------------------------------------------------------------------------
def composite_hyper(key, d, mean_id=1, noise=1e-3):
    """"se*periodic(se)": the locally periodic kernel; "m52+periodic(rq)": trend plus season; both with an ARD period."""
    p = list(0.35 + 0.2 * np.arange(d))
    mean = {0: None, 1: 0.1, 2: (np.linspace(0.5, -0.3, d), 0.05)}[mean_id]
    if key == "se*periodic(se)":
        comps = [so.Comp("SquaredExponential", 0.9, 1.1), pe.PeriodicHyper("SquaredExponential", 0.5, 1.0, p, 1.0)]
        return "Product", [("SquaredExponential", 1), ("Periodic", 1, "SquaredExponential", d)], pe.CompositeHyper("Product", comps, noise, mean)
    comps = [so.Comp("Matern52", list(0.4 + 0.1 * np.arange(d)), 0.8),
             pe.PeriodicHyper(rq.KERNEL, list(0.5 + 0.1 * np.arange(d)), 0.6, p, 1.0, alpha=1.6)]
    return "Sum", [("Matern52", d), ("Periodic", d, rq.KERNEL, d)], pe.CompositeHyper("Sum", comps, noise, mean)


def composite_session(cuda, kind, specs, h, X, y, mean_id=1, engine=None, factorize=True):
    s = cuda.open_session(kind, 0, mean_id, components=specs)
    if engine is not None:
        s.set_predict_mode(*ENGINES[engine])
    s.set_data(X, y)
    if factorize:
        s.factorize(h.theta())
    return s


@pytest.mark.parametrize("key", ["se*periodic(se)", "m52+periodic(rq)"])
@pytest.mark.parametrize("N,d,mean_id", [(1, 2, 1), (129, 3, 0), (300, 4, 2), (1100, 5, 1), (4200, 3, 2), (700, 16, 1)])
def test_composite_neg_lml_and_grad(cuda, key, N, d, mean_id):
    """1100 rows: the int8 K_y^-1 engine; 4200 rows: the hybrid factorisation; d = 16: 48 rows of the sum, 4 dimensions per warp."""
    X, y = synthetic(N, d, seed=N + d)
    kind, specs, h = composite_hyper(key, d, mean_id)
    u = h.pack() + 0.03
    f_ref, g_ref = pe.composite_neg_lml_and_grad(kind, specs, X, y, u, mean_id)
    s = composite_session(cuda, kind, specs, h, X, y, mean_id, factorize=False)
    f, g = s.neg_lml_and_grad(u)
    with pytest.raises(backend.GpsoBackendError, match="hyper-parameters"):
        s.neg_lml_and_grad(u[:-1])
    s.close()
    assert abs(f - f_ref) <= 1e-9 * max(abs(f_ref), N), (f, f_ref)
    assert g.shape == g_ref.shape
    assert np.all(np.abs(g - g_ref) <= 1e-6 * np.maximum(np.abs(g_ref), 1.0)), (g, g_ref)


@pytest.mark.parametrize("key", ["se*periodic(se)", "m52+periodic(rq)"])
@pytest.mark.parametrize("engine", sorted(ENGINES))
def test_composite_posterior(cuda, key, engine):
    N, d, M = 700, 3, 3001
    X, y = synthetic(N, d, seed=5)
    kind, specs, h = composite_hyper(key, d)
    Xc = np.random.default_rng(6).random((M, d))
    Xc[-5:] = Xc[:5]
    s = composite_session(cuda, kind, specs, h, X, y, engine=engine)
    mean_ref, var_ref = pe.composite_predict_y(h, X, y, Xc)
    mean, var = s.predict_y(Xc)
    assert_predict_close(mean, var, mean_ref[:, 0], var_ref[:, 0], y, h.prior_variance)
    mf, cov = s.predict_f_cov(Xc[:400])
    mf_ref, cov_ref = pe.composite_predict_f_full_cov(h, X, y, Xc[:400])
    assert np.all(np.abs(cov - cov_ref) <= 1e-8 * np.maximum(np.abs(cov_ref), h.prior_variance))
    np.testing.assert_allclose(mf, mf_ref, rtol=0, atol=1e-8 * max(np.abs(y).max(), 1.0))
    draw = s.predict_f_samples(Xc[:400], np.zeros((1, 400)), JITTER)[0]
    assert draw.tobytes() == mf.tobytes()
    s.close()


@pytest.mark.parametrize("kind", ["Sum", "Product"])
def test_one_term_combination_of_a_periodic_is_the_bare_kernel(cuda, kind):
    N, d, M = 1100, 3, 70_000
    X, y = synthetic(N, d, seed=3)
    h = hyper(rq.KERNEL, d, True, True)
    theta, u = h.theta(), h.pack() + 0.02
    one = cuda.open_session(kind, 0, 1, components=[("Periodic", d, rq.KERNEL, d)])
    bare = session(cuda, h, X, y, factorize=False)
    one.set_data(X, y)
    (f1, g1), (fb, gb) = one.neg_lml_and_grad(u), bare.neg_lml_and_grad(u)
    assert np.array([f1]).tobytes() == np.array([fb]).tobytes()
    assert np.all(np.abs(g1 - gb) <= 1e-9 * np.maximum(np.abs(gb), 1.0)), (g1 - gb, gb)
    Xc = np.random.default_rng(4).random((M, d))
    for s in (one, bare):
        s.set_window(16_384)
    for mode in (0, 1, 5):
        for s in (one, bare):
            s.set_screen_mode(mode)
            s.factorize(theta)
        assert same_record(one.ucb_argmax(Xc, VARSIGMA), bare.ucb_argmax(Xc, VARSIGMA)), mode
    for a, b in zip(one.predict_y(Xc), bare.predict_y(Xc)):
        assert a.tobytes() == b.tobytes()
    (m1, c1), (mb, cb) = one.predict_f_cov(Xc[:300]), bare.predict_f_cov(Xc[:300])
    assert m1.tobytes() == mb.tobytes() and np.diag(c1).tobytes() == np.diag(cb).tobytes()
    # off the diagonal the bare joint_syrk_kernel may fuse the covariance's last product into the subtraction (one rounding)
    assert np.all(np.abs(c1 - cb) <= 4.0 * np.finfo(np.float64).eps * h.variance)
    one.close()
    bare.close()


@pytest.mark.parametrize("key", ["se*periodic(se)", "m52+periodic(rq)"])
def test_composite_screened_argmax_bit_identical(cuda, key):
    N, d, M = 1100, 3, 70_000
    X, y = synthetic(N, d, seed=N)
    kind, specs, h = composite_hyper(key, d)
    Xc = np.random.default_rng(M).random((M, d))
    Xc[50_000:50_100] = Xc[100:200]
    s = composite_session(cuda, kind, specs, h, X, y)
    s.set_screen_mode(0)
    s.factorize(h.theta())
    ref = s.ucb_argmax(Xc, VARSIGMA)
    mean, var = s.predict_y(Xc)
    assert mean[50_000:50_100].tobytes() == mean[100:200].tobytes()
    s.set_window(16_384)
    screened = 0
    for mode in range(7):
        s.set_screen_mode(mode)
        s.factorize(h.theta())
        got = s.ucb_argmax(Xc, VARSIGMA)
        info = s.screen_info()
        assert same_record(ref, got), (mode, ref, got, info)
        if info["path"] in ("screened", "mean-bound"):
            screened += 1
            u = s.screened_values(M)
            exact = mean if info["path"] == "mean-bound" else mean + VARSIGMA * var
            assert np.max(np.abs(u - exact)) <= info["error_bound"] / 4.0, (mode, info)
        t = s.ucb_topk(Xc, VARSIGMA, 4)
        assert same_record(ref, (int(t[0, 0]), *t[0, 1:]))
    assert screened >= 3
    bounds = np.array([[0.0, 1.0]] * d)
    whole = s.grow_ucb_argmax(bounds, 10, VARSIGMA)
    total = cuda.grow_count(10)
    parts = [s.grow_ucb_argmax(bounds, 10, VARSIGMA, rows=(0, 20_001)), s.grow_ucb_argmax(bounds, 10, VARSIGMA, rows=(20_001, total))]
    assert same_record(whole, max(parts, key=lambda r: (r[3], -r[0])))
    s.close()


def test_composite_state_export_import(cuda):
    import torch

    N, d = 900, 4
    X, y = synthetic(N, d, seed=41)
    kind, specs, h = composite_hyper("m52+periodic(rq)", d)
    a = composite_session(cuda, kind, specs, h, X, y)
    nbytes = a.state_bytes()
    buf = torch.empty(nbytes, dtype=torch.uint8, device=f"cuda:{cuda.device}")
    a.export_state_dev(buf.data_ptr(), nbytes)
    torch.cuda.synchronize()
    b = cuda.open_session(kind, 0, 1, components=specs)
    b.import_state_dev(buf.data_ptr(), nbytes, N, d)
    Xc = np.random.default_rng(42).random((70_000, d))
    assert same_record(b.ucb_argmax(Xc, VARSIGMA), a.ucb_argmax(Xc, VARSIGMA))
    for p, q in zip(a.predict_y(Xc), b.predict_y(Xc)):
        assert p.tobytes() == q.tobytes()
    for p, q in zip(a.predict_f_cov(Xc[:64]), b.predict_f_cov(Xc[:64])):
        assert p.tobytes() == q.tobytes()
    # another base, another period ARD flag, the plain sum: refused
    for other in ([specs[0], ("Periodic", d, "SquaredExponential", d)], [specs[0], ("Periodic", d, rq.KERNEL, 1)],
                  [specs[0], (rq.KERNEL, d)]):
        with pytest.raises(backend.GpsoBackendError, match="mismatch|too small"):
            cuda.open_session(kind, 0, 1, components=other).import_state_dev(buf.data_ptr(), nbytes, N, d)
    a.close()
    b.close()
