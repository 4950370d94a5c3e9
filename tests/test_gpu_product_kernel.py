"""
Product kernel (GPSO_KERNEL_PRODUCT, k = prod_c k_c) on the B200 against the product oracle (tests/product_oracle.py) -- run
with ``-m gpu``.

Tolerances are those of test_gpu_parity.py: LML 1e-9 * max(|LML|, N), gradient 1e-6 * max(|g|, 1), posterior mean / variance
and joint covariance 1e-8 (1e-7 where Matern12 is a factor: its covariance has an infinite slope at r = 0, so the device's
difference-first distances and the oracle's differ most there).  Screened, windowed and imported calls return records
bit-identical to the plain call, every screened value lies within E/4 of the exact UCB, and a one-factor product gives the
bytes of its bare kernel (the joint covariance off its diagonal to one rounding, as for a one-component sum).
"""
import numpy as np
import pytest

from oracle import gpr_oracle as go
from pygpso_b200 import backend
from tests import rq_oracle as rq
from tests import product_oracle as po
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


def comps(case, d):
    ard = list(0.3 + 0.1 * np.arange(d))
    return {
        "se*m12": [po.Comp("SquaredExponential", 0.5, 0.8), po.Comp("Matern12", 0.6, 1.5)],
        "m52*rq": [po.Comp("Matern52", 0.4, 1.1), po.Comp(rq.KERNEL, 0.6, 0.9, alpha=1.7)],
        "four": [po.Comp("Matern32", ard, 0.9), po.Comp("SquaredExponential", 0.9, 1.3), po.Comp(rq.KERNEL, ard, 1.2, alpha=0.8),
                 po.Comp("Matern12", 1.5, 0.7)],
    }[case]


def session(cuda, h, X, y, mean_id=1, engine=None, factorize=True):
    s = cuda.open_session("Product", 0, mean_id, components=[(c.family, c.n_ls) for c in h.comps])
    if engine is not None:
        s.set_predict_mode(*ENGINES[engine])
    s.set_data(X, y)
    if factorize:
        s.factorize(h.theta())
    return s


def has_m12(h):
    return any(c.family == "Matern12" for c in h.comps)


# ---- LML + gradient ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("case,N,d,mean_id", [("se*m12", 1, 2, 1), ("se*m12", 129, 3, 0), ("m52*rq", 300, 4, 1), ("m52*rq", 1100, 5, 2),
                                              ("four", 700, 3, 1), ("four", 700, 12, 2), ("four", 1100, 3, 0), ("four", 4200, 3, 1),
                                              ("se*m12", 4200, 6, 0), ("m52*rq", 4200, 4, 2)])
def test_neg_lml_and_grad(cuda, case, N, d, mean_id):
    """1100 rows: the int8 K_y^-1 engine; 4200 rows: the hybrid factorisation.  "four" has two ARD factors: at d = 12 every
    warp of the gradient's second pass takes more than one dimension."""
    X, y = synthetic(N, d, seed=N + d)
    mean = {0: None, 1: 0.1, 2: (np.linspace(0.5, -0.3, d), 0.05)}[mean_id]
    h = po.ProductHyper(comps(case, d), 2e-3, mean)
    u = h.pack() + 0.03
    fam, nls = [c.family for c in h.comps], [c.n_ls for c in h.comps]
    f_ref, g_ref = po.neg_lml_and_grad(fam, nls, X, y, u, mean_id)
    s = session(cuda, h, X, y, mean_id, factorize=False)
    f, g = s.neg_lml_and_grad(u)
    s.close()
    assert abs(f - f_ref) <= 1e-9 * max(abs(f_ref), N), (f, f_ref)
    assert g.shape == g_ref.shape
    assert np.all(np.abs(g - g_ref) <= 1e-6 * np.maximum(np.abs(g_ref), 1.0)), (g, g_ref)


def test_bad_parameters_are_rejected(cuda):
    X, y = synthetic(20, 2)
    h = po.ProductHyper(comps("m52*rq", 2), 1e-3, 0.1)
    s = session(cuda, h, X, y, factorize=False)
    n = h.theta().size   # (1 + 1) + (1 + 1 + 1) + noise + c = 7
    for p in (n - 2, n - 1, n + 1):
        with pytest.raises(backend.GpsoBackendError, match="hyper-parameters"):
            s.neg_lml_and_grad(np.zeros(p))
        with pytest.raises(backend.GpsoBackendError, match="hyper-parameters"):
            s.factorize(np.ones(p))
    theta = h.theta()
    theta[4] = -1.0   # the RQ factor's variance
    with pytest.raises(backend.GpsoBackendError, match="variances"):
        s.factorize(theta)
    s.close()
    wide = po.ProductHyper([po.Comp("Matern52", 1.0, 1.0)] * 2, 1e-3, 0.1)
    with pytest.raises(backend.GpsoBackendError, match="64"):
        session(cuda, wide, *synthetic(10, 33), factorize=False)


def test_not_positive_definite_reports_info(cuda):
    y = np.array([[0.0], [1.0], [0.3], [0.5]])
    h = po.ProductHyper(comps("se*m12", 2), 1e-3, 0.0)
    s = session(cuda, h, np.full((4, 2), np.nan), y, factorize=False)
    with pytest.raises(np.linalg.LinAlgError, match="pivot"):
        s.factorize(h.theta())
    s.close()


# ---- predict_y ------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("case,N,d,M", [("se*m12", 1, 1, 1), ("m52*rq", 129, 3, 129), ("four", 512, 2, 5000), ("se*m12", 1100, 6, 3001)])
@pytest.mark.parametrize("engine", ["dmma", "int8"])
def test_predict_y(cuda, engine, case, N, d, M):
    X, y = synthetic(N, d)
    h = po.ProductHyper(comps(case, d), 1e-3, 0.05)
    Xc = np.random.default_rng(N + M).random((M, d))
    mean_ref, var_ref = po.predict_y(h, X, y, Xc)
    s = session(cuda, h, X, y, engine=engine)
    assert s.predict_info()["engine"] == ("fp64-dmma" if engine == "dmma" else "int8-tcgen05")
    mean, var = s.predict_y(Xc)
    assert_predict_close(mean, var, mean_ref[:, 0], var_ref[:, 0], y, h.var_prod, rel=1e-7 if has_m12(h) else 1e-8)
    idx, m, v, u = s.ucb_argmax(Xc, VARSIGMA)
    assert idx == go.ucb_argmax(mean_ref, var_ref, VARSIGMA)[0]
    assert m == mean[idx] and v == var[idx] and u == mean[idx] + VARSIGMA * var[idx]
    s.close()


# ---- a one-factor product is its bare kernel, byte for byte ---------------------------------------------------------------
@pytest.mark.parametrize("family,ard", [("Matern52", False), ("Matern12", True), (rq.KERNEL, False), ("SquaredExponential", True),
                                        ("Matern32", True)])
def test_one_factor_is_the_bare_kernel(cuda, family, ard):
    N, d, M = 1100, 4, 70_000
    X, y = synthetic(N, d, seed=3)
    ls = [0.3, 0.5, 0.4, 0.6] if ard else 0.45
    c = po.Comp(family, ls, 1.3, 1.6 if family == rq.KERNEL else None)
    h = po.ProductHyper([c], 1e-3, 0.2)
    theta = h.theta()
    u = h.pack() + 0.02
    one = session(cuda, h, X, y, factorize=False)
    bare = cuda.open_session(family, c.n_ls, True)
    bare.set_data(X, y)
    (f1, g1), (fb, gb) = one.neg_lml_and_grad(u), bare.neg_lml_and_grad(u)
    assert np.array([f1]).tobytes() == np.array([fb]).tobytes()
    # The gradient sums the same terms in another order: with ARD, lml_grad_product_kernel reduces each dimension over the
    # tile in one warp where the bare kernel reduces it across the block, four dimensions per launch.  Rounding apart, a
    # thousandth of the oracle parity bar.
    if ard:
        assert np.all(np.abs(g1 - gb) <= 1e-9 * np.maximum(np.abs(gb), 1.0)), (g1 - gb, gb)
    else:
        assert g1.tobytes() == gb.tobytes()
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
    assert m1.tobytes() == mb.tobytes()
    assert np.diag(c1).tobytes() == np.diag(cb).tobytes()
    # Off the diagonal the bare joint_syrk_kernel rounds one product less: the compiler fuses the covariance's last product
    # with the subtraction of (V^T V)_ij into one DFMA, while the product kernel rounds the covariance first.  One rounding of
    # k <= var apart: a few ulp of var, far below the 1e-8 parity bar.  (On the diagonal that product is exact.)
    assert np.all(np.abs(c1 - cb) <= 4.0 * np.finfo(np.float64).eps * h.var_prod), float(np.max(np.abs(c1 - cb)))
    one.close()
    bare.close()


# ---- screened arg-max, windows, top-k, grow ---------------------------------------------------------------------------------
@pytest.mark.parametrize("case", ["se*m12", "four"])
@pytest.mark.parametrize("host", [True, False])
def test_screened_argmax_bit_identical(cuda, host, case):
    """Screen modes 0-6 with windows of 16384 candidates: the record of mode 0, and top-k record 0 is the arg-max."""
    import torch

    N, d, M = 1100, 3, 70_000
    X, y = synthetic(N, d, seed=N)
    h = po.ProductHyper(comps(case, d), 1e-3, 0.05)
    Xc = np.random.default_rng(M).random((M, d))
    Xc[50_000:50_100] = Xc[100:200]   # duplicated candidates: bit-identical values wherever they sit
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
        t = s.ucb_topk(Xc, VARSIGMA, 4)
        assert same_record(ref, (int(t[0, 0]), *t[0, 1:]))
    assert screened >= 3
    s.close()


def test_grow_whole_and_by_range(cuda):
    N, d, depth = 1100, 3, 11          # grow(11) = 88 573 leaves
    X, y = synthetic(N, d, seed=21)
    h = po.ProductHyper(comps("four", d), 1e-3, 0.0)
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
@pytest.mark.parametrize("case,N,M", [("se*m12", 1, 1), ("m52*rq", 129, 300), ("four", 700, 1000)])
def test_predict_f_full_cov(cuda, case, N, M):
    d = 3
    X, y = synthetic(N, d, seed=N)
    h = po.ProductHyper(comps(case, d), 1e-3, 0.1)
    k = min(N, M // 4)
    Xc = np.vstack([X[:k], np.random.default_rng(M).random((M - k, d))])
    s = session(cuda, h, X, y, engine="dmma")
    mean, cov = s.predict_f_cov(Xc)
    mean_ref, cov_ref = po.predict_f_full_cov(h, X, y, Xc)
    rel = 1e-7 if has_m12(h) else 1e-8
    assert np.all(np.abs(cov - cov_ref) <= rel * np.maximum(np.abs(cov_ref), h.var_prod))
    assert np.array_equal(cov, cov.T)
    np.testing.assert_allclose(mean, mean_ref, rtol=0, atol=rel * max(np.abs(y).max(), 1.0))
    my, _ = s.predict_y(Xc)
    assert mean.tobytes() == my.tobytes()
    draw = s.predict_f_samples(Xc, np.zeros((1, M)), JITTER)[0]
    assert draw.tobytes() == mean.tobytes()
    ms = min(M, 200)
    z = np.random.default_rng(5).standard_normal((3, ms))
    f = s.predict_f_samples(Xc[:ms], z, JITTER)
    f_ref = so.sample_mvn(*po.predict_f_full_cov(h, X, y, Xc[:ms]), z, JITTER)
    np.testing.assert_allclose(f, f_ref, rtol=0, atol=1e-5 * max(np.abs(f_ref).max(), 1.0))
    s.close()


def test_joint_diagonal_starts_from_the_product_variance(cuda):
    """Far from the data K* = 0: the posterior covariance is the prior's, whose diagonal is var_prod = prod_c var_c exactly."""
    d = 2
    X, y = synthetic(300, d, seed=9)
    h = po.ProductHyper([po.Comp("Matern52", 0.3, 0.7), po.Comp("SquaredExponential", 0.5, 0.2), po.Comp("Matern32", 0.2, 0.1)],
                    1e-3, 0.0)
    far = np.array([[1e100, 1e100], [-1e100, 1e100]])
    s = session(cuda, h, X, y)
    mean, cov = s.predict_f_cov(far)
    assert cov[0, 0] == h.var_prod and cov[1, 1] == h.var_prod and cov[0, 1] == 0.0
    assert np.all(mean == 0.0)
    s.close()


# ---- multi-GPU state ------------------------------------------------------------------------------------------------------
def test_state_export_import(cuda):
    import torch

    N, d = 900, 4
    X, y = synthetic(N, d, seed=41)
    h = po.ProductHyper(comps("four", d), 1e-3, 0.1)
    a = session(cuda, h, X, y)
    nbytes = a.state_bytes()
    buf = torch.empty(nbytes, dtype=torch.uint8, device=f"cuda:{cuda.device}")
    a.export_state_dev(buf.data_ptr(), nbytes)
    torch.cuda.synchronize()
    header = buf[: 16 * 8].cpu().numpy().view(np.float64)
    assert header[6] == po.KERNEL_ID and header[2] == h.var_prod
    block = buf[-8 * (1 + sum(4 + c.n_ls for c in h.comps)):].cpu().numpy().view(np.float64)
    assert block[0] == len(h.comps)
    q = 1
    for c in h.comps:   # family, lengthscale count, the factor's own variance, alpha, lengthscales
        assert block[q + 1] == c.n_ls and block[q + 2] == c.variance
        q += 4 + c.n_ls
    comp_spec = [(c.family, c.n_ls) for c in h.comps]
    b = cuda.open_session("Product", 0, 1, components=comp_spec)
    b.import_state_dev(buf.data_ptr(), nbytes, N, d)
    Xc = np.random.default_rng(42).random((70_000, d))
    assert same_record(b.ucb_argmax(Xc, VARSIGMA), a.ucb_argmax(Xc, VARSIGMA))
    ma, va = a.predict_y(Xc)
    mb, vb = b.predict_y(Xc)
    assert np.array_equal(ma, mb) and np.array_equal(va, vb)
    for p, q in zip(a.predict_f_cov(Xc[:64]), b.predict_f_cov(Xc[:64])):
        assert p.tobytes() == q.tobytes()
    # another family, another ARD flag, another count: refused
    others = [[("Matern52", 4)] + comp_spec[1:], comp_spec[:1] + [("SquaredExponential", 4)] + comp_spec[2:], comp_spec[:3]]
    for spec in others:
        with pytest.raises(backend.GpsoBackendError, match="component mismatch|source too small"):
            cuda.open_session("Product", 0, 1, components=spec).import_state_dev(buf.data_ptr(), nbytes, N, d)
    with pytest.raises(backend.GpsoBackendError, match="kernel mismatch"):
        cuda.open_session("Matern32", 4, True).import_state_dev(buf.data_ptr(), nbytes, N, d)
    # the same factor list as a sum, in both directions: the state sizes agree, the kernel id does not
    with pytest.raises(backend.GpsoBackendError, match="kernel mismatch"):
        cuda.open_session("Sum", 0, 1, components=comp_spec).import_state_dev(buf.data_ptr(), nbytes, N, d)
    sm = cuda.open_session("Sum", 0, 1, components=comp_spec)
    sm.set_data(X, y)
    sm.factorize(h.theta())
    assert sm.state_bytes() == nbytes
    sbuf = torch.empty(nbytes, dtype=torch.uint8, device=f"cuda:{cuda.device}")
    sm.export_state_dev(sbuf.data_ptr(), nbytes)
    torch.cuda.synchronize()
    with pytest.raises(backend.GpsoBackendError, match="kernel mismatch"):
        cuda.open_session("Product", 0, 1, components=comp_spec).import_state_dev(sbuf.data_ptr(), nbytes, N, d)
    for s in (a, b, sm):
        s.close()


# ---- every screened value within E / 4 of the exact UCB ---------------------------------------------------------------------
@pytest.mark.parametrize("case", ["four", "var1e-8", "var1e8"])
def test_every_screened_value_within_a_quarter_of_the_bound(cuda, case):
    """Forced screens 2, 3, 4 and 6 and the mean-bound level: |screened - exact| <= E / 4 for every candidate, with E the
    handle's own bound (screen_info) and the exact UCB from the unscreened predict_y.  var_prod = 1e-8 and 1e8 come from four
    factors of 1e-2 and 1e2, so the fp32 screen sees the product variance on the first factor only."""
    N, d, M = 1100, 3, 70_000
    scale = {"four": 1.0, "var1e-8": 1e-4, "var1e8": 1e4}[case]
    X, y = synthetic(N, d, seed=N + 7)
    y = y * scale
    if case == "four":
        comp = comps("four", d)
    else:
        v = 1e-2 if case == "var1e-8" else 1e2
        comp = [po.Comp(f, 0.6, v) for f in ("Matern52", "SquaredExponential", "Matern32", "Matern12")]
    h = po.ProductHyper(comp, 1e-3 * h_var(comp), 0.05 * scale)
    Xc = np.random.default_rng(M).random((M, d))
    s = session(cuda, h, X, y)
    s.set_screen_mode(0)
    s.factorize(h.theta())
    mean, var = s.predict_y(Xc)
    checked = 0
    for mode in (2, 3, 4, 6, 5):
        s.set_screen_mode(mode)
        s.factorize(h.theta())
        rec = s.ucb_argmax(Xc, VARSIGMA)
        info = s.screen_info()
        if info["path"] not in ("screened", "mean-bound"):
            continue
        u = s.screened_values(M)
        exact = mean if info["path"] == "mean-bound" else mean + VARSIGMA * var
        assert np.all(np.isfinite(u))
        ratio = float(np.max(np.abs(u - exact)) / info["error_bound"])
        assert ratio <= 0.25, (mode, ratio, info)
        assert rec[0] == int(np.argmax(mean + VARSIGMA * var))
        checked += 1
    assert checked >= 4
    s.close()


def h_var(comp):
    v = 1.0
    for c in comp:
        v *= c.variance
    return v
