"""
Screened value of EVERY candidate against the fp64 posterior and against an emulation of the screening arithmetic.

The screen-and-refine arg-max (kern_screen.cuh, DESIGN 3.5) discards a candidate when its screened UCB lies more than 2E below
the best screened value; the run-time check compares screened and refined values of the survivors only.  The property the
design rests on is per candidate:  |screened UCB(c) - exact UCB(c)| <= E  for every c.  These tests fetch the screened value
of every candidate of a fused call (``screened_values``) and check, per case and screening level:

  (a) every finite screened UCB against the exact UCB (the engine's unscreened predict_y, itself re-anchored to the numpy
      oracle on a subsample): <= E / 4, the margin the run-time check demands of the survivors
  (b) the screened mean (a varsigma = 0 call) and the screened variance ((u(varsigma) - u(0)) / varsigma) separately:
      <= e_mean / 4 and <= e_var / 4 -- tells the cross-covariance stage from the product stage
  (c) a subsample against tests/screen_oracle.py (device order of operations, numpy's fp32 exp / sqrt instead of MUFU): <= E / 16
  (d) E recomputed from the handle's own L^-1 and alpha through gpso_debug_screen_bound
  (e) the selection, exactly: best screened value, survivor count, the finite exact winner among the survivors, the record
  (f) NaN exactly at the rows with a NaN, an infinite or a too large (|x / l| > 1e15) coordinate
and that the values do not depend on the window size, the stream overlap, where the candidates live or their position in
the batch.
"""
import ctypes

import numpy as np
import pytest

from oracle import gpr_oracle as go
from pygpso_b200 import backend
from tests import linear_mean_oracle as lo
from tests import rq_oracle as rq
from tests.screen_oracle import exact_predict_y, oracle_for
from tests.test_gpu_parity import assert_predict_close
from tests.test_gpu_screen import same_record
from tests.test_screen_windows import windows

pytestmark = pytest.mark.gpu

VARSIGMA = go.VARSIGMA_DEFAULT
LEVEL_OF_MODE = {2: (2, False), 3: (3, False), 4: (4, False), 6: (2, True)}  # forced digit screens; 5 = mean-bound level first
MODES = (2, 3, 4, 6, 5)


@pytest.fixture(scope="module")
def cuda():
    return backend.default_backend()


def same_bytes(a, b):
    return a.shape == b.shape and a.tobytes() == b.tobytes()


def synthetic(N, d, seed, scale=1.0, trend=False):
    rng = np.random.default_rng(seed)
    X = rng.random((N, d))
    y = np.sin(3 * X.sum(1)) + 0.01 * rng.standard_normal(N)
    if trend:
        y = y + 0.8 * X[:, 0] - 0.5 * X[:, -1]
    return X, scale * y[:, None]


# ---- the cases ----------------------------------------------------------------------------------------------------------
# id: N, d, kernel, lengthscale(s), variance, noise, mean ("zero" | "constant" | "linear"), M, extra options
CASES = {
    "n512-m52": (512, 3, "Matern52", None, 1.0, 1e-3, "constant", 65_536, {"varsigmas": (-1.0, 50.0)}),
    "n513-se-ard-zero": (513, 2, "SquaredExponential", [0.3, 0.45], 1.0, 1e-3, "zero", 65_537, {}),
    "n1100-m32": (1100, 4, "Matern32", None, 1.0, 1e-3, "constant", 70_001, {}),
    # the engine's fp64 mean and numpy's differ by up to 1.1e-8 relative here (Matern12, N = 2100): 1e4 below e_mean
    "n2100-m12-ard-linear": (2100, 6, "Matern12", list(0.3 + 0.1 * np.arange(6)), 1.0, 1e-3, "linear", 150_000, {"anchor_rel": 1e-7}),
    "n1100-rq0.5-linear": (1100, 5, rq.KERNEL, None, 1.0, 1e-3, "linear", 80_000, {"rq_alpha": 0.5}),
    "n1100-rq1e4-linear": (1100, 5, rq.KERNEL, None, 1.0, 1e-3, "linear", 80_000, {"rq_alpha": 1e4}),
    "n700-d1": (700, 1, "Matern52", None, 1.0, 1e-3, "constant", 70_000, {}),
    "n600-d64-ard": (600, 64, "Matern52", list(np.linspace(1.5, 3.0, 64)), 1.0, 1e-3, "constant", 66_000, {}),
    # ill-conditioned: noise near its floor, large row scales of L^-1 (case 3 of test_screen_model.py)
    "n512-illcond": (512, 3, "Matern52", 0.3, 2.5, 2e-6, "constant", 70_000, {"anchor_rel": 1e-6}),
    "n1100-var1e-8": (1100, 4, "Matern52", None, 1e-8, 1e-11, "constant", 70_000, {"scale": 1e-8}),
    "n1100-var1e8": (1100, 4, "Matern52", None, 1e8, 1e5, "constant", 70_000, {"scale": 1e8}),
    "c3": (4096, 10, "Matern52", None, 1.0, 1e-3, "constant", 400_000, {"c3": True}),
    # Np = OZ_MAX_NP: L^-1 from the hybrid factorisation, two screening windows at S >= 3
    "n8192-m52": (8192, 8, "Matern52", None, 1.0, 1e-3, "constant", 100_000, {}),
}


def build_case(name):
    N, d, kernel, ls, variance, noise, mean, M, opt = CASES[name]
    ls = 0.25 * np.sqrt(d) if ls is None else ls
    scale = opt.get("scale", 1.0)
    if opt.get("c3"):
        import bench

        X, y = bench.synthetic_training(N, d)
        assert np.allclose(bench.fixed_theta(d), [ls, variance, noise, 0.0])
    else:
        X, y = synthetic(N, d, seed=N + d, scale=scale, trend=mean == "linear")
    c = None if mean != "constant" else (0.0 if opt.get("c3") else 0.05 * scale)
    hk = rq.RQHyper(opt["rq_alpha"], ls, variance, noise, c) if kernel == rq.KERNEL else go.Hyper(ls, variance, noise, c)
    if mean == "linear":
        h = lo.LinearHyper(hk, np.linspace(0.6, -0.4, d), 0.1)
        theta, mean_id = h.theta(), lo.MEAN_ID
    else:
        h = hk
        t = ([hk.alpha] if kernel == rq.KERNEL else []) + list(hk.lengthscales) + [variance, noise]
        theta, mean_id = np.array(t + ([c] if c is not None else [])), int(c is not None)
    return X, y, h, kernel, theta, mean_id, M, opt


def candidates(name, X, h, M):
    """Uniform rows in the box, rows at training points (exact and with 1e-6 jitter), far-away rows, and the rows that must
    screen to NaN (and one just inside the fp32-safe range).  Returns (Xc, rows expected NaN, the row at 0.99e15 l or None)."""
    N, d = X.shape
    rng = np.random.default_rng(M + d)
    if CASES[name][8].get("c3"):
        import bench

        Xc = np.empty((M, d))
        bench.fill_candidates(Xc, 0, M, bench.WORKLOADS["c3"][2], d)
    else:
        Xc = rng.random((M, d))
    n = min(N, 400)
    pos = rng.choice(M, size=2 * n + 64, replace=False)
    Xc[pos[:n]] = X[:n]
    Xc[pos[n:2 * n]] = X[:n] + 1e-6 * rng.standard_normal((n, d))
    Xc[pos[2 * n:]] = 3.0 + rng.random((64, d))
    ls = np.broadcast_to((h.k if isinstance(h, lo.LinearHyper) else h).lengthscales, (d,))
    ls0 = ls[0]
    bad = {7: np.nan, 1000: np.inf, M // 2 + 1: 1e300, M - 2: 1.01e15, 64 * 300: -np.inf}
    for r, v in bad.items():
        Xc[r] = rng.random(d)
        Xc[r, r % d] = v * ls[r % d] if np.isfinite(v) else v  # 1.01e15 / 1e300: in units of that coordinate's lengthscale
    inside = None
    if not isinstance(h, lo.LinearHyper):  # (a linear mean makes it the winner by 1e15: no fp64 comparison resolves that)
        inside = M - 300
        Xc[inside] = rng.random(d)
        Xc[inside, 0] = 0.99e15 * ls0
    return Xc, np.array(sorted(bad)), inside


def subsample(M, Np, u, nan_rows, budget, rng):
    """Rows for the emulation: first and last, window edges of every digit count (automatic windows, with and without the
    ramp), rows next to the NaN rows, the 256 best exact UCBs, 64- and 128-candidate tile edges, random rows."""
    must = {0, M - 1}
    for S in (2, 3, 4):
        W = (2 ** 31 // (Np * S)) // 1024 * 1024
        for ramp in ((True, False) if W < M else ()):  # else one window of all candidates
            for off, n in windows(M, W, ramp, True):
                must |= {off - 1, off, off + n - 1}
    for r in nan_rows:
        must |= {r - 1, r + 1}
    must |= set(np.argsort(-np.nan_to_num(u, nan=-np.inf))[:256].tolist())
    edges = np.arange(64, M, 64)
    edges = np.concatenate([edges - 1, edges, edges[:8] - 1, edges[:8], edges[-8:]])
    rest = max(budget - len(must), 64)
    extra = np.concatenate([rng.choice(edges, size=min(rest // 2, edges.size), replace=False), rng.choice(M, size=rest - rest // 2)])
    sel = np.array(sorted((must | set(extra.tolist())) - set(nan_rows.tolist())))
    return sel[(sel >= 0) & (sel < M)]


def c_bound(N, variance, noise, fit5, S, full, varsigma):
    lib = backend.load_library()
    out = (ctypes.c_double * 3)()
    assert lib.gpso_debug_screen_bound(N, variance, noise, (ctypes.c_double * 5)(*fit5), S, int(full), varsigma, out) == 0
    return tuple(out)


def level_of(mode, info):
    """The screening level whose values scr_ucb holds after the call: (S, all pairs), or 0 for the mean-bound level."""
    if info["path"] == "mean-bound":
        return 0
    if mode in LEVEL_OF_MODE:
        return LEVEL_OF_MODE[mode]
    return (info["digits"], info["all_pairs"])


def check_call(s, mode, vs, rec, ref, M, mean, var, nan_rows, inside, hk, so, N):
    """Checks (a), (d), (e), (f) of one fused call.  Returns (level, screened values or None, E parts, ratio (a))."""
    info = s.screen_info()
    assert same_record(rec, ref), (mode, vs, rec, ref, info)
    try:
        u = s.screened_values(M)
    except backend.GpsoBackendError:  # the early stop after window 1 (too many survivors): nothing to compare past it
        assert info["path"].startswith("full pass"), info
        return None, None, None, None
    lev = level_of(mode, info)
    # (f) NaN exactly at the rows with a NaN, infinite or too large coordinate; nothing infinite
    assert np.array_equal(np.flatnonzero(~np.isfinite(u)), nan_rows), (mode, np.flatnonzero(~np.isfinite(u))[:20])
    assert np.all(np.isnan(u[nan_rows]))
    if inside is not None:
        assert np.isfinite(u[inside])
    # (d) the error bound from the handle's own L^-1 and alpha
    E, e_var, e_mean = c_bound(N, hk.variance, hk.noise_variance, so.fit5, 4 if lev == 0 else lev[0], 0 if lev == 0 else lev[1], vs)
    if lev == 0:
        E = e_mean
        assert abs(info["error_bound"] - e_mean) <= 1e-10 * e_mean, (info, e_mean)
        slack = 2.0 * e_mean + abs(vs) * hk.variance * (1.0 + 2.0e-6)
        exact = mean
    else:
        for got, want in ((info["error_bound"], E), (info["e_var"], e_var), (info["e_mean"], e_mean)):
            assert abs(got - want) <= 1e-10 * want, (info, E, e_var, e_mean)
        slack = 2.0 * E
        exact = mean + vs * var
    # (a) every finite candidate
    fin = np.isfinite(u)
    ratio_a = float(np.max(np.abs(u[fin] - exact[fin])) / E)
    assert ratio_a <= 0.25, (mode, vs, ratio_a, int(np.flatnonzero(fin)[np.argmax(np.abs(u[fin] - exact[fin]))]))
    # (e) the selection, exactly
    best = np.nanmax(u)
    assert np.array([best]).tobytes() == np.array([info["best_screened_ucb"]]).tobytes(), (best, info)
    thr = best - slack
    surv = ~(u < thr)
    assert int(surv.sum()) == info["survivors"], (int(surv.sum()), info)
    w = int(np.flatnonzero(fin)[np.argmax(exact[fin])])  # the best candidate the screen had to keep
    assert surv[w], (w, u[w], thr)
    return lev, u, (E, e_var, e_mean), ratio_a


@pytest.mark.parametrize("name", list(CASES))
def test_every_screened_value(cuda, name):
    X, y, h, kernel, theta, mean_id, M, opt = build_case(name)
    hk = h.k if isinstance(h, lo.LinearHyper) else h
    N, d = X.shape
    Np = (N + 127) // 128 * 128
    Xc, nan_rows, inside = candidates(name, X, h, M)
    varsigmas = (VARSIGMA, 0.0) + tuple(opt.get("varsigmas", ()))
    s = cuda.open_session(kernel, hk.lengthscales.size, mean_id)
    s.set_data(X, y)
    s.set_screen_mode(0)
    s.factorize(theta)
    mean, var = s.predict_y(Xc)
    refs = {vs: s.ucb_argmax(Xc, vs) for vs in varsigmas}
    with pytest.raises(backend.GpsoBackendError, match="screened 0 candidates"):  # unscreened call: no screened values
        s.screened_values(1)
    Linv, alpha = s.debug_fetch(2), s.debug_fetch(3)
    so = oracle_for(kernel, X, Linv, alpha, h)
    # the engine's exact values, re-anchored to the fp64 oracle (finite rows, the best ones among them)
    rng = np.random.default_rng(N)
    u_exact = mean + VARSIGMA * var
    fin = np.flatnonzero(np.isfinite(u_exact) & (np.abs(Xc).max(axis=1) < 1e6))
    anchor = np.unique(np.concatenate([rng.choice(fin, 150, replace=False), fin[np.argsort(-u_exact[fin])[:50]]]))
    m_o, v_o = exact_predict_y(kernel, X, y, h, Xc[anchor])
    assert_predict_close(mean[anchor], var[anchor], m_o, v_o, y, hk.variance, rel=opt.get("anchor_rel", 1e-8))
    # the emulation of every level on one subsample
    budget = 2048 if N <= 2100 else (1024 if N <= 4096 else 160)
    sub = subsample(M, Np, u_exact, nan_rows, budget, rng)
    emul = so.screen(Xc[sub], [0, (2, False), (3, False), (4, False), (2, True)])
    report = []
    means = {}
    for mode in MODES:
        s.set_screen_mode(mode)
        s.factorize(theta)
        got = {}
        for vs in varsigmas:
            rec = s.ucb_argmax(Xc, vs)
            got[vs] = check_call(s, mode, vs, rec, refs[vs], M, mean, var, nan_rows, inside, hk, so, N)
        lev, u1, (E, e_var, e_mean), ra = got[VARSIGMA] if got[VARSIGMA][1] is not None else (None, None, (0, 0, 0), None)
        lev0, u0, bounds0, _ = got[0.0]
        row = {"mode": mode, "a": ra}
        if u0 is not None:
            means[mode] = u0
            fin0 = np.isfinite(u0)
            # (b) the screened mean of every candidate
            row["b_mean"] = float(np.max(np.abs(u0[fin0] - mean[fin0])) / bounds0[2])
            assert row["b_mean"] <= 0.25, (mode, row)
            # (c) the emulated mean
            em0 = emul[0][0]
            row["c_mean"] = float(np.max(np.abs(u0[sub] - em0)) / bounds0[2])
            assert row["c_mean"] <= 1.0 / 16.0, (mode, row)
        if u1 is not None and u0 is not None and lev == lev0 and lev != 0:
            # (b) the screened variance, recovered from the two calls of the same level
            vs_rec = (u1 - u0) / VARSIGMA
            fin1 = np.isfinite(u1)
            row["b_var"] = float(np.max(np.abs(vs_rec[fin1] - var[fin1])) / e_var)
            assert row["b_var"] <= 0.25, (mode, row)
        for vs, (lev_v, u_v, bnd, _) in got.items():
            if u_v is None or vs == 0.0:
                continue
            # (c) the emulated UCB at the level the call ended on
            em_m, em_v = emul[lev_v]
            em_u = em_m if lev_v == 0 else em_m + vs * em_v
            r = float(np.max(np.abs(u_v[sub] - em_u)) / bnd[0])
            row["c" if vs == VARSIGMA else f"c@{vs:g}"] = r
            assert r <= 1.0 / 16.0, (mode, vs, lev_v, r, int(sub[np.argmax(np.abs(u_v[sub] - em_u))]))
        report.append(row)
    s.close()
    # the bound-level mean (mode 5) and the varsigma = 0 value of every digit screen come from the same kernel body
    first = next(iter(means.values()))
    for mode, u0 in means.items():
        assert same_bytes(u0, first), mode
    for row in report:
        print(f"SCREEN-VALUES {name} " + " ".join(f"{k}={v:.3g}" if isinstance(v, float) else f"{k}={v}" for k, v in row.items()))


# ---- the values do not depend on windows, overlap, candidate residence or batch position -------------------------------------
def separable_problem(cuda, mode):
    """test_gpu_screen.py's window problem: modes 3 and 4 screen it without a full pass (no early stop cuts a pass short)."""
    N, d, M = 1100, 4, 90_000
    X, y = synthetic(N, d, seed=8)
    s = cuda.open_session("Matern52", 1, True)
    s.set_data(X, y)
    s.set_screen_mode(mode)
    s.factorize(np.array([0.5, 1.0, 1e-3, 0.0]))
    return s, np.random.default_rng(9).random((M, d))


@pytest.mark.parametrize("mode", [3, 4])
def test_values_independent_of_windows_and_batch(cuda, mode):
    import torch

    s, Xc = separable_problem(cuda, mode)
    M = Xc.shape[0]
    ref = s.ucb_argmax(Xc, VARSIGMA)
    assert s.screen_info()["path"] == "screened"
    base = s.screened_values(M)

    def again(label, **kw):
        got = s.ucb_argmax_dev(kw["xd"].data_ptr(), M, VARSIGMA, torch.cuda.current_stream().cuda_stream) if "xd" in kw else \
            s.ucb_argmax(Xc, VARSIGMA)
        info = s.screen_info()
        assert same_record(ref, got) and info["path"] == "screened", (label, info)
        assert same_bytes(s.screened_values(M), base), label
        return info

    for W in (1024, 16_384):
        s.set_window(W)
        assert again(f"window {W}")["screen_windows"] == (M + W - 1) // W
    s.set_overlap(False)
    again("window 16384, no overlap")
    s.set_overlap(True)
    s.set_window(0)
    again("device candidates", xd=torch.from_numpy(Xc).cuda())
    Xp = np.vstack([np.random.default_rng(1).random((777, Xc.shape[1])), Xc])
    s.ucb_argmax(Xp, VARSIGMA)
    assert same_bytes(s.screened_values(M + 777)[777:], base)
    s.close()


def test_mean_bound_values_independent_of_windows(cuda):
    """Mode 5 at varsigma = 0 (the bound level takes every call): one bound window, sixteen of 16384 rows, and a batch above
    2^19 rows (two automatic bound windows) whose first rows are the same candidates."""
    s, Xc = separable_problem(cuda, 5)
    M = Xc.shape[0]
    s.ucb_argmax(Xc, 0.0)
    assert s.screen_info()["path"] == "mean-bound"
    base = s.screened_values(M)
    s.set_window(16_384)
    s.ucb_argmax(Xc, 0.0)
    info = s.screen_info()
    assert info["path"] == "mean-bound" and info["screen_windows"] == (M + 16_383) // 16_384, info
    assert same_bytes(s.screened_values(M), base)
    s.set_window(0)
    big = np.vstack([Xc, np.random.default_rng(2).random((600_000 - M, Xc.shape[1]))])
    s.ucb_argmax(big, 0.0)
    info = s.screen_info()
    assert info["path"] == "mean-bound" and info["screen_windows"] == 2, info
    assert same_bytes(s.screened_values(big.shape[0])[:M], base)
    s.close()


@pytest.mark.parametrize("mode", [3, 4])
def test_leaf_batch_values(cuda, mode):
    """grow(12) leaves scored by gpso_grow_ucb_argmax, whole and split in two row ranges, screen to the values of
    ucb_argmax on the same leaves."""
    s, _ = separable_problem(cuda, mode)
    bounds = np.array([[0.0, 1.0]] * 4)
    leaves = cuda.grow_leaves(bounds, 12)
    total = leaves.shape[0]
    ref = s.ucb_argmax(leaves, VARSIGMA)
    base = s.screened_values(total)
    assert same_record(s.grow_ucb_argmax(bounds, 12, VARSIGMA), ref)
    assert same_bytes(s.screened_values(total), base)
    cut = 130_000  # both halves >= 65 536 rows: both are screened
    for r0, r1 in ((0, cut), (cut, total)):
        s.grow_ucb_argmax(bounds, 12, VARSIGMA, rows=(r0, r1))
        assert s.screen_info()["path"] != "unscreened"
        assert same_bytes(s.screened_values(r1 - r0), base[r0:r1]), (r0, r1)
    s.close()


def test_screened_values_refused_when_stale(cuda):
    """After the early stop only the windows that ran hold values; after an unscreened call none do."""
    N, d, M = 1100, 3, 70_000
    X, y = synthetic(N, d, seed=2)
    Xc = 50.0 + np.random.default_rng(5).random((M, d))  # plateau: no screen separates these candidates
    s = cuda.open_session("Matern52", 1, True)
    s.set_data(X, y)
    s.set_screen_mode(2)
    s.factorize(np.array([0.05, 1.0, 1e-3, 0.0]))
    s.set_window(1024)
    s.ucb_argmax(Xc, VARSIGMA)
    info = s.screen_info()
    assert info["path"].startswith("full pass") and info["screen_windows"] == 2, info
    assert np.all(np.isfinite(s.screened_values(2048)))
    with pytest.raises(backend.GpsoBackendError, match="screened 2048 candidates"):
        s.screened_values(2049)
    s.set_screen_mode(0)
    s.factorize(np.array([0.05, 1.0, 1e-3, 0.0]))
    s.ucb_argmax(Xc, VARSIGMA)
    with pytest.raises(backend.GpsoBackendError, match="screened 0 candidates"):
        s.screened_values(1)
    s.close()
