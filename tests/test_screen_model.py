"""
Error model of the screen-and-refine arg-max (pygpso_b200/csrc/kern_screen.cuh, gpso_capi.cu: screen_error_model), checked
on the CPU against a numpy emulation of the screening arithmetic: balanced 8-bit digits of L^-1 (per-row power-of-two scale)
and of a float32 cross-covariance, exact integer digit-pair products of the retained levels, float32 epilogue.

The product path never runs this code; it pins the C formula (called through the host-only entry ``gpso_debug_screen_bound``)
so that a change of either side shows up without a GPU.
"""
import ctypes

import numpy as np
import pytest
import scipy.linalg as sl

from oracle import gpr_oracle as go
from pygpso_b200 import backend

VARSIGMA = go.VARSIGMA_DEFAULT


def digits_of(X, S):
    """Balanced base-256 digits (most significant first) of integer array |X| < 2^(8S-2)."""
    C = sum(0x80 << (8 * b) for b in range(S - 1))
    Z = (X.astype(np.int64) + C) ^ C
    out = []
    for p in range(S):
        byte = (Z >> (8 * (S - 1 - p))) & 0xFF
        out.append(((byte + 128) % 256 - 128).astype(np.float64))
    # the top digit keeps the sign of X (arithmetic shift of the remaining bits)
    out[0] = (Z >> (8 * (S - 1))).astype(np.float64)
    return out


def cov32(kernel, r2, var):
    r2 = r2.astype(np.float32)
    var = np.float32(var)
    if kernel == "SquaredExponential":
        return var * np.exp(np.float32(-0.5) * r2)
    r = np.sqrt(np.maximum(r2, np.float32(1e-36)))
    if kernel == "Matern52":
        s = np.float32(2.2360679775) * r
        return var * (np.float32(1) + s + np.float32(1.6666666667) * (r * r)) * np.exp(-s)
    if kernel == "Matern32":
        s = np.float32(1.7320508076) * r
        return var * (np.float32(1) + s) * np.exp(-s)
    return var * np.exp(-r)


def emulate_screen(kernel, X, y, h, Xc, S, full=False, A=None):
    """h.mean_c: the constant of the mean (None: zero mean); A: the slope of a linear mean x . A + mean_c."""
    N = X.shape[0]
    c = h.mean_c if h.has_mean else 0.0
    off, off_c = (X @ A, Xc @ A) if A is not None else (0.0, 0.0)
    K = go.kern(kernel, X, None, h) + h.noise_variance * np.eye(N)
    L = np.linalg.cholesky(K)
    Linv = sl.solve_triangular(L, np.eye(N), lower=True)
    alpha = sl.cho_solve((L, True), (y[:, 0] - c) - off)
    rowmax = np.abs(Linv).max(axis=1)
    rowscale = np.ldexp(1.0, np.frexp(rowmax)[1])  # 2^(ilogb(max)+1)
    beta = np.ldexp(1.0, int(np.floor(np.log2(h.variance))) + 1)
    XA = np.rint(Linv * (2.0 ** (8 * S - 2) / rowscale)[:, None])
    a = digits_of(XA, S)
    ls = np.atleast_1d(h.lengthscales)
    Xs32 = (X / ls).astype(np.float32)
    Cs32 = (Xc / ls).astype(np.float32)
    diff = Xs32[:, None, :] - Cs32[None, :, :]
    r2 = np.einsum("ijk,ijk->ij", diff, diff, dtype=np.float32)
    k32 = cov32(kernel, r2, h.variance)
    XB = np.rint(k32.astype(np.float64) * np.float32(2.0 ** (8 * S - 2) / beta)).astype(np.int64)
    b = digits_of(XB, S)
    acc = np.zeros((N, Xc.shape[0]))
    top = 2 * S - 2 if full else S - 1  # highest digit-pair level kept (full product: all S^2 pairs)
    for p in range(S):
        for q in range(S if full else S - p):
            acc += (a[p] @ b[q]) * 256.0 ** (top - (p + q))  # exact integers in float64
    gscale = beta * 2.0 ** (-2 * (8 * S - 2) + 8 * (S - 1) - 8 * (top - (S - 1)))
    v = (acc.astype(np.float32) * (rowscale * gscale).astype(np.float32)[:, None]).astype(np.float32)
    ss = (v * v).astype(np.float32).sum(axis=0, dtype=np.float32).astype(np.float64)
    var_s = (h.variance - ss) + h.noise_variance
    mean_s = (k32.astype(np.float32).T @ alpha.astype(np.float32)).astype(np.float64) + c + off_c
    # exact
    Ks = go.kern(kernel, X, Xc, h)
    V = Linv @ Ks
    var = (h.variance - (V * V).sum(0)) + h.noise_variance
    mean = Ks.T @ alpha + c + off_c
    rowl2 = np.sqrt((Linv ** 2).sum(axis=1))
    info = {"rho_max": float(rowscale.max()), "rho_l2sq": float((rowscale ** 2).sum()), "rowl2_max": float(rowl2.max()),
            "frob2": float((Linv ** 2).sum()), "alpha_l2": float(np.linalg.norm(alpha)), "k32_err": float(np.abs(k32 - Ks).max()),
            "Linv": Linv, "alpha": alpha}
    return mean_s, var_s, mean, var, info


def c_bound(N, variance, noise, info, S, varsigma, full=False):
    lib = backend.load_library()
    out = (ctypes.c_double * 3)()
    fit5 = (ctypes.c_double * 5)(info["rho_max"], info["rho_l2sq"], info["rowl2_max"], info["frob2"], info["alpha_l2"])
    rc = lib.gpso_debug_screen_bound(N, variance, noise, fit5, S, int(full), varsigma, out)
    assert rc == 0
    return tuple(out)


CONSTANT_MEAN_CASES = [
    ("Matern52", 768, 5, 0.25 * np.sqrt(5), 1.0, 1e-3),
    ("Matern52", 512, 10, 0.25 * np.sqrt(10), 1.0, 1e-3),
    ("Matern52", 512, 3, 0.3, 2.5, 2e-6),       # ill-conditioned: noise near the floor, large row scales
    ("SquaredExponential", 512, 4, 0.5, 0.7, 1e-3),
    ("Matern32", 512, 4, 0.5, 1.3, 1e-2),
    ("Matern12", 512, 4, 0.5, 1.0, 1e-3),
]
CASES = [pytest.param(*c, "constant", id="-".join(map(str, c))) for c in CONSTANT_MEAN_CASES] + [
    ("Matern52", 600, 4, [0.3, 0.45, 0.6, 0.9], 1.0, 1e-3, "constant"),  # ARD lengthscales
    ("SquaredExponential", 513, 2, [0.2, 0.35], 1.0, 1e-3, "zero"),      # 513 rows: 127 padding rows in the last block
    ("Matern12", 700, 6, 0.6, 1.0, 1e-3, "linear"),
    ("Matern52", 600, 4, 0.5, 1e-8, 1e-11, "constant"),     # y, noise and mean scaled with the kernel variance
    ("Matern52", 600, 4, 0.5, 1e8, 1e5, "constant"),
]


@pytest.mark.parametrize("kernel,N,d,ls,variance,noise,mean", CASES)
@pytest.mark.parametrize("S,full", [(2, False), (3, False), (4, False), (2, True)])
def test_screen_error_bound_holds_with_margin(kernel, N, d, ls, variance, noise, mean, S, full):
    from tests.screen_oracle import ScreenOracle

    rng = np.random.default_rng(20240517)
    X = rng.random((N, d))
    scale = variance if variance < 1e-3 or variance > 1e3 else 1.0
    y = scale * (np.sin(3.0 * X.sum(axis=1)) + 0.01 * rng.standard_normal(N))[:, None]
    A = np.linspace(0.6, -0.4, d) if mean == "linear" else None
    h = go.Hyper(ls, variance, noise, None if mean == "zero" else 0.1 * scale)
    Xc = np.vstack([rng.random((1500, d)), X[:100] + 1e-5 * rng.standard_normal((100, d))])
    mean_s, var_s, mean, var, info = emulate_screen(kernel, X, y, h, Xc, S, full, A)
    E, e_var, e_mean = c_bound(N, variance, noise, info, S, VARSIGMA, full)
    assert info["k32_err"] <= 1.0e-6 * variance  # the model assumes 2e-6 * variance for the fp32 covariance
    # the emulation in the device's order of operations (the GPU tests' reference) is held to the same margin
    so = ScreenOracle(kernel, X, info["Linv"], info["alpha"], ls, variance, noise, h.mean_c or 0.0, A)
    assert np.allclose(so.fit5, [info[k] for k in ("rho_max", "rho_l2sq", "rowl2_max", "frob2", "alpha_l2")], rtol=1e-12, atol=0)
    mean_o, var_o = so.screen(Xc, [(S, full)])[(S, full)]
    for ms, vs in ((mean_s, var_s), (mean_o, var_o)):
        dv = np.abs(vs - var).max()
        dm = np.abs(ms - mean).max()
        du = np.abs((ms + VARSIGMA * vs) - (mean + VARSIGMA * var)).max()
        # the run-time check demands observed <= E / 4; the emulation must sit comfortably inside that
        assert dv <= e_var / 8.0, (dv, e_var)
        assert dm <= e_mean / 8.0, (dm, e_mean)
        assert du <= E / 8.0, (du, E)


def test_digits_reconstruct():
    rng = np.random.default_rng(1)
    for S in (2, 3, 4):
        X = rng.integers(-(2 ** (8 * S - 2)) + 1, 2 ** (8 * S - 2), size=1000)
        dig = digits_of(X, S)
        assert all(np.all((dg >= -128) & (dg <= 127)) for dg in dig)
        recon = sum(dg * 256.0 ** (S - 1 - p) for p, dg in enumerate(dig))
        assert np.array_equal(recon, X.astype(np.float64))
