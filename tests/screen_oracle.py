"""
Reference of one screening level of the screen-and-refine arg-max (pygpso_b200/csrc/kern_screen.cuh) in numpy, for the GPU
tests that compare the device's screened value of every candidate (test_gpu_screen_values.py).

It starts from the handle's own L^-1 and alpha (``debug_fetch(2)`` / ``debug_fetch(3)``), so the rounding of the factorisation
is not part of the comparison, and follows the device's order of operations wherever it changes the result:

  mean (crosscov_screen_kernel)   fp32 covariance, 16-term fp32 fma chains per warp slice of a 128-point super-step, fp64
                                  accumulation across super-steps, the fixed 8-way tree, + c0, + the fp64 x . A offset (Linear)
  variance (ozaki_screen_kernel)  balanced 8-bit digits of L^-1 (power-of-two row scale) and of the fp32 covariance, exact
                                  integer digit-pair levels, each converted to fp32 and chained with fmaf(w, 256, level), times
                                  the fp32 row scale, squared, summed in fp32 per 128-row block (the warp-shuffle tree), blocks
                                  summed in fp64 (screen_finalize_kernel), then (variance - ss) + noise.

The fp32 covariance follows cov32x2_from_r2 operation by operation (exp(-s) as 2^(s * -log2 e), r = c * rsqrt(c), the
Matern polynomials' fma): the order matters, since rounding s * log2 e alone costs up to s ulp of the covariance, as much as
the whole screening error of the mean.  What is left to differ is the approximation error of MUFU.EX2 / MUFU.RSQ / MUFU.LG2
and of __fdividef (a few ulp per value); here those are exact results rounded to fp32.  A candidate with a NaN, an infinite
or a scaled coordinate beyond 1e15 gets a NaN screened value.
"""
import numpy as np

from oracle import gpr_oracle as go
from tests import linear_mean_oracle as lo
from tests import rq_oracle as rq
from tests.test_screen_model import digits_of

XK = 128  # training points per super-step of the cross-covariance kernel (OZ_XK)
F32 = np.float32
L2E = F32(1.4426950408889634)


def _ex2(t):
    """ex2.approx.ftz.f32, correctly rounded: subnormal results flush to zero."""
    with np.errstate(over="ignore", under="ignore"):
        e = np.exp2(t.astype(np.float64)).astype(F32)
    return np.where(e < F32(2.0 ** -126), F32(0), e)


def _fma(a, b, c):
    return (a.astype(np.float64) * b + c).astype(F32)  # the product is exact in fp64


def cov32_device(kernel, r2, variance, rq_alpha=None):
    """kern_screen.cuh cov32x2_from_r2 in numpy float32, in the device's order of operations."""
    r2 = r2.astype(F32)
    var = F32(variance)
    with np.errstate(over="ignore", invalid="ignore", divide="ignore"):
        if kernel == rq.KERNEL:
            a = F32(rq_alpha)
            z = (r2 * (F32(0.5) / a)).astype(F32)
            p = np.full_like(z, rq.RQ32_P[5])
            for coef in rq.RQ32_P[4::-1]:
                p = _fma(p, z, coef)
            p = (p * z).astype(F32)
            lg = np.log2((z + F32(1)).astype(np.float64)).astype(F32)
            l2 = np.where(z < rq.RQ32_SPLIT, p, lg)
            return (var * _ex2((l2 * -a).astype(F32))).astype(F32)
        if kernel == "SquaredExponential":
            return (var * _ex2((r2 * F32(-0.5 * L2E)).astype(F32))).astype(F32)
        c = np.where(r2 < F32(1e-36), F32(1e-36), r2)  # a select: NaN propagates
        r = (c * (1.0 / np.sqrt(c.astype(np.float64))).astype(F32)).astype(F32)
        if kernel == "Matern52":
            s = (r * F32(2.2360679775)).astype(F32)
            e = _ex2((s * -L2E).astype(F32))
            poly = (_fma((r * r).astype(F32), F32(1.6666666667), s) + F32(1)).astype(F32)
            return ((var * poly).astype(F32) * e).astype(F32)
        if kernel == "Matern32":
            s = (r * F32(1.7320508076)).astype(F32)
            e = _ex2((s * -L2E).astype(F32))
            return ((var * (s + F32(1)).astype(F32)).astype(F32) * e).astype(F32)
        return (var * _ex2((r * -L2E).astype(F32))).astype(F32)


def fit5(Linv, alpha):
    """What gpso_debug_screen_bound needs to know about the fit: largest power-of-two row scale of L^-1, the sum of their
    squares, the largest row norm, |L^-1|_F^2 and |alpha|_2."""
    rowscale = np.ldexp(1.0, np.frexp(np.abs(Linv).max(axis=1))[1])  # 2^(ilogb(max_k |L^-1_ik|) + 1)
    rowl2 = (Linv ** 2).sum(axis=1)
    return np.array([rowscale.max(), (rowscale ** 2).sum(), np.sqrt(rowl2.max()), rowl2.sum(), np.linalg.norm(alpha)])


class ScreenOracle:
    """One fit: kernel name ("RationalQuadratic" included), training inputs X[N, d], the handle's L^-1 [N, N] and alpha [N],
    lengthscale(s), kernel variance, noise variance, the constant c0 of the mean (0 for Zero, c for Constant, b for Linear),
    A[d] for Linear (else None) and the RationalQuadratic alpha."""

    def __init__(self, kernel, X, Linv, alpha, lengthscales, variance, noise, c0=0.0, A=None, rq_alpha=None):
        self.kernel = kernel
        self.N, self.d = X.shape
        self.Np = (self.N + XK - 1) // XK * XK
        self.ls = np.atleast_1d(np.asarray(lengthscales, dtype=np.float64))
        self.variance, self.noise, self.c0 = float(variance), float(noise), float(c0)
        self.A = None if A is None else np.ravel(A)
        self.rq_alpha = rq_alpha
        self.Linv = Linv
        self.fit5 = fit5(Linv, alpha)
        self.rowscale = np.ldexp(1.0, np.frexp(np.abs(Linv).max(axis=1))[1])
        self.Xs32 = (X / self.ls).astype(np.float32)                     # screen_convert_kernel
        self.al32 = np.zeros(self.Np, dtype=np.float32)
        self.al32[: self.N] = alpha.astype(np.float32)
        self.beta = np.ldexp(1.0, int(np.frexp(self.variance)[1]))      # 2^(ilogb(variance) + 1)

    # ---- fp32 cross-covariance ------------------------------------------------------------------------------------------
    def k32(self, Xc):
        """[n, N] fp32 covariance (r2 by fp32 fma over the dimensions in order) and the mask of NaN rows."""
        x = Xc / self.ls
        bad = ~np.all(np.abs(x) <= 1.0e15, axis=1)
        xc = np.where(bad[:, None], 0.0, x).astype(np.float32)
        r2 = np.zeros((Xc.shape[0], self.N), dtype=np.float32)
        for dim in range(self.d):
            df = (self.Xs32[None, :, dim] - xc[:, dim, None]).astype(np.float32)
            r2 = (df.astype(np.float64) ** 2 + r2).astype(np.float32)   # fma.rn.f32: one rounding
        return cov32_device(self.kernel, r2, self.variance, self.rq_alpha), bad

    def mean(self, k, bad, Xc):
        n = k.shape[0]
        kp = np.zeros((n, self.Np), dtype=np.float32)
        kp[:, : self.N] = k
        kp = kp.reshape(n, self.Np // XK, 8, 16)
        al = self.al32.reshape(self.Np // XK, 8, 16)
        msum = np.zeros((n, self.Np // XK, 8), dtype=np.float32)
        for g in range(16):  # fma chain: the product is exact in fp64, one rounding to fp32
            msum = (kp[..., g].astype(np.float64) * al[None, :, :, g] + msum).astype(np.float32)
        macc = np.zeros((n, 8))
        for ss in range(self.Np // XK):
            macc += msum[:, ss, :].astype(np.float64)
        q = macc
        m = (((q[:, 0] + q[:, 1]) + (q[:, 2] + q[:, 3])) + ((q[:, 4] + q[:, 5]) + (q[:, 6] + q[:, 7]))) + self.c0
        if self.A is not None:
            m = m + lo.offset(np.where(bad[:, None], 0.0, Xc), self.A)
        return np.where(bad, np.nan, m)

    # ---- digit product and fp32 epilogue ----------------------------------------------------------------------------------
    def variance_s(self, k, S, full):
        N = self.N
        a = digits_of(np.rint(self.Linv * (2.0 ** (8 * S - 2) / self.rowscale)[:, None]), S)
        bscale = np.float32(2.0 ** (8 * S - 2) / self.beta)
        b = digits_of(np.rint((k * bscale).astype(np.float32)).astype(np.int64), S)
        levels = 2 * S - 1 if full else S
        acc = [np.zeros((N, k.shape[0])) for _ in range(levels)]      # exact integers (int32 on the device)
        for p in range(S):
            nq = S if full else S - p
            prod = a[p] @ np.concatenate([b[q].T for q in range(nq)], axis=1)
            for q in range(nq):
                acc[p + q] += prod[:, q * k.shape[0]:(q + 1) * k.shape[0]]
        w = acc[0].astype(np.float32)
        for t in range(1, levels):  # fmaf(w, 256, level): w * 256 is exact
            w = (w.astype(np.float64) * 256.0 + acc[t].astype(np.float32)).astype(np.float32)
        top = levels - 1
        gscale = self.beta * 2.0 ** (-2 * (8 * S - 2) + 8 * (S - 1) - 8 * (top - (S - 1)))
        rs = (self.rowscale * gscale).astype(np.float32)
        v = (w * rs[:, None]).astype(np.float32)
        v = (v * v).astype(np.float32)
        vp = np.zeros((self.Np, v.shape[1]), dtype=np.float32)
        vp[:N] = v
        # per 128-row block: the warp-shuffle tree over 32 rows (pairs r, r ^ 16, then ^ 8, ^ 4, ^ 2, ^ 1), then the 4 lane groups
        x = vp.reshape(self.Np // XK, 4, 32, -1)
        for h in (16, 8, 4, 2, 1):
            x = (x[:, :, :h] + x[:, :, h:2 * h]).astype(np.float32)
        g = x[:, :, 0]
        part = ((g[:, 0] + g[:, 1]).astype(np.float32) + (g[:, 2] + g[:, 3]).astype(np.float32)).astype(np.float32)
        ss = np.zeros(v.shape[1])
        for I in range(part.shape[0]):
            ss += part[I].astype(np.float64)
        return (self.variance - ss) + self.noise

    def screen(self, Xc, levels):
        """Screened (mean, variance) of the rows Xc for each level in ``levels``: (S, full) for the digit screens, 0 for the
        mean-only bound level (variance None).  Returns {level: (mean, var)}; rows with a NaN mean are NaN in both."""
        k, bad = self.k32(Xc)
        mean = self.mean(k, bad, Xc)
        out = {}
        for lev in levels:
            if lev == 0:
                out[lev] = (mean, None)
                continue
            var = self.variance_s(np.where(bad[:, None], np.float32(0), k), *lev)
            out[lev] = (mean, np.where(bad, np.nan, var))
        return out


def oracle_for(kernel, X, Linv, alpha, h):
    """ScreenOracle from a go.Hyper / rq.RQHyper (Zero or Constant mean) or lo.LinearHyper."""
    if isinstance(h, lo.LinearHyper):
        hk, c0, A = h.k, h.b, h.A
    else:
        hk, c0, A = h, (h.mean_c if h.has_mean else 0.0), None
    return ScreenOracle(kernel, X, Linv, alpha, hk.lengthscales, hk.variance, hk.noise_variance, c0, A,
                        getattr(hk, "alpha", None))


def exact_predict_y(kernel, X, y, h, Xc):
    """The fp64 posterior (mean, var) of the oracles, for any kernel and mean function."""
    if isinstance(h, lo.LinearHyper):
        m, v = lo.predict_y(kernel, X, y, h, Xc)
    elif kernel == rq.KERNEL:
        m, v = rq.predict_y(X, y, h, Xc)
    else:
        m, v = go.predict_y(kernel, X, y, h, Xc)
    return m[:, 0], v[:, 0]
