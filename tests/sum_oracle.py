"""
Sum kernel in the numpy oracle (test infrastructure only): ``gpflow.kernels.Sum``, k = sum_c k_c over components of the five
families, built from the per-family oracles (``oracle/gpr_oracle.py``, ``tests/rq_oracle.py``).  The log-marginal-likelihood and
its closed-form gradient in GPflow's packing ([c0: (alpha), lengthscale(s), variance ; c1: ... ; noise ; mean entries]),
``predict_y``, ``predict_f(full_cov=True)``, the fp32 screening covariance of a sum, and a checker session / backend for
host-logic tests.

The gradient of a sum with respect to one component's parameters is that component's own gradient: dK/dtheta_c = dk_c/dtheta_c,
contracted with the W = alpha alpha^T - K_y^-1 of the whole sum.
"""
import numpy as np
import scipy.linalg as sla

from oracle import gpr_oracle as go
from tests import rq_oracle as rq
from tests.joint_oracle import sample_mvn
from tests.linear_mean_oracle import LinearOracleBackend
from tests.oracle_backend import OracleSession
from tests.screen_oracle import cov32_device

KERNEL_ID = 5  # GPSO_KERNEL_SUM


class Comp:
    """One component: family name, lengthscale(s) (scalar or [d]), variance, alpha (RationalQuadratic only)."""

    def __init__(self, family, lengthscales, variance, alpha=None):
        self.family = family
        self.lengthscales = np.atleast_1d(np.asarray(lengthscales, dtype=np.float64)).copy()
        self.variance = float(variance)
        self.alpha = None if family != rq.KERNEL else float(1.0 if alpha is None else alpha)

    @property
    def n_ls(self):
        return self.lengthscales.size

    def theta(self):
        return ([self.alpha] if self.alpha is not None else []) + list(self.lengthscales) + [self.variance]


class SumHyper:
    """Components, noise variance and the mean: None (zero), c (constant) or (A[d], b) (linear)."""

    def __init__(self, comps, noise_variance, mean=None):
        self.comps = list(comps)
        self.noise_variance = float(noise_variance)
        self.mean = mean

    @property
    def var_tot(self):
        v = 0.0
        for c in self.comps:
            v += c.variance
        return v

    def theta(self):
        t = [x for c in self.comps for x in c.theta()] + [self.noise_variance]
        if isinstance(self.mean, tuple):
            t += list(np.ravel(self.mean[0])) + [float(self.mean[1])]
        elif self.mean is not None:
            t.append(float(self.mean))
        return np.array(t, dtype=np.float64)

    def pack(self):
        t = self.theta()
        nk = sum(len(c.theta()) for c in self.comps)
        u = t.copy()
        u[:nk] = go.softplus_inv(t[:nk])
        u[nk] = go.softplus_inv(t[nk] - go.NOISE_FLOOR)
        return u

    @classmethod
    def from_theta(cls, families, n_ls, theta, mean_id, d):
        theta = np.asarray(theta, dtype=np.float64)
        comps, pos = [], 0
        for fam, nl in zip(families, n_ls):
            alpha = None
            if fam == rq.KERNEL:
                alpha, pos = theta[pos], pos + 1
            ls = theta[pos:pos + nl]
            comps.append(Comp(fam, ls if nl > 1 else ls[0], theta[pos + nl], alpha))
            pos += nl + 1
        noise = theta[pos]
        m = theta[pos + 1:]
        mean = (m[:d].copy(), m[d]) if mean_id == 2 else (m[0] if mean_id == 1 else None)
        return cls(comps, noise, mean)

    @classmethod
    def unpack(cls, families, n_ls, u, mean_id, d):
        u = np.asarray(u, dtype=np.float64)
        nk = sum(nl + 1 + (f == rq.KERNEL) for f, nl in zip(families, n_ls))
        t = u.copy()
        t[:nk] = go.softplus(u[:nk])
        t[nk] = go.NOISE_FLOOR + go.softplus(u[nk])
        return cls.from_theta(families, n_ls, t, mean_id, d)


# ---- covariance -------------------------------------------------------------------------------------------------------
def scaled_r2(X, X2, lengthscales):
    """Squared distance of the scaled inputs, coordinate differences first as on the device (exact zeros on the diagonal).
    GPflow's expanded |x|^2 + |x'|^2 - 2 x.x' leaves ~1e-13 there, which for a short Matern12 lengthscale moves the LML by
    more than a finite-difference step can resolve."""
    Xs = X / lengthscales
    X2s = Xs if X2 is None else X2 / lengthscales
    return np.sum(np.square(Xs[:, None, :] - X2s[None, :, :]), axis=-1)


def comp_k(c, r2):
    return rq.k_of_r2(r2, c.variance, c.alpha) if c.family == rq.KERNEL else go.k_of_r2(c.family, r2, c.variance)[0]


def comp_kern(c, X, X2):
    return comp_k(c, scaled_r2(X, X2, c.lengthscales))


def kern(h, X, X2):
    K = None
    for c in h.comps:
        k = comp_kern(c, X, X2)
        K = k if K is None else K + k
    return K


def mean_of(h, X):
    if isinstance(h.mean, tuple):
        return float(h.mean[1]) + X @ np.ravel(h.mean[0])
    return np.full(X.shape[0], 0.0 if h.mean is None else float(h.mean))


def _factor(h, X, y):
    N = X.shape[0]
    L = np.linalg.cholesky(kern(h, X, None) + h.noise_variance * np.eye(N))
    r = y[:, 0] - mean_of(h, X)
    a = sla.solve_triangular(L, r, lower=True)
    return L, a


def lml(h, X, y):
    L, a = _factor(h, X, y)
    return float(-0.5 * a @ a - 0.5 * X.shape[0] * np.log(2.0 * np.pi) - np.sum(np.log(np.diag(L))))


def comp_grad(c, X, W):
    """0.5 sum W dk_c/dtheta_c over the component's constrained parameters [(alpha), lengthscale(s), variance]."""
    ls = c.lengthscales
    r2 = scaled_r2(X, None, ls)
    if c.family == rq.KERNEL:
        K = rq.k_of_r2(r2, c.variance, c.alpha)
        with np.errstate(divide="ignore", invalid="ignore"):
            z = 0.5 * r2 / c.alpha
            g = K / (1.0 + z)
            dk_da = np.where(K != 0.0, K * (z / (1.0 + z) - np.log1p(z)), 0.0)
        out = [0.5 * np.sum(W * dk_da)]
    else:
        K, r = go.k_of_r2(c.family, r2, c.variance)
        if c.family == "SquaredExponential":
            g = K
        else:
            if c.family == "Matern52":
                g = (5.0 / 3.0) * c.variance * (1.0 + np.sqrt(5.0) * r) * np.exp(-np.sqrt(5.0) * r)
            elif c.family == "Matern32":
                g = 3.0 * c.variance * np.exp(-np.sqrt(3.0) * r)
            else:
                g = K / r
            g = np.where(r2 > go.R2_CLIP, g, 0.0)
        out = []
    WG = W * g
    if c.n_ls > 1:
        out += [0.5 * np.sum(WG * np.square(X[:, j][:, None] - X[:, j][None, :])) / ls[j] ** 3 for j in range(c.n_ls)]
    else:
        out.append(0.5 * np.sum(WG * np.maximum(r2, 0.0)) / ls[0])
    out.append(0.5 * np.sum(W * K) / c.variance)
    return out


def neg_lml_and_grad(families, n_ls, X, y, u, mean_id):
    """f(u) = -LML and df/du over the packed vector, what TF autodiff gives in closed form."""
    N, d = X.shape
    h = SumHyper.unpack(families, n_ls, u, mean_id, d)
    L, a = _factor(h, X, y)
    alpha = sla.solve_triangular(L, a, lower=True, trans="T")
    val = -0.5 * a @ a - 0.5 * N * np.log(2.0 * np.pi) - np.sum(np.log(np.diag(L)))
    Linv = sla.solve_triangular(L, np.eye(N), lower=True)
    W = np.outer(alpha, alpha) - Linv.T @ Linv
    grad = [x for c in h.comps for x in comp_grad(c, X, W)] + [0.5 * np.trace(W)]
    nk = len(grad)
    chain = list(go.sigmoid(np.asarray(u[:nk], dtype=np.float64)))
    if mean_id == 2:
        grad += list(X.T @ alpha) + [np.sum(alpha)]
        chain += [1.0] * (d + 1)
    elif mean_id == 1:
        grad.append(np.sum(alpha))
        chain.append(1.0)
    return -float(val), -np.array(grad) * np.array(chain)


def predict_f_full_cov(h, X, y, Xnew, full_cov=True):
    """gpflow base_conditional: (mean[M], cov[M,M] or var[M]) of the latent function."""
    N = X.shape[0]
    Lm = np.linalg.cholesky(kern(h, X, None) + h.noise_variance * np.eye(N))
    A = sla.solve_triangular(Lm, kern(h, X, Xnew), lower=True)
    f = (kern(h, Xnew, None) - A.T @ A) if full_cov else h.var_tot - np.sum(np.square(A), axis=0)
    A = sla.solve_triangular(Lm, A, lower=True, trans="T")
    return A.T @ (y[:, 0] - mean_of(h, X)) + mean_of(h, Xnew), f


def predict_y(h, X, y, Xnew):
    mean, fvar = predict_f_full_cov(h, X, y, Xnew, full_cov=False)
    return mean[:, None], (fvar + h.noise_variance)[:, None]


# ---- fp32 screening covariance of a sum ---------------------------------------------------------------------------------
def cov32(h, Xa, Xb):
    """kern_screen.cuh crosscov_screen_kernel<KERNEL_SUM>: per component the fp32 distance of the fp32 scaled inputs and the
    family's fp32 covariance, the component values added in order in fp32.  Returns [len(Xa), len(Xb)] float32."""
    K = None
    for c in h.comps:
        xa = (Xa / c.lengthscales).astype(np.float32)
        xb = (Xb / c.lengthscales).astype(np.float32)
        r2 = np.zeros((xa.shape[0], xb.shape[0]), dtype=np.float32)
        for j in range(xa.shape[1]):
            df = (xb[None, :, j] - xa[:, None, j]).astype(np.float32)
            r2 = (df.astype(np.float64) * df + r2).astype(np.float32)  # fma: the product is exact in fp64
        k = cov32_device(c.family, r2, c.variance, c.alpha)
        K = k if K is None else (K + k).astype(np.float32)
    return K


# ---- checker session / backend --------------------------------------------------------------------------------------
class SumOracleSession(OracleSession):
    """OracleSession for a Sum kernel: theta / u carry every component's block, then the noise and the mean entries."""

    def __init__(self, components, has_mean, rowwise=False):
        super().__init__("Sum", 0, has_mean, rowwise=rowwise)
        self.families = [fam for fam, _ in components]
        self.n_lss = [int(nl) for _, nl in components]
        self.mean_id = int(has_mean)

    def neg_lml_and_grad(self, u):
        self.calls["neg_lml_and_grad"] += 1
        return neg_lml_and_grad(self.families, self.n_lss, self.X, self.y, u, self.mean_id)

    def factorize(self, theta):
        self.calls["factorize"] += 1
        self.h = SumHyper.from_theta(self.families, self.n_lss, theta, self.mean_id, self.X.shape[1])

    def log_marginal_likelihood(self):
        return lml(self.h, self.X, self.y)

    def _predict(self, xnew):
        if not self.rowwise:
            return predict_y(self.h, self.X, self.y, xnew)
        parts = [predict_y(self.h, self.X, self.y, xnew[i:i + 1]) for i in range(xnew.shape[0])]
        return np.vstack([p[0] for p in parts]), np.vstack([p[1] for p in parts])

    def ucb_topk(self, xnew, varsigma, k):
        mean, var = self._predict(xnew)
        mean, var = mean[:, 0], var[:, 0]
        ucb = mean + varsigma * var
        nan = np.isnan(ucb)
        order = np.lexsort((np.arange(len(ucb)), -np.where(nan, np.inf, ucb), ~nan))[:k]
        return np.column_stack([order.astype(float), mean[order], var[order], ucb[order]])

    def predict_f_cov(self, xnew):
        return predict_f_full_cov(self.h, self.X, self.y, np.ascontiguousarray(xnew, dtype=np.float64))

    def predict_f_samples(self, xnew, z, jitter):
        mean, cov = self.predict_f_cov(xnew)
        return sample_mvn(mean, cov, np.asarray(z, dtype=np.float64), jitter)


class SumOracleBackend(LinearOracleBackend):
    """Checker backend: Sum sessions through this oracle, every other kernel and mean through the existing checkers."""

    def open_session(self, kernel, n_lengthscales, has_mean, components=None):
        if kernel != "Sum":
            return super().open_session(kernel, n_lengthscales, has_mean)
        session = SumOracleSession(components, has_mean, rowwise=self.rowwise)
        self.sessions.append(session)
        return session
