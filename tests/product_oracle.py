"""
Product kernel in the numpy oracle (test infrastructure only): ``gpflow.kernels.Product``, k = prod_c k_c over factors of the
five families, built on the sum oracle's components (``tests/sum_oracle.py``).  The log-marginal-likelihood and its closed-form
gradient in GPflow's packing ([f0: (alpha), lengthscale(s), variance ; f1: ... ; noise ; mean entries]), ``predict_y``,
``predict_f(full_cov=True)``, the fp32 screening covariance of a product, and a checker session / backend for host-logic tests.

The gradient with respect to one factor's parameters is dK/dtheta_c = P_-c dk_c/dtheta_c with P_-c = prod_{j != c} k_j: the
factor's own gradient contracted with W * P_-c instead of W (W = alpha alpha^T - K_y^-1 of the whole product).
"""
import numpy as np
import scipy.linalg as sla

from oracle import gpr_oracle as go
from tests import sum_oracle as so
from tests.joint_oracle import sample_mvn
from tests.screen_oracle import cov32_device

KERNEL_ID = 6  # GPSO_KERNEL_PRODUCT
Comp = so.Comp


class ProductHyper(so.SumHyper):
    """Factors, noise variance and the mean (the sum oracle's packing)."""

    @property
    def var_prod(self):
        v = None
        for c in self.comps:
            v = c.variance if v is None else v * c.variance
        return v

    @classmethod
    def from_theta(cls, families, n_ls, theta, mean_id, d):
        h = so.SumHyper.from_theta(families, n_ls, theta, mean_id, d)
        return cls(h.comps, h.noise_variance, h.mean)

    @classmethod
    def unpack(cls, families, n_ls, u, mean_id, d):
        h = so.SumHyper.unpack(families, n_ls, u, mean_id, d)
        return cls(h.comps, h.noise_variance, h.mean)


# ---- covariance -------------------------------------------------------------------------------------------------------
def factors(h, X, X2):
    return [so.comp_kern(c, X, X2) for c in h.comps]


def kern(h, X, X2):
    K = None
    for k in factors(h, X, X2):
        K = k if K is None else K * k
    return K


def _cholesky(h, X):
    return np.linalg.cholesky(kern(h, X, None) + h.noise_variance * np.eye(X.shape[0]))


def lml(h, X, y):
    L = _cholesky(h, X)
    a = sla.solve_triangular(L, y[:, 0] - so.mean_of(h, X), lower=True)
    return float(-0.5 * a @ a - 0.5 * X.shape[0] * np.log(2.0 * np.pi) - np.sum(np.log(np.diag(L))))


def others(ks, c):
    """P_-c = prod_{j != c} k_j, without dividing by k_c (which can be 0)."""
    P = np.ones_like(ks[0])
    for j, k in enumerate(ks):
        if j != c:
            P = P * k
    return P


def neg_lml_and_grad(families, n_ls, X, y, u, mean_id):
    """f(u) = -LML and df/du over the packed vector, what TF autodiff gives in closed form."""
    N, d = X.shape
    h = ProductHyper.unpack(families, n_ls, u, mean_id, d)
    L = _cholesky(h, X)
    a = sla.solve_triangular(L, y[:, 0] - so.mean_of(h, X), lower=True)
    alpha = sla.solve_triangular(L, a, lower=True, trans="T")
    val = -0.5 * a @ a - 0.5 * N * np.log(2.0 * np.pi) - np.sum(np.log(np.diag(L)))
    Linv = sla.solve_triangular(L, np.eye(N), lower=True)
    W = np.outer(alpha, alpha) - Linv.T @ Linv
    ks = factors(h, X, None)
    grad = [x for i, c in enumerate(h.comps) for x in so.comp_grad(c, X, W * others(ks, i))] + [0.5 * np.trace(W)]
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
    Lm = _cholesky(h, X)
    A = sla.solve_triangular(Lm, kern(h, X, Xnew), lower=True)
    f = (kern(h, Xnew, None) - A.T @ A) if full_cov else h.var_prod - np.sum(np.square(A), axis=0)
    A = sla.solve_triangular(Lm, A, lower=True, trans="T")
    return A.T @ (y[:, 0] - so.mean_of(h, X)) + so.mean_of(h, Xnew), f


def predict_y(h, X, y, Xnew):
    mean, fvar = predict_f_full_cov(h, X, y, Xnew, full_cov=False)
    return mean[:, None], (fvar + h.noise_variance)[:, None]


# ---- fp32 screening covariance of a product -----------------------------------------------------------------------------
def cov32(h, Xa, Xb):
    """kern_screen.cuh crosscov_screen_kernel<KERNEL_PRODUCT>: per factor the fp32 distance of the fp32 scaled inputs and the
    family's fp32 covariance, the first factor with variance (float)var_prod and the others with variance 1, multiplied in
    order in fp32.  Returns [len(Xa), len(Xb)] float32."""
    K = None
    for i, c in enumerate(h.comps):
        xa = (Xa / c.lengthscales).astype(np.float32)
        xb = (Xb / c.lengthscales).astype(np.float32)
        r2 = np.zeros((xa.shape[0], xb.shape[0]), dtype=np.float32)
        for j in range(xa.shape[1]):
            df = (xb[None, :, j] - xa[:, None, j]).astype(np.float32)
            r2 = (df.astype(np.float64) * df + r2).astype(np.float32)  # fma: the product is exact in fp64
        k = cov32_device(c.family, r2, h.var_prod if i == 0 else 1.0, c.alpha)
        K = k if K is None else (K * k).astype(np.float32)
    return K


# ---- checker session / backend --------------------------------------------------------------------------------------
class ProductOracleSession(so.SumOracleSession):
    """SumOracleSession with the product's LML, gradient and posterior."""

    def __init__(self, components, has_mean, rowwise=False):
        super().__init__(components, has_mean, rowwise=rowwise)
        self.kernel = "Product"

    def neg_lml_and_grad(self, u):
        self.calls["neg_lml_and_grad"] += 1
        return neg_lml_and_grad(self.families, self.n_lss, self.X, self.y, u, self.mean_id)

    def factorize(self, theta):
        self.calls["factorize"] += 1
        self.h = ProductHyper.from_theta(self.families, self.n_lss, theta, self.mean_id, self.X.shape[1])

    def log_marginal_likelihood(self):
        return lml(self.h, self.X, self.y)

    def _predict(self, xnew):
        if not self.rowwise:
            return predict_y(self.h, self.X, self.y, xnew)
        parts = [predict_y(self.h, self.X, self.y, xnew[i:i + 1]) for i in range(xnew.shape[0])]
        return np.vstack([p[0] for p in parts]), np.vstack([p[1] for p in parts])

    def predict_f_cov(self, xnew):
        return predict_f_full_cov(self.h, self.X, self.y, np.ascontiguousarray(xnew, dtype=np.float64))

    def predict_f_samples(self, xnew, z, jitter):
        mean, cov = self.predict_f_cov(xnew)
        return sample_mvn(mean, cov, np.asarray(z, dtype=np.float64), jitter)


class ProductOracleBackend(so.SumOracleBackend):
    """Checker backend: Product sessions through this oracle, every other kernel and mean through the existing checkers."""

    def open_session(self, kernel, n_lengthscales, has_mean, components=None):
        if kernel != "Product":
            return super().open_session(kernel, n_lengthscales, has_mean, components)
        session = ProductOracleSession(components, has_mean, rowwise=self.rowwise)
        self.sessions.append(session)
        return session
