"""
``gpflow.kernels.Linear`` in the numpy oracle (test infrastructure only).  A kernel is a list of leaves combined by a sum (a bare
kernel is a one-leaf sum), each seeing ``X[:, dims[c]]``; a Linear leaf is ``K = (X * variance) @ X2.T`` (GPflow's arithmetic)
with ``K_diag = sum(X^2 * variance)``, the other leaves the existing sum / periodic / active-dims oracle components.  The
log-marginal-likelihood and its closed-form gradient in GPflow's packing (a Linear leaf packs [variance(s)] only,
dK/dvariance_j = x_j x_j^T), ``predict_y``, ``predict_f(full_cov=True)`` and a checker backend.

A leaf spec is the session's: ``(family, n_lengthscales)``, ``("Periodic", n_lengthscales, base family, n_periods)`` or
``("Linear", n_variances)``.
"""
import numpy as np
import scipy.linalg as sla

from oracle import gpr_oracle as go
from tests import active_dims_oracle as ad
from tests import periodic_oracle as pe
from tests import rq_oracle as rq
from tests import sum_oracle as so


class LinearHyper:
    def __init__(self, variance):
        self.variance = np.atleast_1d(np.asarray(variance, dtype=np.float64))

    def theta(self):
        return list(self.variance)


def leaves_of(kernel, n_lengthscales, components):
    if kernel == "Linear":
        return "Sum", [("Linear", int(n_lengthscales))]
    return ad.leaves_of(kernel, n_lengthscales, components)


def _spec_size(s):
    if s[0] == "Linear":
        return s[1]
    base = s[2] if s[0] == "Periodic" else s[0]
    return s[1] + 1 + (base == rq.KERNEL) + (s[3] if s[0] == "Periodic" else 0)


class Hyper(pe.CompositeHyper):
    """A sum whose leaves may be Linear."""

    def comp_theta(self, c):
        return c.theta() if isinstance(c, LinearHyper) else pe.comp_theta(c) if isinstance(c, pe.PeriodicHyper) else c.theta()

    def theta(self):
        t = [x for c in self.comps for x in self.comp_theta(c)] + [self.noise_variance]
        if isinstance(self.mean, tuple):
            t += list(np.ravel(self.mean[0])) + [float(self.mean[1])]
        elif self.mean is not None:
            t.append(float(self.mean))
        return np.array(t, dtype=np.float64)

    def pack(self):
        t = self.theta()
        nk = sum(len(self.comp_theta(c)) for c in self.comps)
        u = t.copy()
        u[:nk] = go.softplus_inv(t[:nk])
        u[nk] = go.softplus_inv(t[nk] - go.NOISE_FLOOR)
        return u

    @classmethod
    def from_theta(cls, kind, specs, theta, mean_id, d):
        t = list(np.asarray(theta, dtype=np.float64))
        comps = []
        for spec in specs:
            n = _spec_size(spec)
            if spec[0] == "Linear":
                comps.append(LinearHyper(t[:n]))
            else:
                comps.append(pe.CompositeHyper.from_theta(kind, [spec], t[:n] + [1.0], 0, d).comps[0])
            t = t[n:]
        noise, t = t[0], t[1:]
        mean = None if mean_id == 0 else (t[0] if mean_id == 1 else (np.array(t[:d]), t[d]))
        return cls(kind, comps, noise, mean)

    @classmethod
    def unpack(cls, kind, specs, u, mean_id, d):
        u = np.asarray(u, dtype=np.float64)
        nk = sum(_spec_size(s) for s in specs)
        t = u.copy()
        t[:nk] = go.softplus(u[:nk])
        t[nk] = go.NOISE_FLOOR + go.softplus(u[nk])
        return cls.from_theta(kind, specs, t, mean_id, d)


def _leaf_kern(c, cols, X, X2):
    if isinstance(c, LinearHyper):
        Xa = X[:, cols]
        Xb = Xa if X2 is None else X2[:, cols]
        v = c.variance if c.variance.size > 1 else c.variance[0]
        return (Xa * v) @ Xb.T
    return ad._leaf_kern(c, cols, X, X2)


def kern(h, dims, X, X2=None):
    K = None
    for c, cols in zip(h.comps, dims):
        k = _leaf_kern(c, cols, X, X2)
        K = k if K is None else K + k
    return K


def kern_diag(h, dims, X):
    """k(x, x) of every row: sum(x^2 * variance) for a Linear leaf (GPflow's K_diag), the variance of the others."""
    out = np.zeros(X.shape[0])
    for c, cols in zip(h.comps, dims):
        if isinstance(c, LinearHyper):
            v = c.variance if c.variance.size > 1 else c.variance[0]
            out = out + np.sum(np.square(X[:, cols]) * v, axis=1)
        else:
            out = out + c.variance
    return out


def _factor(h, dims, X, y):
    L = np.linalg.cholesky(kern(h, dims, X) + h.noise_variance * np.eye(X.shape[0]))
    return L, sla.solve_triangular(L, y[:, 0] - so.mean_of(h, X), lower=True)


def linear_grad(c, Xc, W):
    """dLML/dvariance: 0.5 x_j^T W x_j per column, summed for a scalar variance."""
    q = 0.5 * np.einsum("ij,ik,kj->j", Xc, W, Xc)
    return list(q) if c.variance.size > 1 else [float(np.sum(q))]


def neg_lml_and_grad(kind, specs, dims, X, y, u, mean_id):
    N, d = X.shape
    h = Hyper.unpack(kind, specs, u, mean_id, d)
    L, a = _factor(h, dims, X, y)
    alpha = sla.solve_triangular(L, a, lower=True, trans="T")
    val = -0.5 * a @ a - 0.5 * N * np.log(2.0 * np.pi) - np.sum(np.log(np.diag(L)))
    Linv = sla.solve_triangular(L, np.eye(N), lower=True)
    W = np.outer(alpha, alpha) - Linv.T @ Linv
    grad = []
    for c, cols in zip(h.comps, dims):
        if isinstance(c, LinearHyper):
            grad += linear_grad(c, X[:, cols], W)
        elif isinstance(c, pe.PeriodicHyper):
            grad += pe.comp_grad(c, X[:, cols], W)
        else:
            grad += so.comp_grad(c, X[:, cols], W)
    grad.append(0.5 * np.trace(W))
    nk = len(grad)
    chain = list(go.sigmoid(np.asarray(u[:nk], dtype=np.float64)))
    if mean_id == 2:
        grad += list(X.T @ alpha) + [np.sum(alpha)]
        chain += [1.0] * (d + 1)
    elif mean_id == 1:
        grad.append(np.sum(alpha))
        chain.append(1.0)
    return -float(val), -np.array(grad) * np.array(chain)


def lml(h, dims, X, y):
    L, a = _factor(h, dims, X, y)
    return float(-0.5 * a @ a - 0.5 * X.shape[0] * np.log(2.0 * np.pi) - np.sum(np.log(np.diag(L))))


def predict_f_full_cov(h, dims, X, y, Xnew, full_cov=True):
    Lm, _ = _factor(h, dims, X, y)
    A = sla.solve_triangular(Lm, kern(h, dims, X, Xnew), lower=True)
    f = (kern(h, dims, Xnew) - A.T @ A) if full_cov else kern_diag(h, dims, Xnew) - np.sum(np.square(A), axis=0)
    A = sla.solve_triangular(Lm, A, lower=True, trans="T")
    return A.T @ (y[:, 0] - so.mean_of(h, X)) + so.mean_of(h, Xnew), f


def predict_y(h, dims, X, y, Xnew):
    mean, fvar = predict_f_full_cov(h, dims, X, y, Xnew, full_cov=False)
    return mean[:, None], (fvar + h.noise_variance)[:, None]


# ---- checker session / backend --------------------------------------------------------------------------------------
class LinearOracleSession(ad.ActiveDimsOracleSession):
    def __init__(self, kernel, n_lengthscales, components, has_mean, rowwise=False):
        super().__init__("Sum", 1, [("SquaredExponential", 1)], has_mean, rowwise=rowwise)
        self.kernel = kernel
        self.kind, self.specs = leaves_of(kernel, n_lengthscales, components)

    def neg_lml_and_grad(self, u):
        self.calls["neg_lml_and_grad"] += 1
        return neg_lml_and_grad(self.kind, self.specs, self._dims(), self.X, self.y, u, self.mean_id)

    def factorize(self, theta):
        self.calls["factorize"] += 1
        self.h = Hyper.from_theta(self.kind, self.specs, theta, self.mean_id, self.X.shape[1])

    def log_marginal_likelihood(self):
        return lml(self.h, self._dims(), self.X, self.y)

    def _predict(self, xnew):
        return predict_y(self.h, self._dims(), self.X, self.y, xnew)

    def predict_f_cov(self, xnew):
        return predict_f_full_cov(self.h, self._dims(), self.X, self.y, np.ascontiguousarray(xnew, dtype=np.float64))


class LinearOracleBackend(ad.ActiveDimsOracleBackend):
    """Checker backend: every kernel, Linear leaves included, through this oracle."""

    def open_session(self, kernel, n_lengthscales, has_mean, components=None):
        session = LinearOracleSession(kernel, n_lengthscales, components, has_mean, rowwise=self.rowwise)
        self.sessions.append(session)
        return session
