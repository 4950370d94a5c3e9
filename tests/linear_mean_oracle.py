"""
Linear mean function in the numpy oracle (test infrastructure only): ``gpflow.mean_functions.Linear`` (m(X) = X A + b) with
every kernel of the package, the log-marginal-likelihood and its closed-form gradient in GPflow's packing
([alpha], lengthscale(s), variance, noise variance, A (d entries), b -- tf.Module's sorted names, 'A' < 'b'), ``predict_y``,
``predict_f(full_cov=True)`` and a checker session / backend for host-logic tests.

With r = (y - b) - X A the model is the zero-mean GP on r: the kernel part of the LML and its gradient are those of the
shared oracles at mean None, and d(-LML)/dA = -X^T alpha, d(-LML)/db = -sum(alpha) with alpha = K_y^-1 r.
"""
import numpy as np
import scipy.linalg as sla

from oracle import gpr_oracle as go
from tests import joint_oracle
from tests import rq_oracle as rq
from tests.joint_oracle import sample_mvn
from tests.oracle_backend import OracleSession
from tests.rq_oracle import RQOracleBackend

MEAN_ID = 2  # GPSO_MEAN_LINEAR


class LinearHyper:
    """Kernel hyper-parameters (go.Hyper / rq.RQHyper without a mean) plus A[d] and b."""

    def __init__(self, kernel_hyper, A, b):
        self.k = kernel_hyper
        self.A = np.ravel(np.asarray(A, dtype=np.float64)).copy()
        self.b = float(np.ravel(b)[0])

    def pack(self):
        return np.concatenate([self.k.pack(), self.A, [self.b]])

    def theta(self):
        k = self.k
        t = ([k.alpha] if isinstance(k, rq.RQHyper) else []) + list(k.lengthscales) + [k.variance, k.noise_variance]
        return np.array(t + list(self.A) + [self.b])

    @classmethod
    def unpack(cls, kernel, u, n_ls, d):
        u = np.asarray(u, dtype=np.float64)
        nk = len(u) - d - 1
        base = rq.RQHyper.unpack(u[:nk], n_ls, False) if kernel == rq.KERNEL else go.Hyper.unpack(u[:nk], n_ls, False)
        return cls(base, u[nk:nk + d], u[nk + d])

    @classmethod
    def from_theta(cls, kernel, theta, n_ls, d):
        t = np.asarray(theta, dtype=np.float64)
        o = 1 if kernel == rq.KERNEL else 0
        ls = t[o:o + n_ls] if n_ls > 1 else t[o]
        var, noise = t[o + n_ls], t[o + n_ls + 1]
        base = rq.RQHyper(t[0], ls, var, noise) if o else go.Hyper(ls, var, noise)
        return cls(base, t[o + n_ls + 2:o + n_ls + 2 + d], t[o + n_ls + 2 + d])


def offset(X, A):
    return np.asarray(X, dtype=np.float64) @ np.ravel(A)


def residual(X, y, h):
    """(y - b) - X A, the device's operation order."""
    return (np.ravel(y) - h.b) - offset(X, h.A)


def kern(kernel, X, X2, hk):
    return rq.kern(X, X2, hk) if kernel == rq.KERNEL else go.kern(kernel, X, X2, hk)


def _alpha(kernel, X, hk, r):
    L = np.linalg.cholesky(kern(kernel, X, None, hk) + hk.noise_variance * np.eye(X.shape[0]))
    return sla.cho_solve((L, True), r)


def lml(kernel, X, y, h):
    r = residual(X, y, h)[:, None]
    return rq.lml(X, r, h.k) if kernel == rq.KERNEL else go.lml(kernel, X, r, h.k)


def neg_lml_and_grad(kernel, X, y, u, n_ls):
    """f(u) = -LML and df/du over [alpha], lengthscale(s), variance, noise, A, b."""
    d = X.shape[1]
    h = LinearHyper.unpack(kernel, u, n_ls, d)
    nk = len(u) - d - 1
    r = residual(X, y, h)[:, None]
    if kernel == rq.KERNEL:
        f, gk = rq.neg_lml_and_grad(X, r, u[:nk], n_ls, False)
    else:
        f, gk = go.neg_lml_and_grad(kernel, X, r, u[:nk], n_ls, False)
    alpha = _alpha(kernel, X, h.k, r[:, 0])
    return f, np.concatenate([gk, -(X.T @ alpha), [-np.sum(alpha)]])


def predict_f_full_cov(kernel, X, y, h, Xnew, full_cov=True):
    """(mean[M], cov[M,M] or var[M]) of the latent function: the zero-mean posterior of r plus m(Xnew)."""
    r = residual(X, y, h)[:, None]
    if kernel == rq.KERNEL:
        mean, f = rq.predict_f_full_cov(X, r, h.k, Xnew, full_cov=full_cov)
    elif full_cov:
        mean, f = joint_oracle.predict_f_full_cov(kernel, X, r, h.k, Xnew)
        mean = mean[:, 0]
    else:
        mean, var = go.predict_y(kernel, X, r, h.k, Xnew)
        mean, f = mean[:, 0], var[:, 0] - h.k.noise_variance
    return mean + (offset(Xnew, h.A) + h.b), f


def predict_y(kernel, X, y, h, Xnew):
    mean, fvar = predict_f_full_cov(kernel, X, y, h, Xnew, full_cov=False)
    return mean[:, None], (fvar + h.k.noise_variance)[:, None]


# ---- checker session / backend --------------------------------------------------------------------------------------
class LinearOracleSession(OracleSession):
    """OracleSession for mean id 2: theta / u carry A (d entries) and b after the noise variance."""

    def neg_lml_and_grad(self, u):
        self.calls["neg_lml_and_grad"] += 1
        return neg_lml_and_grad(self.kernel, self.X, self.y, u, self.n_ls)

    def factorize(self, theta):
        self.calls["factorize"] += 1
        self.h = LinearHyper.from_theta(self.kernel, theta, self.n_ls, self.X.shape[1])

    def log_marginal_likelihood(self):
        return lml(self.kernel, self.X, self.y, self.h)

    def _predict(self, xnew):
        if not self.rowwise:
            return predict_y(self.kernel, self.X, self.y, self.h, xnew)
        parts = [predict_y(self.kernel, self.X, self.y, self.h, xnew[i:i + 1]) for i in range(xnew.shape[0])]
        return np.vstack([p[0] for p in parts]), np.vstack([p[1] for p in parts])

    def ucb_topk(self, xnew, varsigma, k):
        mean, var = self._predict(xnew)
        mean, var = mean[:, 0], var[:, 0]
        ucb = mean + varsigma * var
        nan = np.isnan(ucb)
        order = np.lexsort((np.arange(len(ucb)), -np.where(nan, np.inf, ucb), ~nan))[:k]
        return np.column_stack([order.astype(float), mean[order], var[order], ucb[order]])

    def predict_f_cov(self, xnew):
        return predict_f_full_cov(self.kernel, self.X, self.y, self.h, np.ascontiguousarray(xnew, dtype=np.float64))

    def predict_f_samples(self, xnew, z, jitter):
        mean, cov = self.predict_f_cov(xnew)
        return sample_mvn(mean, cov, np.asarray(z, dtype=np.float64), jitter)


class LinearOracleBackend(RQOracleBackend):
    """Checker backend: linear-mean sessions (mean id 2, any kernel) through this oracle, the others as before."""

    def open_session(self, kernel, n_lengthscales, has_mean):
        if has_mean != MEAN_ID:
            return super().open_session(kernel, n_lengthscales, has_mean)
        session = LinearOracleSession(kernel, n_lengthscales, has_mean, rowwise=self.rowwise)
        self.sessions.append(session)
        return session
