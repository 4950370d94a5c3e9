"""
Kernels on a subset of the inputs (GPflow's ``active_dims``) in the numpy oracle (test infrastructure only).  Every kernel is a
list of leaves combined by a sum or a product (a bare kernel is a one-leaf sum); leaf c is one of the five stationary families or
a periodic kernel and sees ``X[:, dims[c]]`` -- the existing ``sum_oracle`` / ``periodic_oracle`` component functions on the
gathered columns.  The mean function reads all d columns.  The log-marginal-likelihood and its closed-form gradient in GPflow's
packing, ``predict_y``, ``predict_f(full_cov=True)`` and a checker backend whose sessions take ``set_active_dims``.

A leaf spec is the session's: ``(family, n_lengthscales)`` or ``("Periodic", n_lengthscales, base family, n_periods)``.
"""
import numpy as np
import scipy.linalg as sla

from oracle import gpr_oracle as go
from tests import periodic_oracle as pe
from tests import product_oracle as po
from tests import sum_oracle as so
from tests.joint_oracle import sample_mvn


def leaves_of(kernel, n_lengthscales, components):
    """(kind, leaf specs) of an ``open_session`` call: a bare kernel is a one-leaf sum."""
    if kernel in ("Sum", "Product"):
        return kernel, [tuple(c) for c in components]
    if kernel == "Periodic":
        (base, n_p), = components
        return "Sum", [("Periodic", int(n_lengthscales), base, int(n_p))]
    return "Sum", [(kernel, int(n_lengthscales))]


def _leaf_kern(c, dims, X, X2):
    Xa = X[:, dims]
    Xb = None if X2 is None else X2[:, dims]
    return pe.kern(c, Xa, Xb) if isinstance(c, pe.PeriodicHyper) else so.comp_kern(c, Xa, Xb)


def kern(h, dims, X, X2):
    K = None
    for c, cols in zip(h.comps, dims):
        k = _leaf_kern(c, cols, X, X2)
        K = k if K is None else (K * k if h.kind == "Product" else K + k)
    return K


def _factor(h, dims, X, y):
    L = np.linalg.cholesky(kern(h, dims, X, None) + h.noise_variance * np.eye(X.shape[0]))
    return L, sla.solve_triangular(L, y[:, 0] - so.mean_of(h, X), lower=True)


def neg_lml_and_grad(kind, specs, dims, X, y, u, mean_id):
    """f(u) = -LML and df/du; a product's factor c takes W * prod_{j != c} k_j, every leaf its own columns."""
    N, d = X.shape
    h = pe.CompositeHyper.unpack(kind, specs, u, mean_id, d)
    L, a = _factor(h, dims, X, y)
    alpha = sla.solve_triangular(L, a, lower=True, trans="T")
    val = -0.5 * a @ a - 0.5 * N * np.log(2.0 * np.pi) - np.sum(np.log(np.diag(L)))
    Linv = sla.solve_triangular(L, np.eye(N), lower=True)
    W = np.outer(alpha, alpha) - Linv.T @ Linv
    ks = [_leaf_kern(c, cols, X, None) for c, cols in zip(h.comps, dims)]
    grad = []
    for i, (c, cols) in enumerate(zip(h.comps, dims)):
        Wc = W * po.others(ks, i) if kind == "Product" else W
        grad += pe.comp_grad(c, X[:, cols], Wc) if isinstance(c, pe.PeriodicHyper) else so.comp_grad(c, X[:, cols], Wc)
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
    f = (kern(h, dims, Xnew, None) - A.T @ A) if full_cov else h.prior_variance - np.sum(np.square(A), axis=0)
    A = sla.solve_triangular(Lm, A, lower=True, trans="T")
    return A.T @ (y[:, 0] - so.mean_of(h, X)) + so.mean_of(h, Xnew), f


def predict_y(h, dims, X, y, Xnew):
    mean, fvar = predict_f_full_cov(h, dims, X, y, Xnew, full_cov=False)
    return mean[:, None], (fvar + h.noise_variance)[:, None]


# ---- checker session / backend --------------------------------------------------------------------------------------
class ActiveDimsOracleSession(so.SumOracleSession):
    """The sum checker's session interface for any kernel with a column map (``set_active_dims``; None: every column)."""

    def __init__(self, kernel, n_lengthscales, components, has_mean, rowwise=False):
        super().__init__([("SquaredExponential", 1)], has_mean, rowwise=rowwise)
        self.kernel = kernel
        self.kind, self.specs = leaves_of(kernel, n_lengthscales, components)
        self.leaf_dims = None
        self.calls["set_active_dims"] = 0

    def set_active_dims(self, leaf_dims):
        self.calls["set_active_dims"] += 1
        if leaf_dims is not None and len(leaf_dims) != len(self.specs):
            raise ValueError("one column list per leaf")
        self.leaf_dims = None if leaf_dims is None else [list(map(int, cols)) for cols in leaf_dims]
        self.X = self.y = self.h = None

    def _dims(self):
        return self.leaf_dims or [list(range(self.X.shape[1]))] * len(self.specs)

    def neg_lml_and_grad(self, u):
        self.calls["neg_lml_and_grad"] += 1
        return neg_lml_and_grad(self.kind, self.specs, self._dims(), self.X, self.y, u, self.mean_id)

    def factorize(self, theta):
        self.calls["factorize"] += 1
        self.h = pe.CompositeHyper.from_theta(self.kind, self.specs, theta, self.mean_id, self.X.shape[1])

    def log_marginal_likelihood(self):
        return lml(self.h, self._dims(), self.X, self.y)

    def _predict(self, xnew):
        rows = [xnew[i:i + 1] for i in range(xnew.shape[0])] if self.rowwise else [xnew]
        parts = [predict_y(self.h, self._dims(), self.X, self.y, r) for r in rows]
        return np.vstack([p[0] for p in parts]), np.vstack([p[1] for p in parts])

    def predict_f_cov(self, xnew):
        return predict_f_full_cov(self.h, self._dims(), self.X, self.y, np.ascontiguousarray(xnew, dtype=np.float64))

    def predict_f_samples(self, xnew, z, jitter):
        mean, cov = self.predict_f_cov(xnew)
        return sample_mvn(mean, cov, np.asarray(z, dtype=np.float64), jitter)


class ActiveDimsOracleBackend(pe.PeriodicOracleBackend):
    """Checker backend: every kernel through this oracle, with or without a column map."""

    def open_session(self, kernel, n_lengthscales, has_mean, components=None):
        session = ActiveDimsOracleSession(kernel, n_lengthscales, components, has_mean, rowwise=self.rowwise)
        self.sessions.append(session)
        return session
