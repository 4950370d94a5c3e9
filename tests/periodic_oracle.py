"""
Periodic kernel in the numpy oracle (test infrastructure only): ``gpflow.kernels.Periodic(base_kernel, period)`` with a
SquaredExponential or RationalQuadratic base, in GPflow 2's op order (``Periodic.K``, the ``K_r2`` branch: difference first,
then ``sin``):

    r = pi * (x_j - x'_j) / p_j,   s_j = sin(r) / l_j,   r2 = sum_j s_j^2,   k = base.K_r2(r2)

The log-marginal-likelihood and its closed-form gradient in GPflow's packing ([(alpha), lengthscale(s), variance, period(s),
noise, mean entries]), ``predict_y``, ``predict_f(full_cov=True)``, the device's embedding of the inputs, the fp32 screening
covariance on the embedded rows in the device's order of operations, and a checker session / backend for host-logic tests.

Gradient: with g = -2 dk/dr2 and r2_j = sin^2(pi delta_j / p_j) / l_j^2,
    dK/dl_j = g r2_j / l_j,     dK/dp_j = g pi delta_j sin(2 pi delta_j / p_j) / (2 l_j^2 p_j^2).
"""
import numpy as np
import scipy.linalg as sla

from oracle import gpr_oracle as go
from tests import product_oracle as po
from tests import rq_oracle as rq
from tests import sum_oracle as so
from tests.joint_oracle import sample_mvn
from tests.screen_oracle import cov32_device

BASES = ("SquaredExponential", "RationalQuadratic")


class PeriodicHyper:
    """Base family, (alpha), lengthscale(s), variance, period(s), noise variance and the mean (None, c or (A[d], b))."""

    def __init__(self, base, lengthscales, variance, period, noise_variance, alpha=None, mean=None):
        self.base = base
        self.lengthscales = np.atleast_1d(np.asarray(lengthscales, dtype=np.float64))
        self.variance = float(variance)
        self.period = np.atleast_1d(np.asarray(period, dtype=np.float64))
        self.noise_variance = float(noise_variance)
        self.alpha = None if alpha is None else float(alpha)
        self.mean = mean

    def theta(self):
        t = ([self.alpha] if self.base == rq.KERNEL else []) + list(self.lengthscales) + [self.variance] + list(self.period)
        t.append(self.noise_variance)
        if isinstance(self.mean, tuple):
            t += list(np.ravel(self.mean[0])) + [float(self.mean[1])]
        elif self.mean is not None:
            t.append(float(self.mean))
        return np.array(t, dtype=np.float64)

    def pack(self):
        """The unconstrained vector: softplus^-1 of the positive entries, the noise over its 1e-6 floor, the mean as is."""
        t = self.theta()
        nk = (self.base == rq.KERNEL) + self.lengthscales.size + 1 + self.period.size
        u = t.copy()
        u[:nk] = go.softplus_inv(t[:nk])
        u[nk] = go.softplus_inv(t[nk] - go.NOISE_FLOOR)
        return u

    @classmethod
    def from_theta(cls, base, n_ls, n_p, theta, mean_id, d):
        t = list(np.asarray(theta, dtype=np.float64))
        alpha = t.pop(0) if base == rq.KERNEL else None
        ls, t = t[:n_ls], t[n_ls:]
        var, t = t[0], t[1:]
        p, t = t[:n_p], t[n_p:]
        noise, t = t[0], t[1:]
        mean = None if mean_id == 0 else (t[0] if mean_id == 1 else (np.array(t[:d]), t[d]))
        return cls(base, ls, var, p, noise, alpha, mean)

    @classmethod
    def unpack(cls, base, n_ls, n_p, u, mean_id, d):
        u = np.asarray(u, dtype=np.float64)
        nk = (base == rq.KERNEL) + n_ls + 1 + n_p
        t = u.copy()
        t[:nk] = go.softplus(u[:nk])
        t[nk] = go.NOISE_FLOOR + go.softplus(u[nk])
        return cls.from_theta(base, n_ls, n_p, t, mean_id, d)


# ---- covariance -------------------------------------------------------------------------------------------------------
def _deltas(X, X2):
    return X[:, None, :] - (X if X2 is None else X2)[None, :, :]


def r2_parts(h, X, X2):
    """[n, m, d] per-dimension sin^2(pi delta / p) / l^2, difference first as in GPflow."""
    s = np.sin(np.pi * _deltas(X, X2) / h.period) / h.lengthscales
    return s * s


def k_of_r2(h, r2):
    if h.base == rq.KERNEL:
        return rq.k_of_r2(r2, h.variance, h.alpha)
    return h.variance * np.exp(-0.5 * r2)


def kern(h, X, X2):
    return k_of_r2(h, r2_parts(h, X, X2).sum(-1))


def _factor(h, X, y):
    L = np.linalg.cholesky(kern(h, X, None) + h.noise_variance * np.eye(X.shape[0]))
    a = sla.solve_triangular(L, y[:, 0] - so.mean_of(h, X), lower=True)
    return L, a


def lml(h, X, y):
    L, a = _factor(h, X, y)
    return float(-0.5 * a @ a - 0.5 * X.shape[0] * np.log(2.0 * np.pi) - np.sum(np.log(np.diag(L))))


def comp_grad(h, X, W):
    """0.5 sum W dk/dtheta over the periodic kernel's constrained parameters [(alpha), lengthscale(s), variance, period(s)]."""
    n_ls, n_p = h.lengthscales.size, h.period.size
    parts = r2_parts(h, X, None)
    r2 = parts.sum(-1)
    K = k_of_r2(h, r2)
    if h.base == rq.KERNEL:
        z = 0.5 * r2 / h.alpha
        g = K / (1.0 + z)
        dalpha = K * (z / (1.0 + z) - np.log1p(z))
    else:
        g = K
    delta = _deltas(X, None)
    dl = np.einsum("ij,ijk->k", W * g, parts) / h.lengthscales if n_ls > 1 else [np.sum(W * g * r2) / h.lengthscales[0]]
    dp_dims = np.einsum("ij,ijk->k", W * g, np.pi * delta * np.sin(2.0 * np.pi * delta / h.period)) / (2.0 * h.lengthscales ** 2 * h.period ** 2)
    dp = dp_dims if n_p > 1 else [np.sum(dp_dims)]
    grad = ([0.5 * np.sum(W * dalpha)] if h.base == rq.KERNEL else []) + [0.5 * x for x in dl] + [0.5 * np.sum(W * K) / h.variance]
    return grad + [0.5 * x for x in dp]


def comp_theta(h):
    """A periodic component's block of the packed vector: [(alpha), lengthscale(s), variance, period(s)]."""
    return ([h.alpha] if h.base == rq.KERNEL else []) + list(h.lengthscales) + [h.variance] + list(h.period)


def neg_lml_and_grad(base, n_ls, n_p, X, y, u, mean_id):
    """f(u) = -LML and df/du over the packed vector, what TF autodiff gives in closed form."""
    N, d = X.shape
    h = PeriodicHyper.unpack(base, n_ls, n_p, u, mean_id, d)
    L, a = _factor(h, X, y)
    alpha = sla.solve_triangular(L, a, lower=True, trans="T")
    val = -0.5 * a @ a - 0.5 * N * np.log(2.0 * np.pi) - np.sum(np.log(np.diag(L)))
    Linv = sla.solve_triangular(L, np.eye(N), lower=True)
    W = np.outer(alpha, alpha) - Linv.T @ Linv
    grad = comp_grad(h, X, W) + [0.5 * np.trace(W)]
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
    Lm, _ = _factor(h, X, y)
    A = sla.solve_triangular(Lm, kern(h, X, Xnew), lower=True)
    f = (kern(h, Xnew, None) - A.T @ A) if full_cov else h.variance - np.sum(np.square(A), axis=0)
    A = sla.solve_triangular(Lm, A, lower=True, trans="T")
    return A.T @ (y[:, 0] - so.mean_of(h, X)) + so.mean_of(h, Xnew), f


def predict_y(h, X, y, Xnew):
    mean, fvar = predict_f_full_cov(h, X, y, Xnew, full_cov=False)
    return mean[:, None], (fvar + h.noise_variance)[:, None]


# ---- sums and products with periodic components --------------------------------------------------------------------------
# A component spec is (family, n_ls) for the five families or ("Periodic", n_ls, base, n_p); a component is a sum_oracle.Comp or a
# PeriodicHyper (its noise and mean unused).
class CompositeHyper:
    """kind "Sum" or "Product", components in order, noise variance and the mean (None, c or (A[d], b))."""

    def __init__(self, kind, comps, noise_variance, mean=None):
        self.kind, self.comps, self.noise_variance, self.mean = kind, list(comps), float(noise_variance), mean

    @property
    def prior_variance(self):
        v = None
        for c in self.comps:
            v = c.variance if v is None else (v * c.variance if self.kind == "Product" else v + c.variance)
        return v

    def theta(self):
        t = [x for c in self.comps for x in (comp_theta(c) if isinstance(c, PeriodicHyper) else c.theta())] + [self.noise_variance]
        if isinstance(self.mean, tuple):
            t += list(np.ravel(self.mean[0])) + [float(self.mean[1])]
        elif self.mean is not None:
            t.append(float(self.mean))
        return np.array(t, dtype=np.float64)

    def pack(self):
        t = self.theta()
        nk = sum(len(comp_theta(c) if isinstance(c, PeriodicHyper) else c.theta()) for c in self.comps)
        u = t.copy()
        u[:nk] = go.softplus_inv(t[:nk])
        u[nk] = go.softplus_inv(t[nk] - go.NOISE_FLOOR)
        return u

    @classmethod
    def from_theta(cls, kind, specs, theta, mean_id, d):
        t = list(np.asarray(theta, dtype=np.float64))
        comps = []
        for spec in specs:
            base = spec[2] if spec[0] == "Periodic" else spec[0]
            alpha = t.pop(0) if base == rq.KERNEL else None
            ls, t = t[:spec[1]], t[spec[1]:]
            var, t = t[0], t[1:]
            if spec[0] == "Periodic":
                p, t = t[:spec[3]], t[spec[3]:]
                comps.append(PeriodicHyper(base, ls, var, p, 1.0, alpha=alpha))
            else:
                comps.append(so.Comp(base, ls if len(ls) > 1 else ls[0], var, alpha))
        noise, t = t[0], t[1:]
        mean = None if mean_id == 0 else (t[0] if mean_id == 1 else (np.array(t[:d]), t[d]))
        return cls(kind, comps, noise, mean)

    @classmethod
    def unpack(cls, kind, specs, u, mean_id, d):
        u = np.asarray(u, dtype=np.float64)
        nk = sum(s[1] + 1 + ((s[2] if s[0] == "Periodic" else s[0]) == rq.KERNEL) + (s[3] if s[0] == "Periodic" else 0) for s in specs)
        t = u.copy()
        t[:nk] = go.softplus(u[:nk])
        t[nk] = go.NOISE_FLOOR + go.softplus(u[nk])
        return cls.from_theta(kind, specs, t, mean_id, d)


def _comp_kern(c, X, X2):
    return kern(c, X, X2) if isinstance(c, PeriodicHyper) else so.comp_kern(c, X, X2)


def composite_kern(h, X, X2):
    K = None
    for c in h.comps:
        k = _comp_kern(c, X, X2)
        K = k if K is None else (K * k if h.kind == "Product" else K + k)
    return K


def _composite_factor(h, X, y):
    L = np.linalg.cholesky(composite_kern(h, X, None) + h.noise_variance * np.eye(X.shape[0]))
    return L, sla.solve_triangular(L, y[:, 0] - so.mean_of(h, X), lower=True)


def composite_neg_lml_and_grad(kind, specs, X, y, u, mean_id):
    """f(u) = -LML and df/du of a sum (product) with periodic components; a product's factor c takes W * prod_{j != c} k_j."""
    N, d = X.shape
    h = CompositeHyper.unpack(kind, specs, u, mean_id, d)
    L, a = _composite_factor(h, X, y)
    alpha = sla.solve_triangular(L, a, lower=True, trans="T")
    val = -0.5 * a @ a - 0.5 * N * np.log(2.0 * np.pi) - np.sum(np.log(np.diag(L)))
    Linv = sla.solve_triangular(L, np.eye(N), lower=True)
    W = np.outer(alpha, alpha) - Linv.T @ Linv
    ks = [_comp_kern(c, X, None) for c in h.comps]
    grad = []
    for i, c in enumerate(h.comps):
        Wc = W * po.others(ks, i) if kind == "Product" else W
        grad += comp_grad(c, X, Wc) if isinstance(c, PeriodicHyper) else so.comp_grad(c, X, Wc)
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


def composite_lml(h, X, y):
    L, a = _composite_factor(h, X, y)
    return float(-0.5 * a @ a - 0.5 * X.shape[0] * np.log(2.0 * np.pi) - np.sum(np.log(np.diag(L))))


def composite_predict_f_full_cov(h, X, y, Xnew, full_cov=True):
    Lm, _ = _composite_factor(h, X, y)
    A = sla.solve_triangular(Lm, composite_kern(h, X, Xnew), lower=True)
    f = (composite_kern(h, Xnew, None) - A.T @ A) if full_cov else h.prior_variance - np.sum(np.square(A), axis=0)
    A = sla.solve_triangular(Lm, A, lower=True, trans="T")
    return A.T @ (y[:, 0] - so.mean_of(h, X)) + so.mean_of(h, Xnew), f


def composite_predict_y(h, X, y, Xnew):
    mean, fvar = composite_predict_f_full_cov(h, X, y, Xnew, full_cov=False)
    return mean[:, None], (fvar + h.noise_variance)[:, None]


# ---- the device's embedding and its fp32 screening covariance -----------------------------------------------------------
def embed(X, lengthscales, period):
    """kern_cov.cuh periodic_embed_kernel: [n, 2d] rows (cos, sin)(2 pi x / p) / (2 l); numpy's cos(pi t) stands in for sincospi(t)."""
    d = X.shape[1]
    ls = np.broadcast_to(np.atleast_1d(lengthscales), (d,))
    p = np.broadcast_to(np.atleast_1d(period), (d,))
    t = np.pi * (2.0 * X / p)
    return np.concatenate([np.cos(t) / (2.0 * ls), np.sin(t) / (2.0 * ls)], axis=1)


def embedded_r2(h, X, X2):
    ea, eb = embed(X, h.lengthscales, h.period), embed(X if X2 is None else X2, h.lengthscales, h.period)
    return np.sum(np.square(ea[:, None, :] - eb[None, :, :]), axis=-1)


def cov32(h, Xa, Xb):
    """kern_screen.cuh crosscov_screen_kernel<base> on the embedded rows at unit lengthscale: fp32 copies of the fp64 embedded rows
    (the training rows through screen_convert_kernel, the candidates' rows staged as (float)(e / 1.0)), the fp32 distance as an fma
    chain over the 2d rows, and the base family's fp32 covariance.  Returns [len(Xa), len(Xb)] float32."""
    xa = embed(Xa, h.lengthscales, h.period).astype(np.float32)
    xb = embed(Xb, h.lengthscales, h.period).astype(np.float32)
    r2 = np.zeros((xa.shape[0], xb.shape[0]), dtype=np.float32)
    for j in range(xa.shape[1]):
        df = (xb[None, :, j] - xa[:, None, j]).astype(np.float32)
        r2 = (df.astype(np.float64) * df + r2).astype(np.float32)  # fma: the product is exact in fp64
    return cov32_device(h.base, r2, h.variance, h.alpha)


# ---- checker session / backend --------------------------------------------------------------------------------------
class PeriodicOracleSession(so.SumOracleSession):
    """The sum checker's session interface with the periodic kernel's LML, gradient and posterior."""

    def __init__(self, n_lengthscales, components, has_mean, rowwise=False):
        super().__init__([("SquaredExponential", 1)], has_mean, rowwise=rowwise)
        self.kernel = "Periodic"
        (self.base, n_p), = components
        self.n_ls, self.n_p = int(n_lengthscales), int(n_p)

    def neg_lml_and_grad(self, u):
        self.calls["neg_lml_and_grad"] += 1
        return neg_lml_and_grad(self.base, self.n_ls, self.n_p, self.X, self.y, u, self.mean_id)

    def factorize(self, theta):
        self.calls["factorize"] += 1
        self.h = PeriodicHyper.from_theta(self.base, self.n_ls, self.n_p, theta, self.mean_id, self.X.shape[1])

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


class CompositeOracleSession(so.SumOracleSession):
    """The sum checker's session interface for a sum or product with periodic components."""

    def __init__(self, kind, components, has_mean, rowwise=False):
        super().__init__([("SquaredExponential", 1)], has_mean, rowwise=rowwise)
        self.kernel, self.specs = kind, [tuple(c) for c in components]

    def neg_lml_and_grad(self, u):
        self.calls["neg_lml_and_grad"] += 1
        return composite_neg_lml_and_grad(self.kernel, self.specs, self.X, self.y, u, self.mean_id)

    def factorize(self, theta):
        self.calls["factorize"] += 1
        self.h = CompositeHyper.from_theta(self.kernel, self.specs, theta, self.mean_id, self.X.shape[1])

    def log_marginal_likelihood(self):
        return composite_lml(self.h, self.X, self.y)

    def _predict(self, xnew):
        rows = [xnew[i:i + 1] for i in range(xnew.shape[0])] if self.rowwise else [xnew]
        parts = [composite_predict_y(self.h, self.X, self.y, r) for r in rows]
        return np.vstack([p[0] for p in parts]), np.vstack([p[1] for p in parts])

    def predict_f_cov(self, xnew):
        return composite_predict_f_full_cov(self.h, self.X, self.y, np.ascontiguousarray(xnew, dtype=np.float64))

    def predict_f_samples(self, xnew, z, jitter):
        mean, cov = self.predict_f_cov(xnew)
        return sample_mvn(mean, cov, np.asarray(z, dtype=np.float64), jitter)


class PeriodicOracleBackend(po.ProductOracleBackend):
    """Checker backend: Periodic sessions and sums / products with periodic components through this oracle, every other kernel and
    mean through the existing checkers."""

    def open_session(self, kernel, n_lengthscales, has_mean, components=None):
        if kernel in ("Sum", "Product") and any(c[0] == "Periodic" for c in components):
            session = CompositeOracleSession(kernel, components, has_mean, rowwise=self.rowwise)
            self.sessions.append(session)
            return session
        if kernel != "Periodic":
            return super().open_session(kernel, n_lengthscales, has_mean, components)
        session = PeriodicOracleSession(n_lengthscales, components, has_mean, rowwise=self.rowwise)
        self.sessions.append(session)
        return session
