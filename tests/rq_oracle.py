"""
RationalQuadratic kernel in the numpy oracle (test infrastructure only): ``gpflow.kernels.RationalQuadratic`` restated in
GPflow 2's op order, the log-marginal-likelihood and its closed-form gradient in GPflow's packing (kernel.alpha first:
tf.Module lists attributes in sorted name order), ``predict_y`` and ``predict_f(full_cov=True)``, numpy emulations of the
device's FP64 log1p and of its float32 screening covariance, and a checker session / backend for host-logic tests.

    k = variance * (1 + 0.5 * r2 / alpha) ** (-alpha)        (RationalQuadratic.K_r2; r2 >= 0, no 1e-36 clip)
"""
import numpy as np
import scipy.linalg as sla

from oracle import gpr_oracle as go
from oracle import grow_oracle
from tests.joint_oracle import sample_mvn
from tests.oracle_backend import OracleBackend, OracleSession

KERNEL = "RationalQuadratic"


class RQHyper(go.Hyper):
    """go.Hyper plus alpha; packed vector [alpha, lengthscale(s), variance, noise variance, (mean c)]."""

    def __init__(self, alpha, lengthscales, variance, noise_variance, mean_c=None):
        super().__init__(lengthscales, variance, noise_variance, mean_c)
        self.alpha = float(alpha)

    def pack(self):
        return np.concatenate([[float(go.softplus_inv(self.alpha))], super().pack()])

    @classmethod
    def unpack(cls, u, n_ls, has_mean):
        u = np.asarray(u, dtype=np.float64)
        h = go.Hyper.unpack(u[1:], n_ls, has_mean)
        return cls(float(go.softplus(u[0])), h.lengthscales if n_ls > 1 else h.lengthscales[0], h.variance,
                   h.noise_variance, h.mean_c)

    def theta(self):
        t = [self.alpha] + list(self.lengthscales) + [self.variance, self.noise_variance]
        return np.array(t + ([self.mean_c] if self.has_mean else []))


def k_of_r2(r2, variance, alpha):
    with np.errstate(divide="ignore", invalid="ignore"):
        return variance * np.power(1.0 + 0.5 * r2 / alpha, -alpha)  # alpha = 0: pow(x, -0) = 1, as in TensorFlow


def scaled_r2(X, X2, lengthscales):
    """GPflow's expanded |x|^2 + |x'|^2 - 2 x.x' on scaled inputs, clipped at 0.  The expansion leaves ~-1e-17 on the diagonal;
    for a subnormal alpha (softplus(u) below u = -710) that makes 1 + r2 / (2 alpha) = -inf and k = NaN there.  The device takes
    coordinate differences first (r2 = 0 exactly); the clip states the same covariance, and changes nothing above ~1e-17."""
    Xs = X / lengthscales
    X2s = None if X2 is None else X2 / lengthscales
    return np.maximum(go.square_distance(Xs, X2s), 0.0)


def kern(X, X2, h):
    return k_of_r2(scaled_r2(X, X2, h.lengthscales), h.variance, h.alpha)


def lml(X, y, h):
    N = X.shape[0]
    L = np.linalg.cholesky(kern(X, None, h) + h.noise_variance * np.eye(N))
    a = sla.solve_triangular(L, y[:, 0] - (h.mean_c if h.has_mean else 0.0), lower=True)
    return float(-0.5 * a @ a - 0.5 * N * np.log(2.0 * np.pi) - np.sum(np.log(np.diag(L))))


def neg_lml_and_grad(X, y, u, n_ls, has_mean):
    """f(u) = -LML and df/du over [alpha, lengthscale(s), variance, noise, (c)], what TF autodiff gives in closed form."""
    h = RQHyper.unpack(u, n_ls, has_mean)
    N = X.shape[0]
    ls = h.lengthscales
    r2 = scaled_r2(X, None, ls)
    K = k_of_r2(r2, h.variance, h.alpha)
    L = np.linalg.cholesky(K + h.noise_variance * np.eye(N))
    a = sla.solve_triangular(L, y[:, 0] - (h.mean_c if has_mean else 0.0), lower=True)
    alpha_v = sla.solve_triangular(L, a, lower=True, trans="T")
    val = -0.5 * a @ a - 0.5 * N * np.log(2.0 * np.pi) - np.sum(np.log(np.diag(L)))
    Linv = sla.solve_triangular(L, np.eye(N), lower=True)
    W = np.outer(alpha_v, alpha_v) - Linv.T @ Linv
    live = h.alpha > 0.0
    with np.errstate(divide="ignore", invalid="ignore"):
        z = 0.5 * r2 / h.alpha
        g = K / (1.0 + z) if live else np.zeros_like(K)                    # dK/dls = g * r2 / ls
        # where k = 0 (z overflowed: alpha near the softplus underflow) dk/dalpha is its limit 0, not 0 * (inf / inf - inf)
        dk_da = np.where(K != 0.0, K * (z / (1.0 + z) - np.log1p(z)), 0.0) if live else np.zeros_like(K)
    WG = W * g
    if n_ls > 1:
        d_ls = np.array([0.5 * np.sum(WG * np.square(X[:, j][:, None] - X[:, j][None, :])) / ls[j] ** 3 for j in range(n_ls)])
    else:
        d_ls = np.array([0.5 * np.sum(WG * np.maximum(r2, 0.0)) / ls[0]])
    d_var = 0.5 * np.sum(W * K) / h.variance if h.variance > 0.0 else 0.0
    d_alpha = 0.5 * np.sum(W * dk_da) if live else 0.0  # chain factor sigmoid(u) is 0 where softplus underflowed
    grad_theta = [d_alpha] + list(d_ls) + [d_var, 0.5 * np.trace(W)]
    chain = list(go.sigmoid(u[: n_ls + 3]))
    if has_mean:
        grad_theta.append(np.sum(alpha_v))
        chain.append(1.0)
    return -float(val), -np.array(grad_theta) * np.array(chain)


def predict_f_full_cov(X, y, h, Xnew, full_cov=True):
    """gpflow base_conditional: (mean[M], cov[M,M] or var[M]) of the latent function."""
    N = X.shape[0]
    c = h.mean_c if h.has_mean else 0.0
    Lm = np.linalg.cholesky(kern(X, None, h) + h.noise_variance * np.eye(N))
    A = sla.solve_triangular(Lm, kern(X, Xnew, h), lower=True)
    f = (kern(Xnew, None, h) - A.T @ A) if full_cov else h.variance - np.sum(np.square(A), axis=0)
    A = sla.solve_triangular(Lm, A, lower=True, trans="T")
    return A.T @ (y[:, 0] - c) + c, f


def predict_y(X, y, h, Xnew):
    mean, fvar = predict_f_full_cov(X, y, h, Xnew, full_cov=False)
    return mean[:, None], (fvar + h.noise_variance)[:, None]


# ---- emulations of the device arithmetic ------------------------------------------------------------------------------
def rq_z(r2, alpha):
    """common.cuh rq_scale / rq_z: z = (r2 * ia) * sc, ia = 0.5 / (alpha / sc), sc = 2^600 below alpha = 2^-1000."""
    tiny = alpha < 2.0 ** -1000
    sc = 2.0 ** 600 if tiny else 1.0
    with np.errstate(divide="ignore", over="ignore", invalid="ignore"):
        ia = 0.5 / (alpha * sc if tiny else alpha)
        return (np.asarray(r2, dtype=np.float64) * ia) * sc


LG = [6.666666666666735130e-01, 3.999999999940941908e-01, 2.857142874366239149e-01, 2.222219843214978396e-01,
      1.818357216161805012e-01, 1.531383769920937332e-01, 1.479819860511658591e-01]


def log1p_pos(z):
    """common.cuh log1p_pos in numpy float64 (no FMA contraction, exact reciprocals): the reduction and fdlibm's kernel."""
    z = np.asarray(z, dtype=np.float64)
    big = z >= np.sqrt(2.0) - 1.0
    a = np.where(big, np.maximum(z, 1.0), 1.0)
    b = np.where(big, np.minimum(z, 1.0), z)
    u = a + b
    c = b - (u - a)
    m, e = np.frexp(u)                     # u = m 2^e, m in [0.5, 1)
    low = m < np.sqrt(0.5)
    m = np.where(low, 2.0 * m, m)
    e = np.where(low, e - 1, e)
    f = np.where(big, m - 1.0, z)
    e = np.where(big, e, 0).astype(np.float64)
    cu = np.where(big, c / u, 0.0)
    s = f / (2.0 + f)
    w = s * s
    R = LG[6]
    for coef in LG[5::-1]:
        R = R * w + coef
    R = R * w
    hfsq = 0.5 * f * f
    v = e * 6.93147180369123816490e-01 - ((hfsq - (s * (hfsq + R) + (e * 1.90821492927058770002e-10 + cu))) - f)
    return np.where(np.isposinf(z), z, v)


RQ32_SPLIT = np.float32(0.25)
RQ32_P = np.array([1.4426950216293335, -0.7213437557220459, 0.48071789741516113, -0.357472687959671, 0.26215097308158875,
                   -0.1332305371761322], dtype=np.float32)


def cov32(r2, variance, alpha):
    """kern_screen.cuh cov32x2_from_r2<KERNEL_RQ> in numpy float32 (MUFU.LG2 / MUFU.EX2 replaced by numpy's log2 / exp2)."""
    r2 = np.asarray(r2, dtype=np.float32)
    alpha = np.float32(alpha)
    z = r2 * (np.float32(0.5) / alpha)
    p = RQ32_P[5]
    for coef in RQ32_P[4::-1]:
        p = (p * z + coef).astype(np.float32)
    with np.errstate(over="ignore"):
        l2 = np.where(z < RQ32_SPLIT, (p * z).astype(np.float32), np.log2(np.float32(1.0) + z)).astype(np.float32)
    return np.float32(variance) * np.exp2((l2 * -alpha).astype(np.float32)).astype(np.float32)


# ---- checker session / backend --------------------------------------------------------------------------------------
class RQOracleSession(OracleSession):
    """OracleSession for the RationalQuadratic kernel (the theta / u vectors carry alpha first)."""

    def neg_lml_and_grad(self, u):
        self.calls["neg_lml_and_grad"] += 1
        return neg_lml_and_grad(self.X, self.y, u, self.n_ls, self.has_mean)

    def factorize(self, theta):
        self.calls["factorize"] += 1
        n = self.n_ls
        self.h = RQHyper(theta[0], theta[1:1 + n] if n > 1 else theta[1], theta[n + 1], theta[n + 2],
                         theta[n + 3] if self.has_mean else None)

    def log_marginal_likelihood(self):
        return lml(self.X, self.y, self.h)

    def _predict(self, xnew):
        if not self.rowwise:
            return predict_y(self.X, self.y, self.h, xnew)
        parts = [predict_y(self.X, self.y, self.h, xnew[i:i + 1]) for i in range(xnew.shape[0])]
        return np.vstack([p[0] for p in parts]), np.vstack([p[1] for p in parts])

    def ucb_topk(self, xnew, varsigma, k):
        mean, var = self._predict(xnew)
        mean, var = mean[:, 0], var[:, 0]
        ucb = mean + varsigma * var
        nan = np.isnan(ucb)
        order = np.lexsort((np.arange(len(ucb)), -np.where(nan, np.inf, ucb), ~nan))[:k]
        return np.column_stack([order.astype(float), mean[order], var[order], ucb[order]])

    def grow_ucb_argmax(self, bounds, depth, varsigma, rows=None):
        leaves = grow_oracle.grow_by_level(bounds, depth)
        if rows is None:
            return self.ucb_argmax(leaves, varsigma)
        idx, mean, var, ucb = self.ucb_argmax(leaves[rows[0]:rows[1]], varsigma)
        return idx + rows[0], mean, var, ucb

    def predict_f_cov(self, xnew):
        return predict_f_full_cov(self.X, self.y, self.h, np.ascontiguousarray(xnew, dtype=np.float64))

    def predict_f_samples(self, xnew, z, jitter):
        mean, cov = self.predict_f_cov(xnew)
        return sample_mvn(mean, cov, np.asarray(z, dtype=np.float64), jitter)


class RQOracleBackend(OracleBackend):
    """Checker backend: RationalQuadratic sessions through the RQ oracle, every other kernel through the shared one."""

    def open_session(self, kernel, n_lengthscales, has_mean):
        if kernel != KERNEL:
            return super().open_session(kernel, n_lengthscales, has_mean)
        session = RQOracleSession(kernel, n_lengthscales, has_mean, rowwise=self.rowwise)
        self.sessions.append(session)
        return session
