"""
Joint posterior in the numpy oracle (test infrastructure only): ``gpflow.models.GPR.predict_f(Xnew, full_cov=True)`` and the
sampling of ``predict_f_samples``, restated in GPflow 2's op order, and a checker session with the two joint calls on top of
``tests/oracle_backend.OracleSession``.
"""
import numpy as np
import scipy.linalg as sla

from oracle import gpr_oracle as go
from tests.oracle_backend import OracleBackend, OracleSession


def predict_f_full_cov(kernel, X, y, h, Xnew):
    """gpflow.conditionals.base_conditional(full_cov=True): (mean[M,1], cov[M,M]) with cov = Knn - A^T A, A = Lm^-1 Kmn."""
    N = X.shape[0]
    c = h.mean_c if h.has_mean else 0.0
    Kmm = go.kern(kernel, X, None, h) + h.noise_variance * np.eye(N)
    Lm = np.linalg.cholesky(Kmm)
    Kmn = go.kern(kernel, X, Xnew, h)
    Knn = go.kern(kernel, Xnew, None, h)
    A = sla.solve_triangular(Lm, Kmn, lower=True)
    fcov = Knn - A.T @ A
    A = sla.solve_triangular(Lm, A, lower=True, trans="T")
    fmean = A.T @ (y[:, 0] - c)
    return (fmean + c)[:, None], fcov


def sample_mvn(mean, cov, z, jitter):
    """Draws [S,M] = mean + z chol(cov + jitter I)^T for standard normals z[S,M] (gpflow.conditionals.util.sample_mvn)."""
    L = np.linalg.cholesky(cov + jitter * np.eye(cov.shape[0]))
    return np.ravel(mean)[None, :] + z @ L.T


class JointOracleSession(OracleSession):
    def predict_f_cov(self, xnew):
        mean, cov = predict_f_full_cov(self.kernel, self.X, self.y, self.h, np.ascontiguousarray(xnew, dtype=np.float64))
        return mean[:, 0], cov

    def predict_f_samples(self, xnew, z, jitter):
        mean, cov = self.predict_f_cov(xnew)
        return sample_mvn(mean, cov, np.asarray(z, dtype=np.float64), jitter)


class JointOracleBackend(OracleBackend):
    def open_session(self, kernel, n_lengthscales, has_mean):
        session = JointOracleSession(kernel, n_lengthscales, has_mean, rowwise=self.rowwise)
        self.sessions.append(session)
        return session
