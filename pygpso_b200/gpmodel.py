"""
Light-weight stand-ins for the handful of GPflow objects pyGPSO touches, backed by the B200 C-ABI library.

The reference builds ``gpflow.kernels.Matern52``, ``gpflow.mean_functions.Constant``, ``gpflow.optimizers.Scipy``
and ``gpflow.models.GPR`` (gpso/gp_surrogate.py:138,165-169,397,424-429,463-473,490-503) and afterwards only uses

    model.data = (x, y)                      gp_surrogate.py:498
    optimiser.minimize(model.training_loss, model.trainable_variables)     :500-503
    model.predict_y(Xnew) -> (mean[M,1], var[M,1]) with ``.numpy()``      :298,325; plotting.py:351-356
    model.predict_f(Xnew, full_cov=True), model.predict_f_samples(Xnew, S)   (joint posterior, user code)
    model.kernel.lengthscales / .variance, model.likelihood.variance, model.mean_function.c   (summaries, save)
    gpflow.utilities.parameter_dict / multiple_assign / freeze            :462-473,514-519

so exactly that surface is provided here under the same names (``kernels``, ``mean_functions``, ``likelihoods``,
``optimizers``, ``models``, ``utilities``).  All arithmetic (Gram, Cholesky, log-marginal-likelihood and gradient,
posterior mean/variance, UCB argmax) is done by the CUDA library through ``pygpso_b200.backend``; there is no CPU
implementation in this package.

Parameterisation follows GPflow 2: positive parameters are softplus-transformed, the Gaussian likelihood variance has
the 1e-6 floor, and ``trainable_variables`` are ordered kernel.lengthscales, kernel.variance, likelihood.variance,
mean_function.c.
"""
import types

import numpy as np
import scipy.optimize

from . import backend as _backend

NOISE_VARIANCE_FLOOR = 1.0e-6
SAMPLE_JITTER = 1.0e-6  # gpflow.config.default_jitter(): added to the posterior covariance before its Cholesky in predict_f_samples


# ---------------------------------------------------------------------------------------------------------------------
# parameters and transforms
# ---------------------------------------------------------------------------------------------------------------------
def _softplus(u):
    return np.logaddexp(0.0, u)


def _softplus_inv(v):
    # log(expm1(v)); beyond v = 30 the overflow-free form v + log1p(-exp(-v)) (tfp.math.softplus_inverse is stable too)
    v = np.asarray(v, dtype=np.float64)
    small = np.minimum(v, 30.0)
    return np.where(v > 30.0, v + np.log1p(-np.exp(-np.maximum(v, 30.0))), np.log(np.expm1(small)))


class _Shape(tuple):
    """Tuple with TensorShape's ``as_list`` (the reference serialises ``param.shape.as_list()``, :523-527)."""

    def as_list(self):
        return list(self)


class Parameter:
    """
    A (possibly positive-constrained) hyper-parameter.  The constrained value is stored verbatim, so a value that is
    assigned (e.g. when loading a saved model) is used bit-for-bit.  The unconstrained image an optimiser assigned is kept
    beside it (a noise variance that rounds to exactly its 1e-6 floor still has a finite unconstrained value); after an
    explicit ``assign`` it is derived on demand, clamped away from softplus^-1(0) = -inf.
    """

    def __init__(self, value, positive=False, lower=0.0, trainable=True, name=""):
        self._value = np.array(value, dtype=np.float64)
        self._unconstrained = None
        self.positive = positive
        self.lower = float(lower)
        self.trainable = trainable
        self.name = name
        if positive and np.any(self._value <= self.lower):
            raise ValueError(f"parameter {name} must be > {self.lower}, got {self._value}")

    def numpy(self):
        return self._value.copy() if self._value.ndim else np.float64(self._value)

    def __array__(self, dtype=None, copy=None):
        return np.array(self._value, dtype=dtype)

    def __float__(self):
        return float(self._value.reshape(-1)[0]) if self._value.size == 1 else float(self._value)

    @property
    def shape(self):
        return _Shape(self._value.shape)

    @property
    def size(self):
        return int(self._value.size)

    def assign(self, value):
        value = np.array(value, dtype=np.float64)
        if value.shape != self._value.shape:
            if value.size != self._value.size:
                raise ValueError(f"cannot assign shape {value.shape} to parameter of shape {self._value.shape}")
            value = value.reshape(self._value.shape)
        if self.positive and np.any(value <= self.lower):
            raise ValueError(f"parameter {self.name} must be > {self.lower}")
        self._value = value
        self._unconstrained = None

    @property
    def unconstrained(self):
        if self._unconstrained is not None:
            return self._unconstrained.copy()
        flat = self._value.reshape(-1)
        if not self.positive:
            return flat.copy()
        return _softplus_inv(np.maximum(flat - self.lower, np.finfo(np.float64).tiny))

    def assign_unconstrained(self, u):
        u = np.array(u, dtype=np.float64).reshape(self._value.shape)
        self._value = np.array(self.lower + _softplus(u) if self.positive else u, dtype=np.float64)
        self._unconstrained = u.reshape(-1).copy()

    def __repr__(self):
        return f"Parameter({self.name}={self._value!r})"


# ---------------------------------------------------------------------------------------------------------------------
# kernels / mean functions / likelihood
# ---------------------------------------------------------------------------------------------------------------------
class Kernel:
    pass


class Stationary(Kernel):
    """Isotropic / ARD stationary kernel; ``lengthscales`` scalar or one per dimension."""

    def __init__(self, variance=1.0, lengthscales=1.0):
        self.variance = Parameter(variance, positive=True, name="kernel.variance")
        self.lengthscales = Parameter(lengthscales, positive=True, name="kernel.lengthscales")

    @property
    def ard(self):
        return self.lengthscales.size > 1 or len(self.lengthscales.shape) > 0 and self.lengthscales.shape[0] > 1

    @property
    def parameters(self):
        return (self.lengthscales, self.variance)


class Matern12(Stationary):
    pass


class Matern32(Stationary):
    pass


class Matern52(Stationary):
    pass


class SquaredExponential(Stationary):
    pass


RBF = SquaredExponential


class MeanFunction:
    parameters = ()


class Zero(MeanFunction):
    pass


class Constant(MeanFunction):
    def __init__(self, c=None):
        c = np.zeros(1) if c is None else c
        self.c = Parameter(c, positive=False, name="mean_function.c")
        if self.c.size != 1:
            raise ValueError("only a scalar constant mean is supported (pyGPSO scores are one-dimensional)")

    @property
    def parameters(self):
        return (self.c,)


class Gaussian:
    def __init__(self, variance=1.0):
        self.variance = Parameter(variance, positive=True, lower=NOISE_VARIANCE_FLOOR, name="likelihood.variance")

    @property
    def parameters(self):
        return (self.variance,)


# ---------------------------------------------------------------------------------------------------------------------
# host-side result type
# ---------------------------------------------------------------------------------------------------------------------
class HostTensor(np.ndarray):
    """ndarray that also answers ``.numpy()`` (callers written against tf.Tensor do ``predict_y(x)[0].numpy()``)."""

    def numpy(self):
        return np.asarray(self)


def _as_host_tensor(a):
    return np.ascontiguousarray(a, dtype=np.float64).view(HostTensor)


# ---------------------------------------------------------------------------------------------------------------------
# the model
# ---------------------------------------------------------------------------------------------------------------------
class GPModel:
    pass


class GPR(GPModel):
    """
    Gaussian-process regression with a Gaussian likelihood; the role of ``gpflow.models.GPR``.  Owns one session of
    the device library (training data, Cholesky factor, inverse factor and alpha stay resident in HBM between calls).
    """

    def __init__(self, data, kernel, mean_function=None, noise_variance=1.0, backend=None):
        if not isinstance(kernel, Stationary):
            raise TypeError("kernel must be one of Matern12 / Matern32 / Matern52 / SquaredExponential")
        self.kernel = kernel
        self.mean_function = Zero() if mean_function is None else mean_function
        if not isinstance(self.mean_function, (Zero, Constant)):
            raise TypeError("mean_function must be Zero or Constant")
        self.likelihood = Gaussian(noise_variance)
        self._backend = backend if backend is not None else _backend.default_backend()
        self._session = self._backend.open_session(
            kernel=type(kernel).__name__,
            n_lengthscales=self.kernel.lengthscales.size,
            has_mean=isinstance(self.mean_function, Constant),
        )
        self._factor_key = None
        self.n_loss_evaluations = 0
        self.data = data

    # -- data ---------------------------------------------------------------------------------------------------------
    @property
    def data(self):
        return self._data

    @data.setter
    def data(self, value):
        x, y = value
        x = np.ascontiguousarray(x, dtype=np.float64)
        y = np.ascontiguousarray(y, dtype=np.float64)
        if x.ndim != 2 or y.ndim != 2 or y.shape != (x.shape[0], 1):
            raise ValueError(f"data must be (X[N,d], Y[N,1]); got {x.shape}, {y.shape}")
        if self.kernel.lengthscales.size not in (1, x.shape[1]):
            raise ValueError("ARD lengthscales must have one entry per input dimension")
        self._data = (x, y)
        self._session.set_data(x, y)
        self._factor_key = None

    # -- parameters ---------------------------------------------------------------------------------------------------
    @property
    def _ordered_parameters(self):
        params = [self.kernel.lengthscales, self.kernel.variance, self.likelihood.variance]
        params.extend(self.mean_function.parameters)
        return params

    @property
    def trainable_variables(self):
        return tuple(p for p in self._ordered_parameters if p.trainable)

    @property
    def parameters(self):
        return tuple(self._ordered_parameters)

    def _pack(self):
        return np.concatenate([p.unconstrained for p in self._ordered_parameters])

    def _unpack(self, u):
        pos = 0
        for p in self._ordered_parameters:
            p.assign_unconstrained(u[pos:pos + p.size])
            pos += p.size

    def _theta(self):
        """Constrained vector in packing order: lengthscale(s), kernel variance, noise variance, [mean c]."""
        return np.concatenate([np.asarray(p, dtype=np.float64).reshape(-1) for p in self._ordered_parameters])

    # -- objective ----------------------------------------------------------------------------------------------------
    def neg_log_marginal_likelihood_and_grad(self, u):
        """(-LML, d(-LML)/du) at the packed unconstrained vector ``u``; evaluated on the device."""
        self.n_loss_evaluations += 1
        self._factor_key = None  # the evaluation overwrites the device factor
        return self._session.neg_lml_and_grad(np.ascontiguousarray(u, dtype=np.float64))

    def training_loss(self):
        return self.neg_log_marginal_likelihood_and_grad(self._pack())[0]

    def log_marginal_likelihood(self):
        return -self.training_loss()

    # -- posterior ----------------------------------------------------------------------------------------------------
    def _ensure_factor(self):
        theta = self._theta()
        key = theta.tobytes()
        # the session drops its factor whenever a loss evaluation or an engine switch overwrote it (same theta or not)
        if key != self._factor_key or not getattr(self._session, "factorized", True):
            self._session.factorize(theta)
            self._factor_key = key

    def _candidates(self, Xnew):
        Xnew = np.ascontiguousarray(Xnew, dtype=np.float64)
        if Xnew.ndim != 2 or Xnew.shape[1] != self._data[0].shape[1]:
            raise ValueError(f"Xnew must be [M,{self._data[0].shape[1]}], got {Xnew.shape}")
        return Xnew

    def predict_y(self, Xnew):
        """Posterior mean and variance *including* the noise variance, both ``[M,1]``."""
        Xnew = self._candidates(Xnew)
        self._ensure_factor()
        mean, var = self._session.predict_y(Xnew)
        return _as_host_tensor(mean).reshape(-1, 1), _as_host_tensor(var).reshape(-1, 1)

    def predict_f(self, Xnew, full_cov=False, full_output_cov=False):
        """Posterior of the latent function: mean ``[M,1]`` and variance ``[M,1]``, or with ``full_cov`` the covariance
        ``[1,M,M]`` of the M candidates jointly (no noise variance; at most ``backend.MAX_JOINT`` candidates per call).
        ``full_output_cov`` has no effect: the model has a single output."""
        if not full_cov:
            mean, var = self.predict_y(Xnew)
            return mean, _as_host_tensor(var - float(self.likelihood.variance))
        Xnew = self._candidates(Xnew)
        self._ensure_factor()
        mean, cov = self._session.predict_f_cov(Xnew)
        return _as_host_tensor(mean).reshape(-1, 1), _as_host_tensor(cov).reshape(1, Xnew.shape[0], Xnew.shape[0])

    def predict_f_samples(self, Xnew, num_samples=None, full_cov=True, full_output_cov=False, seed=None):
        """Draws of the latent function at ``Xnew``: ``[S,M,1]``, or ``[M,1]`` when ``num_samples`` is None.
        ``full_cov``: joint draws ``mean + chol(cov + SAMPLE_JITTER I) z``; otherwise independent ``mean + sqrt(var) z``.
        The standard normals ``z[S,M]`` come from ``np.random.default_rng(seed)`` (the one keyword GPflow lacks: its
        TensorFlow random stream cannot be reproduced, a seed makes draws reproducible)."""
        Xnew = self._candidates(Xnew)
        S = 1 if num_samples is None else int(num_samples)
        if S < 1:
            raise ValueError(f"num_samples must be positive, got {num_samples}")
        z = np.random.default_rng(seed).standard_normal((S, Xnew.shape[0]))
        if full_cov:
            self._ensure_factor()
            f = self._session.predict_f_samples(Xnew, z, SAMPLE_JITTER)
        else:
            mean, var = self.predict_f(Xnew)
            f = mean[:, 0] + np.sqrt(var[:, 0]) * z
        f = _as_host_tensor(f)
        return f[0].reshape(-1, 1) if num_samples is None else f.reshape(S, -1, 1)

    def ucb_argmax(self, Xnew, varsigma):
        """Fused predict_y + ``mean + varsigma*var`` + first-max argmax.  Returns (index, mean, var, ucb)."""
        Xnew = np.ascontiguousarray(Xnew, dtype=np.float64)
        self._ensure_factor()
        return self._session.ucb_argmax(Xnew, float(varsigma))

    def ucb_topk(self, Xnew, varsigma, k):
        """The k candidates with the highest ``mean + varsigma * var`` in arg-max order: rows (index, mean, var, ucb)."""
        self._ensure_factor()
        return self._session.ucb_topk(np.asarray(Xnew, dtype=np.float64), varsigma, k)

    def grow_ucb_argmax(self, bounds, depth, varsigma):
        """Generate the ``grow(depth)`` leaf-centre batch of the box ``bounds[d,2]`` on the device and score it."""
        self._ensure_factor()
        return self._session.grow_ucb_argmax(np.ascontiguousarray(bounds, dtype=np.float64), int(depth), float(varsigma))

    def close(self):
        if self._session is not None:
            self._session.close()
            self._session = None


# ---------------------------------------------------------------------------------------------------------------------
# optimiser
# ---------------------------------------------------------------------------------------------------------------------
class Scipy:
    """
    ``gpflow.optimizers.Scipy``: SciPy L-BFGS-B (SciPy defaults) over the packed unconstrained variables; only the
    objective/gradient closure runs on the GPU, the line search and two-loop recursion stay in SciPy on the host.
    """

    def minimize(self, closure, variables, method="L-BFGS-B", **scipy_kwargs):
        model = getattr(closure, "__self__", None)
        if not isinstance(model, GPR):
            raise TypeError("Scipy.minimize expects the bound method `model.training_loss` of a GPR model")
        u_full = model._pack()
        # optimise over `variables` only (GPflow passes model.trainable_variables): entries of the packed vector that belong
        # to parameters outside that set (or with trainable=False) stay at their current values
        wanted = {id(v) for v in variables} if variables is not None else None
        free = np.zeros(u_full.size, dtype=bool)
        pos = 0
        for p in model._ordered_parameters:
            free[pos:pos + p.size] = p.trainable and (wanted is None or id(p) in wanted)
            pos += p.size
        if free.all():
            objective = model.neg_log_marginal_likelihood_and_grad
        else:
            def objective(u_free):
                u = u_full.copy()
                u[free] = u_free
                f, g = model.neg_log_marginal_likelihood_and_grad(u)
                return f, g[free]
        result = scipy.optimize.minimize(objective, u_full[free], jac=True, method=method, **scipy_kwargs)
        u_full[free] = result.x
        model._unpack(u_full)
        return result


# ---------------------------------------------------------------------------------------------------------------------
# gpflow.utilities look-alikes (used by save / load)
# ---------------------------------------------------------------------------------------------------------------------
def parameter_dict(model):
    out = {
        ".kernel.lengthscales": model.kernel.lengthscales,
        ".kernel.variance": model.kernel.variance,
        ".likelihood.variance": model.likelihood.variance,
    }
    if isinstance(model.mean_function, Constant):
        out[".mean_function.c"] = model.mean_function.c
    return out


def multiple_assign(model, values):
    targets = parameter_dict(model)
    for key, value in values.items():
        if key not in targets:
            raise KeyError(f"model has no parameter {key}")
        targets[key].assign(value.numpy() if hasattr(value, "numpy") else value)
    model._factor_key = None


def freeze(model):
    return model


def tabulate_module_summary(model):
    rows = ["name                      shape   value"]
    for key, p in parameter_dict(model).items():
        rows.append(f"GPR{key:<22} {str(tuple(p.shape)):<7} {np.asarray(p)!r}")
    return "\n".join(rows)


kernels = types.SimpleNamespace(
    Kernel=Kernel, Stationary=Stationary, Matern12=Matern12, Matern32=Matern32, Matern52=Matern52,
    SquaredExponential=SquaredExponential, RBF=RBF,
)
mean_functions = types.SimpleNamespace(MeanFunction=MeanFunction, Zero=Zero, Constant=Constant)
likelihoods = types.SimpleNamespace(Gaussian=Gaussian)
optimizers = types.SimpleNamespace(Scipy=Scipy)
models = types.SimpleNamespace(GPModel=GPModel, GPR=GPR)
utilities = types.SimpleNamespace(
    parameter_dict=parameter_dict, multiple_assign=multiple_assign, freeze=freeze,
    tabulate_module_summary=tabulate_module_summary,
)
