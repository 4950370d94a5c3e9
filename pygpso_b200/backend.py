"""
ctypes binding of the C-ABI library ``libgpso_b200.so`` (declared in ``include/gpso_b200.h``).

This is the only compute backend of the package.  If the shared library is missing, cannot be loaded, or no sm_100
GPU is visible, every entry point raises ``GpsoBackendError`` -- there is deliberately no CPU fallback (the numpy
oracle under ``oracle/`` is test infrastructure and is never imported from here).

A *session* is one ``gpso_handle``: the device-resident state of one GPR surrogate on one GPU.
"""
import ctypes
import os

import numpy as np

KERNEL_IDS = {"Matern12": 0, "Matern32": 1, "Matern52": 2, "SquaredExponential": 3, "RationalQuadratic": 4}
KERNEL_PERIODIC = 7  # GPSO_KERNEL_PERIODIC
KERNEL_LINEAR = 10  # GPSO_KERNEL_LINEAR (gpflow.kernels.Linear)
_LIB_NAME = "libgpso_b200.so"
_ABI_VERSION = 1

_c_double_p = ctypes.POINTER(ctypes.c_double)
MAX_JOINT = 8192  # GPSO_MAX_JOINT: candidates per joint-posterior call (predict_f_cov / predict_f_samples)


class GpsoBackendError(RuntimeError):
    """The CUDA library is unavailable or a device call failed."""


class NotPositiveDefiniteError(np.linalg.LinAlgError):
    """Cholesky of K + noise*I broke down (the C ABI returned a LAPACK-style info > 0)."""


def _dptr(a):
    return a.ctypes.data_as(_c_double_p)


def library_path():
    """The in-tree library; ``GPSO_LIBRARY`` points at another build of the same sources (A/B experiments of compile-time
    kernel parameters)."""
    return os.environ.get("GPSO_LIBRARY") or os.path.join(os.path.dirname(os.path.abspath(__file__)), _LIB_NAME)


_lib = None
_cuda_touched = False


def cuda_initialised():
    """True once this process has opened a CUDA context through this package or through torch (fork safety of the
    objective worker pool, optimisation.py)."""
    if _cuda_touched:
        return True
    import sys

    torch = sys.modules.get("torch")
    try:
        return bool(torch is not None and torch.cuda.is_initialized())
    except Exception:
        return False


def load_library():
    """dlopen the in-tree library and declare the prototypes.  Raises GpsoBackendError when it is not there."""
    global _lib
    if _lib is not None:
        return _lib
    path = library_path()
    if not os.path.exists(path):
        raise GpsoBackendError(
            f"{path} not found: build it with `python -m pygpso_b200._build` (needs nvcc). "
            "pygpso_b200 has no CPU fallback."
        )
    try:
        lib = ctypes.CDLL(path)
    except OSError as err:
        raise GpsoBackendError(f"cannot load {path}: {err}") from err
    H = ctypes.c_void_p
    i32, i64, dbl = ctypes.c_int, ctypes.c_int64, ctypes.c_double
    protos = {
        "gpso_version": (i32, []),
        "gpso_last_error": (ctypes.c_char_p, []),
        "gpso_device_count": (i32, []),
        "gpso_create": (i32, [i32, i32, i32, i32, ctypes.POINTER(H)]),
        "gpso_create_sum": (i32, [i32, i32, ctypes.POINTER(ctypes.c_int), ctypes.POINTER(ctypes.c_int), i32, ctypes.POINTER(H)]),
        "gpso_create_product": (i32, [i32, i32, ctypes.POINTER(ctypes.c_int), ctypes.POINTER(ctypes.c_int), i32, ctypes.POINTER(H)]),
        "gpso_create_periodic": (i32, [i32, i32, i32, i32, i32, ctypes.POINTER(H)]),
        "gpso_create_combination": (i32, [i32, i32, i32, ctypes.POINTER(ctypes.c_int), ctypes.POINTER(ctypes.c_int),
                                          ctypes.POINTER(ctypes.c_int), ctypes.POINTER(ctypes.c_int), i32, ctypes.POINTER(H)]),
        "gpso_destroy": (i32, [H]),
        "gpso_set_data": (i32, [H, _c_double_p, _c_double_p, i32, i32]),
        "gpso_set_active_dims": (i32, [H, i32, ctypes.POINTER(ctypes.c_int), ctypes.POINTER(ctypes.c_int)]),
        "gpso_neg_lml_grad": (i32, [H, _c_double_p, i32, _c_double_p, _c_double_p]),
        "gpso_factorize": (i32, [H, _c_double_p, i32]),
        "gpso_factor_lml": (i32, [H, _c_double_p]),
        "gpso_predict_y_host": (i32, [H, _c_double_p, i64, _c_double_p, _c_double_p]),
        "gpso_predict_y_dev": (i32, [H, ctypes.c_void_p, i64, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p]),
        "gpso_predict_f_cov_host": (i32, [H, _c_double_p, i64, _c_double_p, _c_double_p]),
        "gpso_predict_f_cov_dev": (i32, [H, ctypes.c_void_p, i64, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p]),
        "gpso_predict_f_samples_host": (i32, [H, _c_double_p, i64, i32, dbl, _c_double_p, _c_double_p]),
        "gpso_predict_f_samples_dev": (i32, [H, ctypes.c_void_p, i64, i32, dbl, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p]),
        "gpso_ucb_argmax_host": (i32, [H, _c_double_p, i64, dbl, _c_double_p]),
        "gpso_ucb_argmax_dev": (i32, [H, ctypes.c_void_p, i64, dbl, _c_double_p, ctypes.c_void_p]),
        "gpso_ucb_topk_host": (i32, [H, _c_double_p, i64, dbl, i32, _c_double_p, ctypes.POINTER(ctypes.c_int)]),
        "gpso_ucb_topk_dev": (i32, [H, ctypes.c_void_p, i64, dbl, i32, _c_double_p, ctypes.POINTER(ctypes.c_int), ctypes.c_void_p]),
        "gpso_grow_count": (i64, [i32]),
        "gpso_grow_leaves_host": (i32, [i32, _c_double_p, i32, i32, _c_double_p]),
        "gpso_grow_leaves_dev": (i32, [i32, _c_double_p, i32, i32, ctypes.c_void_p, ctypes.c_void_p]),
        "gpso_grow_ucb_argmax": (i32, [H, _c_double_p, i32, i32, dbl, _c_double_p]),
        "gpso_grow_ucb_argmax_range": (i32, [H, _c_double_p, i32, i32, dbl, i64, i64, _c_double_p]),
        "gpso_state_bytes": (i32, [H, i32, i32, ctypes.POINTER(i64)]),
        "gpso_export_state_dev": (i32, [H, ctypes.c_void_p, i64, ctypes.c_void_p]),
        "gpso_import_state_dev": (i32, [H, ctypes.c_void_p, i64, i32, i32, ctypes.c_void_p]),
        "gpso_launch_count": (i64, [H]),
        "gpso_debug_fetch": (i32, [H, i32, _c_double_p, i64]),
        "gpso_last_timing": (i32, [H, _c_double_p]),
        "gpso_set_window": (i32, [H, i64]),
        "gpso_set_predict_mode": (i32, [H, i32, i32]),
        "gpso_predict_info": (i32, [H, _c_double_p]),
        "gpso_set_overlap": (i32, [H, i32]),
        "gpso_set_factor_mode": (i32, [H, i32]),
        "gpso_factor_info": (i32, [H, ctypes.POINTER(ctypes.c_int)]),
        "gpso_trim_pool": (i32, [i32, ctypes.POINTER(ctypes.c_int64)]),
        "gpso_debug_screen_windows": (i64, [i64, i64, i32, i32, ctypes.POINTER(ctypes.c_int64), i64]),
        "gpso_debug_hybrid_plan": (i64, [i32, i32, ctypes.POINTER(ctypes.c_int), i64]),
        "gpso_debug_hybrid_items": (i64, [i32, i32, i32, i32, ctypes.POINTER(ctypes.c_int), i64, ctypes.POINTER(ctypes.c_int)]),
        "gpso_debug_factor_tasks": (i32, [i32, i32, ctypes.POINTER(ctypes.c_int), i64, ctypes.POINTER(ctypes.c_int), ctypes.POINTER(ctypes.c_int)]),
        "gpso_debug_factor_tasks_cap": (i32, [i32, i32, i32, ctypes.POINTER(ctypes.c_int), i64, ctypes.POINTER(ctypes.c_int), ctypes.POINTER(ctypes.c_int)]),
        "gpso_set_profile": (i32, [H, i32]),
        "gpso_last_windows": (i64, [H]),
        "gpso_debug_trace": (i64, [H, _c_double_p, i64]),
        "gpso_set_kinv_mode": (i32, [H, i32]),
        "gpso_set_inverse_mode": (i32, [H, i32]),
        "gpso_set_l2_window": (i32, [H, i32]),
        "gpso_set_screen_mode": (i32, [H, i32]),
        "gpso_screen_info": (i32, [H, _c_double_p]),
        "gpso_probe_peaks": (i32, [i32, _c_double_p]),
        "gpso_debug_screen_bound": (i32, [i32, dbl, dbl, _c_double_p, i32, i32, dbl, _c_double_p]),
        "gpso_debug_product_items": (i64, [i32, i32, i32, ctypes.POINTER(ctypes.c_int), i64, ctypes.POINTER(ctypes.c_int), i32,
                                           ctypes.POINTER(ctypes.c_int)]),
    }
    for name, (restype, argtypes) in protos.items():
        try:
            fn = getattr(lib, name)
        except AttributeError as err:
            raise GpsoBackendError(f"{path} does not export {name}") from err
        fn.restype = restype
        fn.argtypes = argtypes
    if lib.gpso_version() != _ABI_VERSION:
        raise GpsoBackendError(f"{path}: ABI version {lib.gpso_version()} != expected {_ABI_VERSION}")
    _lib = lib
    return lib


EXPORTED_SYMBOLS = (
    "gpso_version gpso_last_error gpso_device_count gpso_create gpso_create_sum gpso_create_product gpso_create_periodic gpso_create_combination gpso_destroy gpso_set_data gpso_set_active_dims gpso_neg_lml_grad "
    "gpso_factorize gpso_factor_lml gpso_predict_y_host gpso_predict_y_dev gpso_ucb_argmax_host gpso_ucb_argmax_dev "
    "gpso_ucb_topk_host gpso_ucb_topk_dev "
    "gpso_predict_f_cov_host gpso_predict_f_cov_dev gpso_predict_f_samples_host gpso_predict_f_samples_dev "
    "gpso_grow_count gpso_grow_leaves_host gpso_grow_leaves_dev gpso_grow_ucb_argmax gpso_grow_ucb_argmax_range gpso_state_bytes "
    "gpso_export_state_dev gpso_import_state_dev gpso_launch_count gpso_debug_fetch gpso_last_timing gpso_set_window "
    "gpso_set_profile gpso_last_windows gpso_set_predict_mode gpso_predict_info gpso_set_overlap "
    "gpso_set_factor_mode gpso_factor_info gpso_trim_pool gpso_debug_screen_windows gpso_debug_hybrid_plan gpso_debug_hybrid_items gpso_debug_factor_tasks gpso_debug_factor_tasks_cap gpso_debug_trace gpso_set_kinv_mode gpso_set_inverse_mode gpso_set_l2_window gpso_debug_product_items "
    "gpso_set_screen_mode gpso_screen_info gpso_debug_screen_bound gpso_probe_peaks"
).split()


def _check(lib, rc, what):
    if rc == 0:
        return
    text = lib.gpso_last_error().decode("utf-8", "replace")
    if rc > 0:
        raise NotPositiveDefiniteError(f"{what}: {text}")
    raise GpsoBackendError(f"{what} failed (status {rc}): {text}")


def _joint_candidates(xnew):
    xnew = np.ascontiguousarray(xnew, dtype=np.float64)
    if not 1 <= xnew.shape[0] <= MAX_JOINT:
        raise ValueError(f"the joint posterior takes 1..{MAX_JOINT} candidates per call, got {xnew.shape[0]}; draw larger sets in batches")
    return xnew


def default_device():
    """GPU index for this process: GPSO_DEVICE if set, else LOCAL_RANK (torchrun), else 0."""
    for var in ("GPSO_DEVICE", "LOCAL_RANK"):
        if var in os.environ:
            return int(os.environ[var])
    return 0


class CudaSession:
    """One gpso_handle."""

    def __init__(self, lib, device, kernel, n_lengthscales, has_mean, components=None):
        """``components``: for ``kernel="Sum"`` (``"Product"``) the list ``[(family, n_lengthscales), ...]`` of the sum's
        components (the product's factors), ``("Periodic", n_lengthscales, base family, n_periods)`` for a periodic one; for
        ``kernel="Periodic"`` the one entry ``[(base family, n_periods)]``, the base
        being SquaredExponential or RationalQuadratic with ``n_lengthscales`` lengthscales.  A sum's component may be
        ``("Linear", n_variances)``; ``kernel="Linear"`` is a bare Linear kernel with ``n_lengthscales`` variances."""
        self._lib = lib
        self.device = device
        self.kernel = kernel
        # has_mean is the mean id of the C ABI: 0 / False none, 1 / True constant, 2 linear (m(x) = x . A + b)
        self.mean_id = int(has_mean)
        self.has_mean = bool(has_mean)
        handle = ctypes.c_void_p()
        if kernel in ("Sum", "Product"):
            def known(c):
                return (c[0] in KERNEL_IDS or (c[0] == "Periodic" and len(c) == 4 and c[2] in ("SquaredExponential", "RationalQuadratic"))
                        or (c[0] == "Linear" and len(c) == 2))
            if not components or not all(known(c) for c in components):
                raise ValueError(f"a {kernel} session needs components from {sorted(KERNEL_IDS)} or periodic ones, got {components!r}")
            self.components = [tuple(c) for c in components]
            self.ard = False
            n = len(self.components)
            periodic = [c[0] == "Periodic" for c in self.components]
            linear = [c[0] == "Linear" for c in self.components]
            ids = (ctypes.c_int * n)(*[KERNEL_PERIODIC if p else KERNEL_LINEAR if lin else KERNEL_IDS[c[0]]
                                       for c, p, lin in zip(self.components, periodic, linear)])
            ards = (ctypes.c_int * n)(*[int(c[1] > 1) for c in self.components])
            if any(periodic) or any(linear):
                bases = (ctypes.c_int * n)(*[KERNEL_IDS[c[2]] if p else 0 for c, p in zip(self.components, periodic)])
                pards = (ctypes.c_int * n)(*[int(c[3] > 1) if p else 0 for c, p in zip(self.components, periodic)])
                kind = 5 if kernel == "Sum" else 6
                _check(lib, lib.gpso_create_combination(device, kind, n, ids, ards, bases, pards, self.mean_id, ctypes.byref(handle)),
                       "gpso_create_combination")
            else:
                create = "gpso_create_sum" if kernel == "Sum" else "gpso_create_product"
                _check(lib, getattr(lib, create)(device, n, ids, ards, self.mean_id, ctypes.byref(handle)), create)
        elif kernel == "Periodic":
            if not components or len(components) != 1 or components[0][0] not in ("SquaredExponential", "RationalQuadratic"):
                raise ValueError(f"a Periodic session needs [(base family, n_periods)] with a SquaredExponential or RationalQuadratic "
                                 f"base, got {components!r}")
            base, n_periods = components[0]
            self.components = [(base, int(n_periods))]
            self.ard = n_lengthscales > 1
            _check(lib, lib.gpso_create_periodic(device, KERNEL_IDS[base], int(self.ard), int(n_periods > 1), self.mean_id,
                                                 ctypes.byref(handle)), "gpso_create_periodic")
        elif kernel == "Linear":
            self.ard = n_lengthscales > 1
            _check(lib, lib.gpso_create(device, KERNEL_LINEAR, int(self.ard), self.mean_id, ctypes.byref(handle)), "gpso_create")
        else:
            if kernel not in KERNEL_IDS:
                raise ValueError(f"unsupported kernel {kernel!r}; choose from {sorted(KERNEL_IDS)}, Sum or Product")
            self.ard = n_lengthscales > 1
            _check(lib, lib.gpso_create(device, KERNEL_IDS[kernel], int(self.ard), self.mean_id, ctypes.byref(handle)),
                   "gpso_create")
        self._h = handle
        self.N = self.d = 0
        # mirrors the handle's own flag: every call that overwrites the device factor (a loss evaluation, new data, an engine
        # switch) clears it, so the model re-factorises before the next prediction even at unchanged hyper-parameters
        self.factorized = False

    # -- fit ----------------------------------------------------------------------------------------------------------
    def set_active_dims(self, leaf_dims):
        """The input columns of each leaf (the bare kernel, or each component / factor in order; a periodic one's base), or None
        for every column in order.  Drops the data: call ``set_data`` next."""
        dims = [] if leaf_dims is None else [[int(i) for i in cols] for cols in leaf_dims]
        counts = (ctypes.c_int * max(len(dims), 1))(*[len(cols) for cols in dims])
        flat = [i for cols in dims for i in cols]
        cols = (ctypes.c_int * max(len(flat), 1))(*flat)
        self.factorized = False
        _check(self._lib, self._lib.gpso_set_active_dims(self._h, len(dims), counts, cols), "gpso_set_active_dims")
        self.N = self.d = 0

    def set_data(self, x, y):
        x = np.ascontiguousarray(x, dtype=np.float64)
        y = np.ascontiguousarray(y, dtype=np.float64).reshape(-1)
        self.factorized = False
        _check(self._lib, self._lib.gpso_set_data(self._h, _dptr(x), _dptr(y), x.shape[0], x.shape[1]), "gpso_set_data")
        self.N, self.d = x.shape

    def neg_lml_and_grad(self, u):
        u = np.ascontiguousarray(u, dtype=np.float64)
        f = ctypes.c_double()
        grad = np.empty_like(u)
        self.factorized = False
        _check(self._lib, self._lib.gpso_neg_lml_grad(self._h, _dptr(u), u.size, ctypes.byref(f), _dptr(grad)),
               "gpso_neg_lml_grad")
        return float(f.value), grad

    def factorize(self, theta):
        theta = np.ascontiguousarray(theta, dtype=np.float64)
        self.factorized = False
        _check(self._lib, self._lib.gpso_factorize(self._h, _dptr(theta), theta.size), "gpso_factorize")
        self.factorized = True

    def log_marginal_likelihood(self):
        v = ctypes.c_double()
        _check(self._lib, self._lib.gpso_factor_lml(self._h, ctypes.byref(v)), "gpso_factor_lml")
        return float(v.value)

    # -- predict ------------------------------------------------------------------------------------------------------
    def predict_y(self, xnew):
        xnew = np.ascontiguousarray(xnew, dtype=np.float64)
        m = xnew.shape[0]
        mean = np.empty(m)
        var = np.empty(m)
        if m:
            _check(self._lib, self._lib.gpso_predict_y_host(self._h, _dptr(xnew), m, _dptr(mean), _dptr(var)),
                   "gpso_predict_y_host")
        return mean, var

    def predict_f_cov(self, xnew):
        """Joint posterior of the latent function: mean[M] and the full covariance cov[M,M] (no noise variance)."""
        xnew = _joint_candidates(xnew)
        m = xnew.shape[0]
        mean = np.empty(m)
        cov = np.empty((m, m))
        _check(self._lib, self._lib.gpso_predict_f_cov_host(self._h, _dptr(xnew), m, _dptr(mean), _dptr(cov)),
               "gpso_predict_f_cov_host")
        return mean, cov

    def predict_f_samples(self, xnew, z, jitter):
        """Posterior draws [S,M] = mean + z chol(cov + jitter I)^T for standard normals z[S,M]; a covariance that is not
        positive definite raises NotPositiveDefiniteError."""
        xnew = _joint_candidates(xnew)
        z = np.ascontiguousarray(z, dtype=np.float64)
        if z.ndim != 2 or z.shape[1] != xnew.shape[0] or z.shape[0] < 1:
            raise ValueError(f"z must be [S,{xnew.shape[0]}] with S >= 1, got {z.shape}")
        out = np.empty(z.shape)
        _check(self._lib, self._lib.gpso_predict_f_samples_host(self._h, _dptr(xnew), xnew.shape[0], z.shape[0], float(jitter),
                                                                _dptr(z), _dptr(out)), "gpso_predict_f_samples_host")
        return out

    def ucb_argmax(self, xnew, varsigma):
        xnew = np.ascontiguousarray(xnew, dtype=np.float64)
        out = np.empty(4)
        _check(self._lib, self._lib.gpso_ucb_argmax_host(self._h, _dptr(xnew), xnew.shape[0], float(varsigma), _dptr(out)),
               "gpso_ucb_argmax_host")
        return int(out[0]), float(out[1]), float(out[2]), float(out[3])

    def ucb_topk(self, xnew, varsigma, k):
        """The k best candidates in arg-max order: array [found, 4] of (index, mean, var, ucb); row 0 == ``ucb_argmax``."""
        xnew = np.ascontiguousarray(xnew, dtype=np.float64)
        out = np.zeros((int(k), 4))
        found = ctypes.c_int(0)
        _check(self._lib, self._lib.gpso_ucb_topk_host(self._h, _dptr(xnew), xnew.shape[0], float(varsigma), int(k), _dptr(out),
                                                       ctypes.byref(found)), "gpso_ucb_topk_host")
        return out[: found.value]

    def ucb_topk_dev(self, xc_ptr, m, varsigma, k, stream=0):
        out = np.zeros((int(k), 4))
        found = ctypes.c_int(0)
        _check(self._lib, self._lib.gpso_ucb_topk_dev(self._h, xc_ptr, m, float(varsigma), int(k), _dptr(out), ctypes.byref(found),
                                                      stream), "gpso_ucb_topk_dev")
        return out[: found.value]

    def grow_ucb_argmax(self, bounds, depth, varsigma, rows=None):
        """Arg-max over the ``grow(depth)`` leaf batch of the box, or over its rows ``[rows[0], rows[1])`` only (index = row
        number in the full batch either way)."""
        bounds = np.ascontiguousarray(bounds, dtype=np.float64)
        out = np.empty(4)
        if rows is None:
            _check(self._lib, self._lib.gpso_grow_ucb_argmax(self._h, _dptr(bounds), bounds.shape[0], int(depth), float(varsigma),
                                                             _dptr(out)), "gpso_grow_ucb_argmax")
        else:
            _check(self._lib, self._lib.gpso_grow_ucb_argmax_range(self._h, _dptr(bounds), bounds.shape[0], int(depth), float(varsigma),
                                                                   int(rows[0]), int(rows[1]), _dptr(out)), "gpso_grow_ucb_argmax_range")
        return int(out[0]), float(out[1]), float(out[2]), float(out[3])

    # -- device-pointer variants (benchmarks, multi-GPU sharding): pointers are ints (e.g. torch.Tensor.data_ptr()) -----
    def predict_y_dev(self, xc_ptr, m, mean_ptr, var_ptr, stream=0):
        _check(self._lib, self._lib.gpso_predict_y_dev(self._h, xc_ptr, m, mean_ptr, var_ptr, stream), "gpso_predict_y_dev")

    def predict_f_cov_dev(self, xc_ptr, m, mean_ptr, cov_ptr, stream=0):
        _check(self._lib, self._lib.gpso_predict_f_cov_dev(self._h, xc_ptr, m, mean_ptr, cov_ptr, stream), "gpso_predict_f_cov_dev")

    def predict_f_samples_dev(self, xc_ptr, m, s, jitter, z_ptr, out_ptr, stream=0):
        _check(self._lib, self._lib.gpso_predict_f_samples_dev(self._h, xc_ptr, m, int(s), float(jitter), z_ptr, out_ptr, stream),
               "gpso_predict_f_samples_dev")

    def ucb_argmax_dev(self, xc_ptr, m, varsigma, stream=0):
        out = np.empty(4)
        _check(self._lib, self._lib.gpso_ucb_argmax_dev(self._h, xc_ptr, m, float(varsigma), _dptr(out), stream),
               "gpso_ucb_argmax_dev")
        return int(out[0]), float(out[1]), float(out[2]), float(out[3])

    def state_bytes(self, n=None, d=None):
        v = ctypes.c_int64()
        _check(self._lib, self._lib.gpso_state_bytes(self._h, n or self.N, d or self.d, ctypes.byref(v)), "gpso_state_bytes")
        return int(v.value)

    def export_state_dev(self, dst_ptr, nbytes, stream=0):
        _check(self._lib, self._lib.gpso_export_state_dev(self._h, dst_ptr, nbytes, stream), "gpso_export_state_dev")

    def import_state_dev(self, src_ptr, nbytes, n, d, stream=0):
        self.factorized = False
        _check(self._lib, self._lib.gpso_import_state_dev(self._h, src_ptr, nbytes, n, d, stream), "gpso_import_state_dev")
        self.N, self.d = n, d
        self.factorized = True

    # -- introspection ------------------------------------------------------------------------------------------------
    def launch_count(self):
        return int(self._lib.gpso_launch_count(self._h))

    def last_timing_ms(self):
        out = np.zeros(4)
        _check(self._lib, self._lib.gpso_last_timing(self._h, _dptr(out)), "gpso_last_timing")
        return out

    def set_profile(self, enabled=True):
        """True/1: per-stage events (windows run in order); 2: timeline trace with the stream overlap kept; 0 off."""
        _check(self._lib, self._lib.gpso_set_profile(self._h, int(enabled)), "gpso_set_profile")

    def trace(self):
        """Timeline of the last scoring call after ``set_profile(2)``: array of (tag, window, ms) rows."""
        n = int(self._lib.gpso_debug_trace(self._h, None, 0))
        out = np.zeros(max(n, 1))
        self._lib.gpso_debug_trace(self._h, _dptr(out), n)
        return out[:n].reshape(-1, 3)

    def last_windows(self):
        return int(self._lib.gpso_last_windows(self._h))

    def set_predict_mode(self, mode=0, slices=0):
        """0 automatic, 1 FP64 DMMA, 2 int8 tcgen05 (``slices`` 8-bit digits per operand, 0 = automatic)."""
        self.factorized = False
        _check(self._lib, self._lib.gpso_set_predict_mode(self._h, int(mode), int(slices)), "gpso_set_predict_mode")

    def set_kinv_mode(self, mode=0):
        """K_y^-1 = L^-T L^-1 of the gradient: 0 automatic, 1 FP64 DMMA tiles, 2 int8 tcgen05 (54-bit fixed point)."""
        self.factorized = False
        _check(self._lib, self._lib.gpso_set_kinv_mode(self._h, int(mode)), "gpso_set_kinv_mode")

    def set_l2_window(self, enabled=True):
        """int8 engine: persisting-L2 access window over the digit tiles of L^-1 (default on)."""
        self.factorized = False
        _check(self._lib, self._lib.gpso_set_l2_window(self._h, int(bool(enabled))), "gpso_set_l2_window")

    def set_inverse_mode(self, mode=0):
        """Recursive-doubling L^-1: 0 automatic, 1 FP64 DMMA tile tasks, 2 int8 tcgen05 (62-bit fixed point)."""
        self.factorized = False
        _check(self._lib, self._lib.gpso_set_inverse_mode(self._h, int(mode)), "gpso_set_inverse_mode")

    def set_factor_mode(self, persistent=True, hybrid=None):
        """Cholesky schedule: persistent dataflow kernel (default) or one launch per step.  ``hybrid``: None = automatic
        (matrices above 4096 rows are split recursively: FP64 leaves, int8 tensor-core panels and Schur complements),
        False = always one persistent FP64 kernel, True = split down to leaves of two tiles (tests)."""
        self.factorized = False
        mode = 0 if not persistent else (1 if hybrid is None else (3 if hybrid else 2))
        _check(self._lib, self._lib.gpso_set_factor_mode(self._h, mode), "gpso_set_factor_mode")

    def factor_info(self):
        """Schedule of the last factorisation: {"schedule": "stepwise" | "persistent" | "hybrid", "nodes": inner nodes}."""
        out = (ctypes.c_int * 2)()
        _check(self._lib, self._lib.gpso_factor_info(self._h, out), "gpso_factor_info")
        return {"schedule": ("stepwise", "persistent", "hybrid")[out[0]], "nodes": int(out[1])}

    def set_overlap(self, enabled=True):
        _check(self._lib, self._lib.gpso_set_overlap(self._h, int(bool(enabled))), "gpso_set_overlap")

    def predict_info(self):
        out = np.zeros(3)
        _check(self._lib, self._lib.gpso_predict_info(self._h, _dptr(out)), "gpso_predict_info")
        return {"engine": "int8-tcgen05" if out[0] == 2 else "fp64-dmma", "slices": int(out[1]), "error_estimate_over_tol": float(out[2])}

    def set_screen_mode(self, mode=1):
        """Screen-and-refine arg-max: 0 off, 1 automatic (default), 2..4 forced screening digits (triangular product), 5 mean-bound
        level first, 6 forced 2 digits with all digit pairs; results are bit-identical."""
        self.factorized = False
        _check(self._lib, self._lib.gpso_set_screen_mode(self._h, int(mode)), "gpso_set_screen_mode")

    def screened_values(self, count):
        """Screened UCB (or mean, bound level) of the first ``count`` candidates of the last screened call (tests)."""
        out = np.empty(int(count))
        _check(self._lib, self._lib.gpso_debug_fetch(self._h, 5, _dptr(out), out.size), "gpso_debug_fetch")
        return out

    def screen_info(self):
        out = np.zeros(12)
        _check(self._lib, self._lib.gpso_screen_info(self._h, _dptr(out)), "gpso_screen_info")
        path = {0: "unscreened", 1: "screened", 2: "full pass (too many survivors)", 3: "full pass (bound check failed)",
                4: "mean-bound"}[int(out[0])]
        return {"path": path, "digits": int(out[1]), "survivors": int(out[2]), "error_bound": float(out[3]),
                "max_observed_deviation": float(out[4]), "best_screened_ucb": float(out[5]), "screen_windows": int(out[6]),
                "screen_product_ms": float(out[7]), "refine_windows": int(out[8]), "e_var": float(out[9]), "e_mean": float(out[10]),
                "all_pairs": bool(out[11] == 1.0 and int(out[0]) != 4)}

    def set_window(self, candidates):
        _check(self._lib, self._lib.gpso_set_window(self._h, int(candidates)), "gpso_set_window")

    def debug_fetch(self, which):
        n = self.N
        out = np.empty(n if which == 3 else n * n)
        _check(self._lib, self._lib.gpso_debug_fetch(self._h, which, _dptr(out), out.size), "gpso_debug_fetch")
        return out if which == 3 else out.reshape(n, n)

    def close(self):
        if getattr(self, "_h", None):
            self._lib.gpso_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class CudaBackend:
    """Factory of sessions on one GPU plus the handle-free entry points (leaf generation)."""

    name = "cuda-sm100a"

    def __init__(self, device=None):
        global _cuda_touched
        self._lib = load_library()
        _cuda_touched = True
        n = self._lib.gpso_device_count()
        if n <= 0:
            raise GpsoBackendError(
                "no CUDA device visible: pygpso_b200 runs its surrogate on a B200 GPU and has no CPU fallback "
                f"({self._lib.gpso_last_error().decode('utf-8', 'replace')})"
            )
        self.device = default_device() if device is None else int(device)

    def open_session(self, kernel, n_lengthscales, has_mean, components=None):
        return CudaSession(self._lib, self.device, kernel, n_lengthscales, has_mean, components)

    def trim_pool(self):
        """Give the device memory cached from closed sessions back to the driver; returns the number of bytes released."""
        before = ctypes.c_int64(0)
        _check(self._lib, self._lib.gpso_trim_pool(self.device, ctypes.byref(before)), "gpso_trim_pool")
        return int(before.value)

    def probe_peaks(self):
        """Pipe peaks of this GPU measured now: int8 tensor TOP/s, FP64 DMMA TFLOP/s, L2 -> shared memory GB/s."""
        out = np.zeros(4)
        _check(self._lib, self._lib.gpso_probe_peaks(self.device, _dptr(out)), "gpso_probe_peaks")
        return {"int8_tops": float(out[0]), "fp64_tflops": float(out[1]), "l2_to_smem_gbs": float(out[2]), "sms": int(out[3])}

    def grow_count(self, depth):
        return int(self._lib.gpso_grow_count(int(depth)))

    def grow_leaves(self, bounds, depth):
        """``LeafNode.grow(depth)`` coordinates for the box ``bounds[d,2]``, generated on the GPU, returned as numpy."""
        bounds = np.ascontiguousarray(bounds, dtype=np.float64)
        rows = self.grow_count(depth)
        if rows <= 0:
            raise ValueError(f"bad depth {depth}")
        out = np.empty((rows, bounds.shape[0]))
        _check(self._lib, self._lib.gpso_grow_leaves_host(self.device, _dptr(bounds), bounds.shape[0], int(depth), _dptr(out)),
               "gpso_grow_leaves_host")
        return out

    def grow_leaves_dev(self, bounds, depth, out_ptr, stream=0):
        bounds = np.ascontiguousarray(bounds, dtype=np.float64)
        _check(self._lib, self._lib.gpso_grow_leaves_dev(self.device, _dptr(bounds), bounds.shape[0], int(depth), out_ptr, stream),
               "gpso_grow_leaves_dev")


_default = None


def default_backend():
    """The process-wide CUDA backend (created on first use; raises GpsoBackendError when unavailable)."""
    global _default
    if _default is None:
        _default = CudaBackend()
    return _default


def reset_default_backend():
    global _default
    _default = None
