"""
Periodic kernel (gpflow.kernels.Periodic with a SquaredExponential or RationalQuadratic base) without a GPU: the oracle's
closed-form gradient, the embedding identity the device relies on, periodicity and the long-period limit, the model layer
(packing and leaf names, frozen period, persistence, refusals, an optimiser run through the checker backend), the fp32 screening
covariance on the embedded rows against the contract of the screening error model, and the C argument checks that need no device.
"""
import ctypes
import json

import numpy as np
import pytest

from pygpso_b200 import GPRSurrogate, backend, gpmodel
from tests import periodic_oracle as pe
from tests import rq_oracle as rq
from tests import sum_oracle as so
from tests.screen_oracle import ScreenOracle
from tests.test_oracle_goldens import make_optimiser, seeded_points
from tests.test_sum_kernel import synthetic

VARSIGMA = 1.96


def hyper(base, ls, p, mean=None, var=0.9, noise=2e-3):
    return pe.PeriodicHyper(base, ls, var, p, noise, alpha=1.7 if base == rq.KERNEL else None, mean=mean)


# ---- oracle ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("base", pe.BASES)
@pytest.mark.parametrize("ls,p", [(0.4, 0.7), ([0.3, 0.6, 0.5], 0.8), (0.5, [0.4, 0.9, 1.3]), ([0.3, 0.6, 0.5], [0.4, 0.9, 1.3])],
                         ids=["scalar", "ard_ls", "ard_period", "ard_both"])
@pytest.mark.parametrize("mean_id", [0, 1, 2])
def test_oracle_gradient_matches_finite_differences(base, ls, p, mean_id):
    N, d = 30, 3
    X, y = synthetic(N, d)
    mean = {0: None, 1: 0.2, 2: (np.array([0.3, -0.5, 0.2]), 0.1)}[mean_id]
    h = hyper(base, ls, p, mean)
    n_ls, n_p = h.lengthscales.size, h.period.size
    u = h.pack()
    f, g = pe.neg_lml_and_grad(base, n_ls, n_p, X, y, u, mean_id)
    assert f == pytest.approx(-pe.lml(pe.PeriodicHyper.unpack(base, n_ls, n_p, u, mean_id, d), X, y), rel=1e-12)
    assert g.size == u.size == h.theta().size
    for i in range(u.size):
        e = np.zeros_like(u)
        e[i] = 1e-6
        fd = (pe.neg_lml_and_grad(base, n_ls, n_p, X, y, u + e, mean_id)[0]
              - pe.neg_lml_and_grad(base, n_ls, n_p, X, y, u - e, mean_id)[0]) / 2e-6
        assert g[i] == pytest.approx(fd, rel=2e-5, abs=2e-6), i


@pytest.mark.parametrize("p", [0.05, 0.1, 0.37, 1.0, 3.3, 10.0])
@pytest.mark.parametrize("ls", [0.05, 1.0, 7.0])
def test_embedding_r2_is_the_sine_form(p, ls):
    rng = np.random.default_rng(7)
    X = rng.random((80, 4))
    h = hyper("SquaredExponential", ls, p)
    r2_sin = pe.r2_parts(h, X, None).sum(-1)
    assert np.max(np.abs(pe.embedded_r2(h, X, None) - r2_sin)) <= 1e-13 / ls ** 2


@pytest.mark.parametrize("base", pe.BASES)
def test_shift_by_one_period_leaves_the_kernel(base):
    rng = np.random.default_rng(2)
    h = hyper(base, [0.3, 0.7], [0.6, 1.9])
    X = rng.random((20, 2))
    for j in range(2):
        Xp = X.copy()
        Xp[:, j] += h.period[j]
        np.testing.assert_allclose(np.diag(pe.kern(h, X, Xp)), h.variance, rtol=0, atol=1e-13)


@pytest.mark.parametrize("base", pe.BASES)
def test_long_period_limit_is_the_base_kernel(base):
    """p -> inf with l' = l p / pi fixed: sin(pi delta / p) / l -> delta / l'."""
    rng = np.random.default_rng(4)
    X, X2 = rng.random((15, 2)), rng.random((12, 2))
    lprime = np.array([0.4, 0.8])
    p = 1e5
    h = hyper(base, lprime * np.pi / p, p)
    r2 = np.sum(np.square((X[:, None, :] - X2[None, :, :]) / lprime), axis=-1)
    ref = h.variance * np.exp(-0.5 * r2) if base == "SquaredExponential" else rq.k_of_r2(r2, h.variance, h.alpha)
    np.testing.assert_allclose(pe.kern(h, X, X2), ref, rtol=1e-8, atol=0)


# ---- model layer ------------------------------------------------------------------------------------------------------
def model(kernel, mean=None, d=2, N=40):
    X, y = synthetic(N, d)
    return gpmodel.GPR((X, y), kernel, mean_function=mean, noise_variance=1e-3, backend=pe.PeriodicOracleBackend())


def test_packing_order_and_leaf_names():
    k = gpmodel.Periodic(gpmodel.RationalQuadratic(variance=0.3, lengthscales=[0.5, 0.6], alpha=2.0), period=[0.7, 1.1])
    m = model(k, gpmodel.Linear(np.array([[0.3], [-0.2]]), np.array([0.1])))
    assert np.array_equal(m._theta(), [2.0, 0.5, 0.6, 0.3, 0.7, 1.1, 1e-3, 0.3, -0.2, 0.1])
    names = list(gpmodel.parameter_dict(m))
    assert names == [".kernel.base_kernel.alpha", ".kernel.base_kernel.lengthscales", ".kernel.base_kernel.variance",
                     ".kernel.period", ".likelihood.variance", ".mean_function.A", ".mean_function.b"]
    gpmodel.multiple_assign(m, {".kernel.period": [0.9, 1.4], ".kernel.base_kernel.variance": 0.25})
    assert list(m._theta()[3:6]) == [0.25, 0.9, 1.4]
    summary = gpmodel.tabulate_module_summary(m)
    assert "GPR.kernel.period" in summary and "GPR.kernel.base_kernel.alpha" in summary
    assert type(m._session) is pe.PeriodicOracleSession
    assert (m._session.base, m._session.n_ls, m._session.n_p) == ("RationalQuadratic", 2, 2)
    assert gpmodel.kernels.Periodic is gpmodel.Periodic


def test_training_loss_and_predict_are_the_oracle():
    m = model(gpmodel.Periodic(gpmodel.SquaredExponential(lengthscales=0.4), period=[0.5, 0.8]), gpmodel.Constant(0.1))
    f, g = m.neg_log_marginal_likelihood_and_grad(m._pack())
    f_ref, g_ref = pe.neg_lml_and_grad("SquaredExponential", 1, 2, *m.data, m._pack(), 1)
    assert f == f_ref and np.array_equal(g, g_ref)
    xc = np.random.default_rng(0).random((7, 2))
    mean, var = m.predict_y(xc)
    mf, cov = m.predict_f(xc, full_cov=True)
    np.testing.assert_allclose(mf[:, 0], mean[:, 0], rtol=1e-12)
    np.testing.assert_allclose(np.diag(cov[0]), var[:, 0] - 1e-3, rtol=1e-10, atol=1e-14)


def test_frozen_period_is_left_alone():
    k = gpmodel.Periodic(gpmodel.SquaredExponential(lengthscales=0.5), period=0.6)
    m = model(k, gpmodel.Constant(0.0))
    k.period.trainable = False
    before = k.period.numpy().copy()
    others = [p.numpy().copy() for p in (k.base_kernel.lengthscales, k.base_kernel.variance)]
    res = gpmodel.Scipy().minimize(m.training_loss, m.trainable_variables)
    assert res.success or res.nit > 0
    assert k.period.numpy() == pytest.approx(before, rel=1e-15)
    assert any(not np.array_equal(p.numpy(), o) for p, o in zip((k.base_kernel.lengthscales, k.base_kernel.variance), others))


def _trained_surrogate(kernel, backend_):
    surr = GPRSurrogate(gp_kernel=kernel, gp_meanf=gpmodel.Constant(0.0), points=seeded_points(), backend=backend_)
    x, y = surr.current_training_data
    surr._gp_train(x=x, y=y[:, np.newaxis])
    return surr, x


@pytest.mark.parametrize("base", pe.BASES)
def test_save_from_saved_round_trips_every_parameter(tmp_path, base):
    kernel = gpmodel.Periodic(getattr(gpmodel, base)(lengthscales=[0.5, 0.4]), period=0.9)
    surr = GPRSurrogate(gp_kernel=kernel, gp_meanf=gpmodel.Constant(0.0), points=seeded_points(), backend=pe.PeriodicOracleBackend())
    x, y = surr.current_training_data
    # fitted values without a fit: on these few points the optimum has the noise at its floor, which no model can be loaded with
    surr.gpflow_model = gpmodel.GPR((x, y[:, np.newaxis]), kernel, gpmodel.Constant(0.0), surr.gp_lik_sigma, surr.backend)
    rng = np.random.default_rng(9)
    gpmodel.multiple_assign(surr.gpflow_model, {k: 0.2 + rng.random(np.shape(v)) for k, v in gpmodel.parameter_dict(surr.gpflow_model).items()})
    surr.save(str(tmp_path / "s"))
    with open(tmp_path / "s" / GPRSurrogate.GPR_INFO) as fh:
        info = json.load(fh)
    assert info["gpr_kernel"] == "Periodic" and info["gpr_kernel_shape"] == [2]
    assert info["gpr_kernel_periodic"] == [base, []]
    loaded = GPRSurrogate.from_saved(str(tmp_path / "s"), backend=pe.PeriodicOracleBackend())
    lk = loaded.gpflow_model.kernel
    assert isinstance(lk, gpmodel.Periodic) and type(lk.base_kernel) is getattr(gpmodel, base)
    assert loaded.gpflow_model._theta().tobytes() == surr.gpflow_model._theta().tobytes()
    p, q = surr.gpflow_model.predict_y(x), loaded.gpflow_model.predict_y(x)
    assert np.array_equal(p[0], q[0]) and np.array_equal(p[1], q[1])


def test_non_periodic_save_files_are_unchanged(tmp_path):
    """A bare kernel's saved info is the text the previous release wrote, byte for byte."""
    from tests.oracle_backend import OracleBackend

    surr, _ = _trained_surrogate(gpmodel.Matern52(lengthscales=0.25), OracleBackend())
    surr.save(str(tmp_path / "s"))
    with open(tmp_path / "s" / GPRSurrogate.GPR_INFO) as fh:
        text = fh.read()
    assert text == json.dumps({
        "gpr_kernel": "Matern52", "gpr_kernel_shape": [], "gpr_meanf": "Constant", "gpr_meanf_shape": [],
        "gp_varsigma": surr.gp_varsigma, "gp_likelihood": surr.gp_lik_sigma, "optimiser": ["Scipy"],
    })


def test_optimiser_runs_with_the_periodic_checker_backend():
    from tests.conftest import paper_objective

    opt = make_optimiser(backend=pe.PeriodicOracleBackend(), depth=3, budget=40)
    opt.gp_surr.gp_kernel = gpmodel.Periodic(gpmodel.SquaredExponential(lengthscales=0.5), period=0.8)
    best = opt.run(paper_objective)
    assert isinstance(opt.gp_surr.gpflow_model.kernel, gpmodel.Periodic)
    assert type(opt.gp_surr.gpflow_model._session) is pe.PeriodicOracleSession
    assert opt.n_eval_counter >= 40 and np.isfinite(best.score_mu)


# ---- refusals ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("base", ["Matern12", "Matern32", "Matern52"])
def test_matern_base_is_refused(base):
    with pytest.raises(TypeError, match="SquaredExponential or RationalQuadratic"):
        gpmodel.Periodic(getattr(gpmodel, base)())


@pytest.mark.parametrize("build", [lambda: gpmodel.SquaredExponential() + gpmodel.Matern12(),
                                   lambda: gpmodel.SquaredExponential() * gpmodel.RationalQuadratic(),
                                   lambda: gpmodel.Periodic(gpmodel.SquaredExponential())])
def test_combined_base_is_refused(build):
    with pytest.raises(TypeError, match="IsotropicStationary"):
        gpmodel.Periodic(build())


# ---- periodic terms inside sums and products -----------------------------------------------------------------------------
SPECS = {
    "se*periodic(se)": ("Product", [("SquaredExponential", 1), ("Periodic", 1, "SquaredExponential", 3)]),
    "m52+periodic(rq)": ("Sum", [("Matern52", 3), ("Periodic", 3, rq.KERNEL, 3)]),
    "periodic+periodic*": ("Product", [("Periodic", 1, rq.KERNEL, 1), ("Matern12", 1), ("Periodic", 3, "SquaredExponential", 1)]),
}


def composite(spec_key, d=3, mean=None, noise=2e-3):
    kind, specs = SPECS[spec_key]
    comps = []
    for i, s in enumerate(specs):
        ls = list(0.4 + 0.1 * np.arange(d) + 0.05 * i) if s[1] > 1 else 0.5 + 0.1 * i
        if s[0] == "Periodic":
            p = list(0.6 + 0.3 * np.arange(d)) if s[3] > 1 else 0.8
            comps.append(pe.PeriodicHyper(s[2], ls, 0.9 + 0.2 * i, p, 1.0, alpha=1.4 if s[2] == rq.KERNEL else None))
        else:
            comps.append(so.Comp(s[0], ls, 0.7 + 0.2 * i, 1.3 if s[0] == rq.KERNEL else None))
    return kind, specs, pe.CompositeHyper(kind, comps, noise, mean)


@pytest.mark.parametrize("key", sorted(SPECS))
@pytest.mark.parametrize("mean_id", [0, 1, 2])
def test_composite_oracle_gradient_matches_finite_differences(key, mean_id):
    N, d = 25, 3
    X, y = synthetic(N, d)
    kind, specs, h = composite(key, d, {0: None, 1: 0.2, 2: (np.array([0.3, -0.5, 0.2]), 0.1)}[mean_id])
    u = h.pack()
    f, g = pe.composite_neg_lml_and_grad(kind, specs, X, y, u, mean_id)
    assert f == pytest.approx(-pe.composite_lml(pe.CompositeHyper.unpack(kind, specs, u, mean_id, d), X, y), rel=1e-12)
    assert g.size == u.size == h.theta().size
    for i in range(u.size):
        e = np.zeros_like(u)
        e[i] = 1e-6
        fd = (pe.composite_neg_lml_and_grad(kind, specs, X, y, u + e, mean_id)[0]
              - pe.composite_neg_lml_and_grad(kind, specs, X, y, u - e, mean_id)[0]) / 2e-6
        assert g[i] == pytest.approx(fd, rel=2e-5, abs=2e-6), (i, g[i], fd)


@pytest.mark.parametrize("kind", ["Sum", "Product"])
def test_one_term_combination_of_a_periodic_is_the_bare_kernel(kind):
    X, y = synthetic(20, 2)
    h = pe.PeriodicHyper(rq.KERNEL, [0.4, 0.7], 1.1, [0.6, 0.9], 2e-3, alpha=1.5, mean=0.1)
    c = pe.CompositeHyper(kind, [h], 2e-3, 0.1)
    assert np.array_equal(pe.composite_kern(c, X, None), pe.kern(h, X, None))
    u = c.pack()
    f1, g1 = pe.composite_neg_lml_and_grad(kind, [("Periodic", 2, rq.KERNEL, 2)], X, y, u, 1)
    f2, g2 = pe.neg_lml_and_grad(rq.KERNEL, 2, 2, X, y, u, 1)
    assert f1 == f2 and np.allclose(g1, g2, rtol=1e-12, atol=0)


def test_periodic_terms_pack_and_name_like_gpflow():
    k0 = gpmodel.Matern52(variance=0.8, lengthscales=[0.5, 0.6])
    k1 = gpmodel.Periodic(gpmodel.RationalQuadratic(variance=0.3, lengthscales=0.2, alpha=2.0), period=[0.7, 1.1])
    m = model(k0 + k1, gpmodel.Constant(0.1))
    assert np.array_equal(m._theta(), [0.5, 0.6, 0.8, 2.0, 0.2, 0.3, 0.7, 1.1, 1e-3, 0.1])
    assert list(gpmodel.parameter_dict(m)) == [
        ".kernel.kernels[0].lengthscales", ".kernel.kernels[0].variance", ".kernel.kernels[1].base_kernel.alpha",
        ".kernel.kernels[1].base_kernel.lengthscales", ".kernel.kernels[1].base_kernel.variance", ".kernel.kernels[1].period",
        ".likelihood.variance", ".mean_function.c"]
    assert type(m._session) is pe.CompositeOracleSession
    assert m._session.specs == [("Matern52", 2), ("Periodic", 1, rq.KERNEL, 2)]
    f, g = m.neg_log_marginal_likelihood_and_grad(m._pack())
    f_ref, g_ref = pe.composite_neg_lml_and_grad("Sum", m._session.specs, *m.data, m._pack(), 1)
    assert f == f_ref and np.array_equal(g, g_ref)
    p = gpmodel.SquaredExponential() * gpmodel.Periodic(gpmodel.SquaredExponential())   # the locally periodic kernel
    assert type(model(p)._session) is pe.CompositeOracleSession


def test_same_base_object_twice_is_refused():
    b = gpmodel.SquaredExponential()
    with pytest.raises(ValueError, match="appears twice"):
        gpmodel.Periodic(b) + b
    with pytest.raises(ValueError, match="appears twice"):
        gpmodel.Periodic(b) * gpmodel.Periodic(b)


@pytest.mark.parametrize("build", [lambda p, k: p * k + k.__class__(), lambda p, k: (p + k) * gpmodel.Matern12()])
def test_sums_of_products_with_periodic_terms_are_refused(build):
    with pytest.raises(TypeError, match="sums of products"):
        model(build(gpmodel.Periodic(gpmodel.SquaredExponential()), gpmodel.Matern52()))


def test_save_from_saved_round_trips_a_periodic_component(tmp_path):
    kernel = gpmodel.Matern52(lengthscales=[0.5, 0.4]) * gpmodel.Periodic(gpmodel.RationalQuadratic(lengthscales=0.3), period=[0.6, 0.9])
    surr = GPRSurrogate(gp_kernel=kernel, gp_meanf=gpmodel.Constant(0.0), points=seeded_points(), backend=pe.PeriodicOracleBackend())
    x, y = surr.current_training_data
    surr.gpflow_model = gpmodel.GPR((x, y[:, np.newaxis]), kernel, gpmodel.Constant(0.0), surr.gp_lik_sigma, surr.backend)
    rng = np.random.default_rng(11)
    gpmodel.multiple_assign(surr.gpflow_model, {k: 0.2 + rng.random(np.shape(v)) for k, v in gpmodel.parameter_dict(surr.gpflow_model).items()})
    surr.save(str(tmp_path / "s"))
    with open(tmp_path / "s" / GPRSurrogate.GPR_INFO) as fh:
        info = json.load(fh)
    assert info["gpr_kernel"] == "Product"
    assert info["gpr_kernel_components"] == [["Matern52", [2]], ["Periodic", [], "RationalQuadratic", [2]]]
    loaded = GPRSurrogate.from_saved(str(tmp_path / "s"), backend=pe.PeriodicOracleBackend())
    lk = loaded.gpflow_model.kernel
    assert isinstance(lk, gpmodel.Product) and isinstance(lk.kernels[1], gpmodel.Periodic)
    assert loaded.gpflow_model._theta().tobytes() == surr.gpflow_model._theta().tobytes()


def test_create_combination_rejects_bad_arguments():
    lib = backend.load_library()
    h = ctypes.c_void_p()

    def create(kind, ids, ards, bases, pards, mean=1):
        n = len(ids)
        arr = lambda v: (ctypes.c_int * max(n, 1))(*v)  # noqa: E731
        return lib.gpso_create_combination(0, kind, n, arr(ids), arr(ards), arr(bases), arr(pards), mean, ctypes.byref(h))

    assert create(7, [3, 7], [0, 0], [0, 3], [0, 0]) == -1          # a periodic kernel is not a kind of combination
    assert b"kind" in lib.gpso_last_error()
    assert create(5, [3, 7], [0, 0], [0, 2], [0, 0]) == -1           # a Matern base
    assert b"SquaredExponential or RationalQuadratic" in lib.gpso_last_error()
    assert create(6, [3, 7], [0, 0], [0, 3], [0, 2]) == -1           # period ARD flag
    assert b"ard" in lib.gpso_last_error()
    assert create(6, [3, 8], [0, 0], [0, 3], [0, 0]) == -1
    assert b"kernel id" in lib.gpso_last_error()
    assert create(5, [], [], [], []) == -1
    ids, ards = (ctypes.c_int * 2)(3, 7), (ctypes.c_int * 2)(0, 0)
    for create_old in (lib.gpso_create_sum, lib.gpso_create_product):   # they keep refusing the periodic id
        assert create_old(0, 2, ids, ards, 1, ctypes.byref(h)) == -1
        assert b"kernel id" in lib.gpso_last_error()
    assert not h.value


def test_wrong_ard_lengths_are_refused():
    with pytest.raises(ValueError, match="ARD period"):
        model(gpmodel.Periodic(gpmodel.SquaredExponential(), period=[0.5, 0.6, 0.7]))
    with pytest.raises(ValueError, match="ARD lengthscales"):
        model(gpmodel.Periodic(gpmodel.SquaredExponential(lengthscales=[0.5, 0.6, 0.7]), period=0.5))
    with pytest.raises(ValueError, match="must be > 0"):
        gpmodel.Periodic(gpmodel.SquaredExponential(), period=0.0)


def test_create_periodic_rejects_bad_arguments():
    lib = backend.load_library()
    h = ctypes.c_void_p()
    for base in (0, 1, 2, 5, 6, 7):   # Matern bases, a sum, a product or a periodic kernel
        assert lib.gpso_create_periodic(0, base, 0, 0, 1, ctypes.byref(h)) == -1   # GPSO_E_BADARG before any CUDA call
        assert b"SquaredExponential or RationalQuadratic" in lib.gpso_last_error()
    assert lib.gpso_create_periodic(0, 3, 2, 0, 1, ctypes.byref(h)) == -1
    assert lib.gpso_create_periodic(0, 3, 0, 2, 1, ctypes.byref(h)) == -1
    assert b"ard" in lib.gpso_last_error()
    assert lib.gpso_create_periodic(0, 4, 0, 0, 3, ctypes.byref(h)) == -1
    assert b"mean id" in lib.gpso_last_error()
    assert lib.gpso_create_periodic(0, 3, 0, 0, 1, None) == -1
    assert lib.gpso_create(0, 7, 0, 1, ctypes.byref(h)) == -1   # the periodic id has a base: gpso_create_periodic
    assert not h.value


# ---- fp32 screening covariance on the embedded rows: |k32 - k64| <= 2e-6 variance ----------------------------------------
SCALES = [0.05, 0.2, 1.0, 3.0, 10.0]


@pytest.mark.parametrize("base,alpha", [("SquaredExponential", None)] + [(rq.KERNEL, a) for a in (1e-2, 1.0, 1e2, 1e6)])
@pytest.mark.parametrize("d", [1, 4, 32])
def test_cov32_of_periodic_kernels_within_the_screen_contract(base, alpha, d):
    rng = np.random.default_rng(11 + d)
    Xa = rng.random((120, d))
    Xb = np.vstack([rng.random((150, d)), Xa[:30] + 1e-4 * rng.standard_normal((30, d)), Xa[:5]])
    worst = 0.0
    for ls in SCALES:
        for p in SCALES:
            # the lengthscale scaled with sqrt(d) as well, so that the long-range part of the kernel is exercised at every d
            for lsd in (ls, ls * np.sqrt(d)):
                h = pe.PeriodicHyper(base, lsd, 1.3, p, 1e-3, alpha=alpha)
                k32 = pe.cov32(h, Xa, Xb).astype(np.float64)
                worst = max(worst, np.max(np.abs(k32 - pe.kern(h, Xa, Xb))) / h.variance)
    # half the contract: MUFU.EX2 / LG2 and __fdividef are not emulated (a few ulp each)
    assert worst <= 2e-6 / 2.0, worst


@pytest.mark.parametrize("base", pe.BASES)
@pytest.mark.parametrize("S,full", [(2, True), (3, False), (4, False)])
def test_screen_error_bound_holds_on_embedded_rows(base, S, full):
    """The screening pass of a periodic kernel is its base family's on the embedded rows at unit lengthscale: the device-order
    emulation of that pass stays within E / 8 of the fp64 posterior, with E from the C error model."""
    rng = np.random.default_rng(20240517)
    N, d = 512, 3
    X = rng.random((N, d))
    y = (np.sin(6.0 * X.sum(axis=1)) + 0.01 * rng.standard_normal(N))[:, None]
    h = pe.PeriodicHyper(base, [0.4, 0.7, 0.5], 1.1, [0.3, 0.9, 2.0], 1e-3, alpha=1.5 if base == rq.KERNEL else None, mean=0.1)
    L = np.linalg.cholesky(pe.kern(h, X, None) + h.noise_variance * np.eye(N))
    Linv = np.linalg.solve(L, np.eye(N))
    alpha = Linv.T @ (Linv @ (y[:, 0] - 0.1))
    so = ScreenOracle(base, pe.embed(X, h.lengthscales, h.period), Linv, alpha, 1.0, h.variance, h.noise_variance, 0.1,
                      rq_alpha=h.alpha)
    Xc = np.vstack([rng.random((1500, d)), X[:100] + 1e-5 * rng.standard_normal((100, d))])
    mean_s, var_s = so.screen(pe.embed(Xc, h.lengthscales, h.period), [(S, full)])[(S, full)]
    mean, var = pe.predict_y(h, X, y, Xc)
    out = (ctypes.c_double * 3)()
    lib = backend.load_library()
    assert lib.gpso_debug_screen_bound(N, h.variance, h.noise_variance, (ctypes.c_double * 5)(*so.fit5), S, int(full), VARSIGMA,
                                       out) == 0
    E, e_var, e_mean = tuple(out)
    assert np.abs(var_s - var[:, 0]).max() <= e_var / 8.0
    assert np.abs(mean_s - mean[:, 0]).max() <= e_mean / 8.0
    assert np.abs((mean_s + VARSIGMA * var_s) - (mean[:, 0] + VARSIGMA * var[:, 0])).max() <= E / 8.0
