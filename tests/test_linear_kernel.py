"""gpflow.kernels.Linear for the GPR model (CPU): the oracle's gradient, construction and refusals, packing, save / load through
the checker backend, an optimiser run, and the C ABI's argument checks."""
import ctypes
import json

import numpy as np
import pytest

from pygpso_b200 import GPRSurrogate, backend, gpmodel
from tests import linear_kernel_oracle as lo
from tests import periodic_oracle as pe
from tests import sum_oracle as so
from tests.test_oracle_goldens import make_optimiser, seeded_points
from tests.test_sum_kernel import synthetic

K = gpmodel.kernels


def model(kernel, mean=None, d=4, N=30):
    X, y = synthetic(N, d)
    return gpmodel.GPR((X, y), kernel, mean_function=mean, noise_variance=1e-3, backend=lo.LinearOracleBackend())


# ---- oracle -----------------------------------------------------------------------------------------------------------
CASES = {
    "bare": ("Sum", [("Linear", 1)], [[0, 1, 2, 3]], [lo.LinearHyper(0.7)]),
    "bare_ard": ("Sum", [("Linear", 4)], [[0, 1, 2, 3]], [lo.LinearHyper([0.5, 0.9, 1.3, 0.4])]),
    "plus_m52": ("Sum", [("Linear", 1), ("Matern52", 1)], [[0, 1, 2, 3]] * 2, [lo.LinearHyper(0.6), so.Comp("Matern52", 0.4, 0.9)]),
    "three_terms": ("Sum", [("Linear", 1), ("Matern52", 3), ("Periodic", 1, "SquaredExponential", 1)], [[0], [1, 2, 3], [3]],
                    [lo.LinearHyper(1.1), so.Comp("Matern52", [0.4, 0.5, 0.7], 0.8),
                     pe.PeriodicHyper("SquaredExponential", 0.6, 0.7, 0.8, 1.0)]),
}


@pytest.mark.parametrize("key", sorted(CASES))
@pytest.mark.parametrize("mean_id", [0, 1, 2])
def test_oracle_gradient_matches_finite_differences(key, mean_id):
    kind, specs, dims, comps = CASES[key]
    X, y = synthetic(25, 4)
    mean = {0: None, 1: 0.2, 2: (np.array([0.3, -0.5, 0.2, 0.1]), 0.1)}[mean_id]
    u = lo.Hyper(kind, comps, 2e-3, mean).pack()
    f, g = lo.neg_lml_and_grad(kind, specs, dims, X, y, u, mean_id)
    assert g.size == u.size
    for i in range(u.size):  # -LML is ~1e3 here (a Linear term fits the data badly): a wider step keeps the cancellation small
        e = np.zeros_like(u)
        e[i] = 1e-4
        fd = (lo.neg_lml_and_grad(kind, specs, dims, X, y, u + e, mean_id)[0]
              - lo.neg_lml_and_grad(kind, specs, dims, X, y, u - e, mean_id)[0]) / 2e-4
        assert g[i] == pytest.approx(fd, rel=2e-5, abs=2e-6), i


def test_oracle_prior_variance_is_the_diagonal():
    X, _ = synthetic(12, 3)
    h = lo.Hyper("Sum", [lo.LinearHyper([0.5, 2.0]), so.Comp("Matern52", 0.4, 0.9)], 1e-3)
    dims = [[0, 2], [0, 1, 2]]
    assert np.allclose(lo.kern_diag(h, dims, X), np.diag(lo.kern(h, dims, X)), rtol=1e-14, atol=0)


# ---- construction -----------------------------------------------------------------------------------------------------
def test_kernels_linear_is_the_kernel_and_top_level_linear_the_mean():
    assert K.Linear is gpmodel.LinearKernel and K.Linear.__name__ == "Linear"
    assert gpmodel.Linear is gpmodel.mean_functions.Linear


def test_construction_and_active_dims():
    k = K.Linear(variance=[0.5, 2.0], active_dims=[3, 1])
    assert k.ard and list(k.active_dims) == [3, 1] and k.parameters == (k.variance,)
    m = model(k)
    assert m._leaf_dims == [[3, 1]]
    assert m._session.leaf_dims == [[3, 1]] and m._session.specs == [("Linear", 2)]
    assert not K.Linear().ard and K.Linear().active_dims == slice(None)


def test_ard_count_follows_the_active_columns():
    with pytest.raises(ValueError, match="ARD variances"):
        model(K.Linear(variance=[1.0, 1.0, 1.0]))
    with pytest.raises(ValueError, match=r"\(2 active\)"):
        model(K.Linear(variance=[1.0, 1.0, 1.0], active_dims=[0, 1]))
    model(K.Linear(variance=np.ones(4)))


def test_refusals():
    with pytest.raises(TypeError, match="Linear kernel cannot be a factor of a Product"):
        model(K.Linear() * K.SquaredExponential())
    with pytest.raises(TypeError, match=r"Periodic\(Linear"):
        K.Periodic(K.Linear())
    with pytest.raises(ValueError, match="1..4"):
        K.Linear() + K.Matern52() + K.Matern52() + K.Matern52() + K.Matern12()


def test_row_budget_counts_a_linear_leafs_columns():
    with pytest.raises(ValueError, match="rows"):
        model(K.Linear(active_dims=list(range(40))) + K.Matern52(active_dims=list(range(25))), d=40)


# ---- packing ----------------------------------------------------------------------------------------------------------
def test_packing_and_leaf_names():
    m = model(K.Linear(variance=0.7), mean=gpmodel.Constant(0.1))
    assert list(gpmodel.parameter_dict(m)) == [".kernel.variance", ".likelihood.variance", ".mean_function.c"]
    assert m._theta().tolist() == pytest.approx([0.7, 1e-3, 0.1])
    k = K.Linear(variance=[0.2, 0.3], active_dims=[0, 1]) + K.Matern52(lengthscales=0.4, variance=0.9, active_dims=[2, 3])
    m = model(k)
    assert list(gpmodel.parameter_dict(m)) == [".kernel.kernels[0].variance", ".kernel.kernels[1].lengthscales",
                                               ".kernel.kernels[1].variance", ".likelihood.variance"]
    assert m._theta().tolist() == pytest.approx([0.2, 0.3, 0.4, 0.9, 1e-3])
    gpmodel.multiple_assign(m, {".kernel.kernels[0].variance": np.array([0.5, 0.6])})
    assert k.kernels[0].variance.numpy().tolist() == [0.5, 0.6]
    assert ".kernel.kernels[0].variance" in gpmodel.tabulate_module_summary(m)


def test_loss_and_predict_are_the_oracle_and_a_frozen_variance_stays():
    k = K.Linear(variance=0.5) + K.Matern52(lengthscales=0.4)
    m = model(k, mean=gpmodel.Constant(0.0))
    X, y = m.data
    k.kernels[0].variance.trainable = False
    before = float(k.kernels[0].variance.numpy())
    gpmodel.Scipy().minimize(m.training_loss, m.trainable_variables, options={"maxiter": 20})
    assert float(k.kernels[0].variance.numpy()) == before
    h = lo.Hyper("Sum", [lo.LinearHyper(before), so.Comp("Matern52", float(k.kernels[1].lengthscales.numpy()),
                                                          float(k.kernels[1].variance.numpy()))],
                 float(m.likelihood.variance.numpy()), float(m.mean_function.c.numpy()))
    dims = [list(range(4))] * 2
    assert m.log_marginal_likelihood() == pytest.approx(lo.lml(h, dims, X, y), rel=1e-12)
    xq = np.linspace(-3, 3, 20)[:, None] * np.ones((1, 4))
    mean, var = m.predict_y(xq)
    rm, rv = lo.predict_y(h, dims, X, y, xq)
    assert np.allclose(mean, rm, rtol=1e-12) and np.allclose(var, rv, rtol=1e-12)


# ---- save / load ------------------------------------------------------------------------------------------------------
def _fitted(kernel):
    surr = GPRSurrogate(gp_kernel=kernel, gp_meanf=gpmodel.Constant(0.0), points=seeded_points(), backend=lo.LinearOracleBackend())
    x, y = surr.current_training_data
    surr.gpflow_model = gpmodel.GPR((x, y[:, np.newaxis]), kernel, gpmodel.Constant(0.0), surr.gp_lik_sigma, surr.backend)
    rng = np.random.default_rng(9)
    gpmodel.multiple_assign(surr.gpflow_model, {k: 0.2 + rng.random(np.shape(v)) for k, v in gpmodel.parameter_dict(surr.gpflow_model).items()})
    return surr, x


@pytest.mark.parametrize("make, kernel_name, shape, comps", [
    (lambda d: K.Linear(), "Linear", [], None),
    (lambda d: K.Linear(variance=np.ones(d)), "Linear", ["d"], None),
    (lambda d: K.Linear(active_dims=[0]) + K.Matern52(active_dims=list(range(1, d))), "Sum", [], [["Linear", []], ["Matern52", []]]),
])
def test_save_from_saved_round_trip(tmp_path, make, kernel_name, shape, comps):
    x_dim = seeded_points()[0].normed_coord.size
    surr, x = _fitted(make(x_dim))
    surr.save(str(tmp_path / "s"))
    with open(tmp_path / "s" / GPRSurrogate.GPR_INFO) as fh:
        info = json.load(fh)
    assert info["gpr_kernel"] == kernel_name
    assert info["gpr_kernel_shape"] == [x_dim if s == "d" else s for s in shape]
    if comps is not None:
        assert info["gpr_kernel_components"] == comps
    loaded = GPRSurrogate.from_saved(str(tmp_path / "s"), backend=lo.LinearOracleBackend())
    assert loaded.gpflow_model._theta().tobytes() == surr.gpflow_model._theta().tobytes()
    p, q = surr.gpflow_model.predict_y(x), loaded.gpflow_model.predict_y(x)
    assert np.array_equal(p[0], q[0]) and np.array_equal(p[1], q[1])


def test_other_kernels_saves_are_unchanged(tmp_path):
    surr, _ = _fitted(gpmodel.Matern52(lengthscales=0.25))
    surr.save(str(tmp_path / "s"))
    with open(tmp_path / "s" / GPRSurrogate.GPR_INFO) as fh:
        text = fh.read()
    assert text == json.dumps({
        "gpr_kernel": "Matern52", "gpr_kernel_shape": [], "gpr_meanf": "Constant", "gpr_meanf_shape": [],
        "gp_varsigma": surr.gp_varsigma, "gp_likelihood": surr.gp_lik_sigma, "optimiser": ["Scipy"],
    })


def test_optimiser_runs_with_the_checker_backend():
    from tests.conftest import paper_objective

    opt = make_optimiser(backend=lo.LinearOracleBackend(), depth=3, budget=40)
    opt.gp_surr.gp_kernel = K.Linear() + K.Matern52(lengthscales=0.5)
    best = opt.run(paper_objective)
    assert opt.gp_surr.gpflow_model._session.specs == [("Linear", 1), ("Matern52", 1)]
    assert opt.n_eval_counter >= 40 and np.isfinite(best.score_mu)


# ---- C argument checks ------------------------------------------------------------------------------------------------
LINEAR = backend.KERNEL_LINEAR


def test_create_refuses_a_bad_ard_flag():
    lib = backend.load_library()
    h = ctypes.c_void_p()
    assert lib.gpso_create(0, LINEAR, 2, 0, ctypes.byref(h)) == -1
    assert b"Linear kernel's ard flag" in lib.gpso_last_error()


def test_combination_refuses_a_linear_factor():
    lib = backend.load_library()
    h = ctypes.c_void_p()
    ids, ard, base, pard = (ctypes.c_int * 2)(LINEAR, 2), (ctypes.c_int * 2)(0, 0), (ctypes.c_int * 2)(0, 0), (ctypes.c_int * 2)(0, 0)
    assert lib.gpso_create_combination(0, 6, 2, ids, ard, base, pard, 0, ctypes.byref(h)) == -1
    assert b"Linear kernel cannot be a factor of a product" in lib.gpso_last_error()


@pytest.mark.parametrize("create", ["gpso_create_sum", "gpso_create_product"])
def test_sum_and_product_entry_points_still_refuse_the_id(create):
    lib = backend.load_library()
    h = ctypes.c_void_p()
    ids, ard = (ctypes.c_int * 2)(LINEAR, 2), (ctypes.c_int * 2)(0, 0)
    assert getattr(lib, create)(0, 2, ids, ard, 0, ctypes.byref(h)) == -1
    assert b"unknown component kernel id" in lib.gpso_last_error()
