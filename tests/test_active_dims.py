"""
Kernels on a subset of the inputs (GPflow's active_dims) without a GPU: the oracle's closed-form gradient against finite
differences, the keyword on every family and Periodic's delegation, slice / list / repeat resolution, the refusals, identity maps
that leave the session without a map, the model against the oracle through the checker backend, persistence, an optimiser run,
the 64-row budget, and the C argument checks that need no device.
"""
import ctypes
import json

import numpy as np
import pytest

from pygpso_b200 import GPRSurrogate, backend, gpmodel
from tests import active_dims_oracle as ad
from tests import periodic_oracle as pe
from tests import rq_oracle as rq
from tests import sum_oracle as so
from tests.test_oracle_goldens import make_optimiser, seeded_points
from tests.test_sum_kernel import synthetic

FAMILIES = ("Matern12", "Matern32", "Matern52", "SquaredExponential", "RationalQuadratic")


def model(kernel, mean=None, d=4, N=30, backend_=None):
    X, y = synthetic(N, d)
    return gpmodel.GPR((X, y), kernel, mean_function=mean, noise_variance=1e-3,
                       backend=backend_ or ad.ActiveDimsOracleBackend())


# ---- oracle -----------------------------------------------------------------------------------------------------------
CASES = {
    "m52_subset": ("Sum", [("Matern52", 1)], [[0, 2]], [so.Comp("Matern52", 0.4, 0.9)]),
    "rq_ard_permuted": ("Sum", [(rq.KERNEL, 2)], [[3, 0]], [so.Comp(rq.KERNEL, [0.3, 0.6], 0.7, alpha=1.4)]),
    "periodic_ard": ("Sum", [("Periodic", 1, "SquaredExponential", 2)], [[1, 3]],
                     [pe.PeriodicHyper("SquaredExponential", 0.5, 0.8, [0.6, 0.9], 1.0)]),
    "additive": ("Sum", [("Matern52", 2), ("Periodic", 1, rq.KERNEL, 1)], [[0, 1], [2]],
                 [so.Comp("Matern52", [0.4, 0.5], 0.6), pe.PeriodicHyper(rq.KERNEL, 0.7, 0.5, 0.8, 1.0, alpha=1.3)]),
    "phase_product": ("Product", [("Matern52", 1), ("Periodic", 1, "SquaredExponential", 1)], [[0, 1, 2], [3]],
                      [so.Comp("Matern52", 0.5, 0.9), pe.PeriodicHyper("SquaredExponential", 0.6, 1.2, 0.7, 1.0)]),
    "overlap_repeat": ("Product", [("SquaredExponential", 3), ("Matern32", 1)], [[1, 1, 2], [2, 0]],
                       [so.Comp("SquaredExponential", [0.4, 0.8, 0.5], 0.9), so.Comp("Matern32", 0.6, 1.1)]),
}


@pytest.mark.parametrize("key", sorted(CASES))
@pytest.mark.parametrize("mean_id", [0, 1, 2])
def test_oracle_gradient_matches_finite_differences(key, mean_id):
    kind, specs, dims, comps = CASES[key]
    X, y = synthetic(25, 4)
    mean = {0: None, 1: 0.2, 2: (np.array([0.3, -0.5, 0.2, 0.1]), 0.1)}[mean_id]
    u = pe.CompositeHyper(kind, comps, 2e-3, mean).pack()
    f, g = ad.neg_lml_and_grad(kind, specs, dims, X, y, u, mean_id)
    assert g.size == u.size
    for i in range(u.size):
        e = np.zeros_like(u)
        e[i] = 1e-6
        fd = (ad.neg_lml_and_grad(kind, specs, dims, X, y, u + e, mean_id)[0]
              - ad.neg_lml_and_grad(kind, specs, dims, X, y, u - e, mean_id)[0]) / 2e-6
        assert g[i] == pytest.approx(fd, rel=2e-5, abs=2e-6), i


def test_oracle_with_every_column_is_the_composite_oracle():
    kind, specs, _, comps = CASES["phase_product"]
    X, y = synthetic(25, 4)
    u = pe.CompositeHyper(kind, comps, 2e-3).pack()
    f, g = ad.neg_lml_and_grad(kind, specs, [list(range(4))] * 2, X, y, u, 0)
    f_ref, g_ref = pe.composite_neg_lml_and_grad(kind, specs, X, y, u, 0)
    assert f == f_ref
    np.testing.assert_allclose(g, g_ref, rtol=1e-13, atol=1e-15)


# ---- the keyword --------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("family", FAMILIES)
def test_every_family_takes_the_keyword(family):
    k = getattr(gpmodel, family)(lengthscales=[0.3, 0.4], active_dims=[2, 0])
    assert isinstance(k.active_dims, np.ndarray) and k.active_dims.dtype.kind == "i"
    assert list(k.active_dims) == [2, 0]
    assert getattr(gpmodel, family)().active_dims == slice(None)
    assert getattr(gpmodel, family)(active_dims=slice(1, None)).active_dims == slice(1, None)


def test_periodic_active_dims_is_the_base_kernels():
    base = gpmodel.SquaredExponential(active_dims=[3])
    p = gpmodel.Periodic(base, period=1.0)
    assert list(p.active_dims) == [3]
    p.active_dims = [1, 2]
    assert list(base.active_dims) == [1, 2]
    base.active_dims = None
    assert p.active_dims == slice(None)


def test_active_dims_is_not_a_parameter():
    k = gpmodel.Matern52(active_dims=[0, 1])
    m = model(k)
    assert list(gpmodel.parameter_dict(m)) == [".kernel.lengthscales", ".kernel.variance", ".likelihood.variance"]
    assert all(p.name != "active_dims" for p in m.parameters)


@pytest.mark.parametrize("dims,expect", [(slice(1, None), [1, 2, 3]), (slice(None, None, 2), [0, 2]), (slice(-1, None), [3]),
                                         ([3, 0], [3, 0]), ((1, 1, 2), [1, 1, 2]), (np.array([2]), [2])])
def test_resolution(dims, expect):
    m = model(gpmodel.Matern52(active_dims=dims))
    assert m._leaf_dims == [expect]
    assert m._session.leaf_dims == [expect]


@pytest.mark.parametrize("dims", [None, slice(None), [0, 1, 2, 3], slice(0, 4)])
def test_identity_maps_open_no_map(dims):
    m = model(gpmodel.Matern52(active_dims=dims) + gpmodel.Periodic(gpmodel.SquaredExponential(active_dims=dims)))
    assert m._session.calls["set_active_dims"] == 0 and m._session.leaf_dims is None


def test_identity_map_sessions_of_the_existing_checkers_run_unchanged():
    """The checker backends without set_active_dims still serve every kernel whose map is the identity."""
    m = model(gpmodel.Periodic(gpmodel.SquaredExponential(active_dims=list(range(3)))), d=3, backend_=pe.PeriodicOracleBackend())
    assert np.isfinite(m.training_loss())


def test_map_is_cleared_when_it_becomes_the_identity():
    m = model(gpmodel.Matern52(active_dims=[0, 1]))
    assert m._session.leaf_dims == [[0, 1]]
    X, y = synthetic(30, 2)
    m.data = (X, y)
    assert m._session.calls["set_active_dims"] == 2 and m._session.leaf_dims is None


# ---- refusals ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dims,match", [([0, 4], "outside"), ([-1], "outside"), ([], "no column"), (slice(5, None), "no column")])
def test_bad_selections_are_refused(dims, match):
    with pytest.raises(ValueError, match=match):
        model(gpmodel.Matern52(active_dims=dims))


def test_bad_keyword_values_are_refused():
    with pytest.raises(ValueError, match="active_dims"):
        gpmodel.Matern52(active_dims=[[0, 1]])
    with pytest.raises(ValueError, match="active_dims"):
        gpmodel.Matern52(active_dims=[0.5])


def test_ard_counts_follow_the_active_columns():
    with pytest.raises(ValueError, match="ARD lengthscales.*2 active"):
        model(gpmodel.Matern52(lengthscales=[0.3, 0.4, 0.5, 0.6], active_dims=[0, 1]))
    with pytest.raises(ValueError, match="ARD period.*1 active"):
        model(gpmodel.Periodic(gpmodel.SquaredExponential(active_dims=[3]), period=[0.5, 0.6]))
    m = model(gpmodel.Periodic(gpmodel.SquaredExponential(lengthscales=[0.3, 0.4], active_dims=[3, 1]), period=[0.5, 0.6]))
    assert m._leaf_dims == [[3, 1]]


def test_row_budget():
    """Four components of 16 columns each fit at d = 20 (64 rows); a 65th row is refused."""
    d = 20
    parts = [gpmodel.Matern52(active_dims=list(range(i, i + 16))) for i in range(4)]
    m = model(gpmodel.Sum(parts), d=d)
    assert [len(c) for c in m._leaf_dims] == [16] * 4
    parts = [gpmodel.Matern52(active_dims=list(range(i, i + 16))) for i in range(3)] + [gpmodel.Matern52(active_dims=list(range(17)))]
    with pytest.raises(ValueError, match="65 rows"):
        model(gpmodel.Sum(parts), d=d)
    per = gpmodel.Periodic(gpmodel.SquaredExponential(active_dims=list(range(17))))
    with pytest.raises(ValueError, match="66 rows"):
        model(gpmodel.Sum([gpmodel.Matern52(active_dims=list(range(16))) for _ in range(2)] + [per]), d=d)


# ---- the model against the oracle ---------------------------------------------------------------------------------------
KERNELS = {
    "m52_subset": lambda: gpmodel.Matern52(lengthscales=0.4, active_dims=[0, 2]),
    "rq_ard_permuted": lambda: gpmodel.RationalQuadratic(lengthscales=[0.3, 0.6], alpha=1.4, active_dims=[3, 0]),
    "periodic_ard": lambda: gpmodel.Periodic(gpmodel.SquaredExponential(lengthscales=0.5, active_dims=[1, 3]), period=[0.6, 0.9]),
    "additive": lambda: gpmodel.Matern52(lengthscales=[0.4, 0.5], active_dims=[0, 1])
    + gpmodel.Periodic(gpmodel.RationalQuadratic(lengthscales=0.7, alpha=1.3, active_dims=[2]), period=0.8),
    "phase_product": lambda: gpmodel.Matern52(lengthscales=0.5, active_dims=[0, 1, 2])
    * gpmodel.Periodic(gpmodel.SquaredExponential(lengthscales=0.6, active_dims=[3]), period=0.7),
}


@pytest.mark.parametrize("key", sorted(KERNELS))
def test_training_loss_and_predict_are_the_oracle(key):
    m = model(KERNELS[key](), gpmodel.Constant(0.1))
    session = m._session
    f, g = m.neg_log_marginal_likelihood_and_grad(m._pack())
    f_ref, g_ref = ad.neg_lml_and_grad(session.kind, session.specs, m._leaf_dims, *m.data, m._pack(), 1)
    assert f == f_ref and np.array_equal(g, g_ref)
    xc = np.random.default_rng(0).random((7, 4))
    mean, var = m.predict_y(xc)
    h = pe.CompositeHyper.from_theta(session.kind, session.specs, m._theta(), 1, 4)
    mr, vr = ad.predict_y(h, m._leaf_dims, *m.data, xc)
    np.testing.assert_allclose(mean, mr, rtol=1e-12)
    np.testing.assert_allclose(var, vr, rtol=1e-12)


def test_inactive_columns_do_not_change_the_posterior():
    m = model(gpmodel.Matern52(lengthscales=0.5, active_dims=[0, 1]))
    xc = np.random.default_rng(1).random((5, 4))
    xe = xc.copy()
    xe[:, 2:] = np.random.default_rng(2).random((5, 2))
    a, b = m.predict_y(xc), m.predict_y(xe)
    assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1])


def _fitted(kernel, backend_):
    surr = GPRSurrogate(gp_kernel=kernel, gp_meanf=gpmodel.Constant(0.0), points=seeded_points(), backend=backend_)
    x, y = surr.current_training_data
    surr.gpflow_model = gpmodel.GPR((x, y[:, np.newaxis]), kernel, gpmodel.Constant(0.0), surr.gp_lik_sigma, surr.backend)
    rng = np.random.default_rng(9)
    gpmodel.multiple_assign(surr.gpflow_model, {k: 0.2 + rng.random(np.shape(v)) for k, v in gpmodel.parameter_dict(surr.gpflow_model).items()})
    return surr, x


def test_save_from_saved_round_trips_the_map(tmp_path):
    kernel = gpmodel.Matern52(lengthscales=[0.4, 0.5], active_dims=slice(0, 2)) + gpmodel.Periodic(gpmodel.SquaredExponential())
    surr, x = _fitted(kernel, ad.ActiveDimsOracleBackend())
    d = x.shape[1]
    surr.save(str(tmp_path / "s"))
    with open(tmp_path / "s" / GPRSurrogate.GPR_INFO) as fh:
        info = json.load(fh)
    assert info["gpr_kernel_active_dims"] == [[0, 1], None]
    loaded = GPRSurrogate.from_saved(str(tmp_path / "s"), backend=ad.ActiveDimsOracleBackend())
    lk = loaded.gpflow_model.kernel
    assert list(lk.kernels[0].active_dims) == [0, 1] and lk.kernels[1].active_dims == slice(None)
    assert loaded.gpflow_model._leaf_dims == [[0, 1], list(range(d))]
    assert loaded.gpflow_model._theta().tobytes() == surr.gpflow_model._theta().tobytes()
    p, q = surr.gpflow_model.predict_y(x), loaded.gpflow_model.predict_y(x)
    assert np.array_equal(p[0], q[0]) and np.array_equal(p[1], q[1])


def test_save_of_a_bare_kernel_with_a_map(tmp_path):
    kernel = gpmodel.Periodic(gpmodel.RationalQuadratic(active_dims=[1]), period=0.9)
    surr, x = _fitted(kernel, ad.ActiveDimsOracleBackend())
    surr.save(str(tmp_path / "s"))
    loaded = GPRSurrogate.from_saved(str(tmp_path / "s"), backend=ad.ActiveDimsOracleBackend())
    assert list(loaded.gpflow_model.kernel.active_dims) == [1]
    p, q = surr.gpflow_model.predict_y(x), loaded.gpflow_model.predict_y(x)
    assert np.array_equal(p[0], q[0]) and np.array_equal(p[1], q[1])


@pytest.mark.parametrize("dims", [None, slice(None)])
def test_saves_without_a_map_are_unchanged(tmp_path, dims):
    """A kernel given no columns (or all of them as slice(None)) saves the text the previous release wrote, byte for byte."""
    surr, _ = _fitted(gpmodel.Matern52(lengthscales=0.25, active_dims=dims), ad.ActiveDimsOracleBackend())
    surr.save(str(tmp_path / "s"))
    with open(tmp_path / "s" / GPRSurrogate.GPR_INFO) as fh:
        text = fh.read()
    assert text == json.dumps({
        "gpr_kernel": "Matern52", "gpr_kernel_shape": [], "gpr_meanf": "Constant", "gpr_meanf_shape": [],
        "gp_varsigma": surr.gp_varsigma, "gp_likelihood": surr.gp_lik_sigma, "optimiser": ["Scipy"],
    })


def test_optimiser_runs_with_the_checker_backend():
    from tests.conftest import paper_objective

    opt = make_optimiser(backend=ad.ActiveDimsOracleBackend(), depth=3, budget=40)
    opt.gp_surr.gp_kernel = gpmodel.Matern52(lengthscales=0.5, active_dims=[0]) + gpmodel.Matern52(lengthscales=0.5, active_dims=[1])
    best = opt.run(paper_objective)
    session = opt.gp_surr.gpflow_model._session
    assert session.leaf_dims == [[0], [1]]
    assert opt.n_eval_counter >= 40 and np.isfinite(best.score_mu)


# ---- C argument checks ------------------------------------------------------------------------------------------------
def test_set_active_dims_rejects_a_null_handle():
    lib = backend.load_library()
    counts, dims = (ctypes.c_int * 1)(1), (ctypes.c_int * 1)(0)
    assert lib.gpso_set_active_dims(None, 1, counts, dims) == -1
    assert b"null handle" in lib.gpso_last_error()
