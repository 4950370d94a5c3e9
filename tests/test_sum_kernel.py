"""
Sum kernel (gpflow.kernels.Sum, k = sum_c k_c) without a GPU: the oracle's closed-form gradient, the model layer (flattening,
packing and leaf names, shared objects refused, frozen components, persistence, an optimiser run through the checker backend),
the fp32 screening covariance of a sum against the contract of the screening error model, and the C argument checks that
need no device.
"""
import ctypes
import json
import os

import numpy as np
import pytest

from oracle import gpr_oracle as go
from pygpso_b200 import GPRSurrogate, backend, gpmodel
from tests import rq_oracle as rq
from tests import sum_oracle as so
from tests.test_oracle_goldens import make_optimiser, seeded_points


def synthetic(N, d, seed=11):
    rng = np.random.default_rng(seed)
    X = rng.random((N, d))
    return X, (np.sin(3 * X.sum(1)) + 0.3 * np.sin(40 * X[:, 0]) + 0.01 * rng.standard_normal(N))[:, None]


MIXED = {
    "se+m12": [so.Comp("SquaredExponential", 0.5, 0.8), so.Comp("Matern12", 0.05, 0.2)],
    "m52+rq_ard": [so.Comp("Matern52", 0.4, 1.1), so.Comp(rq.KERNEL, [0.3, 0.6, 0.5], 0.4, alpha=1.7)],
    "four": [so.Comp("Matern32", [0.3, 0.5, 0.7], 0.5), so.Comp("SquaredExponential", 0.6, 0.7),
             so.Comp(rq.KERNEL, 0.2, 0.3, alpha=0.8), so.Comp("Matern12", [0.2, 0.1, 0.4], 0.1)],
}


# ---- oracle ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("case", sorted(MIXED))
@pytest.mark.parametrize("mean_id", [0, 1, 2])
def test_oracle_gradient_matches_finite_differences(case, mean_id):
    N, d = 30, 3
    X, y = synthetic(N, d)
    mean = {0: None, 1: 0.2, 2: (np.array([0.3, -0.5, 0.2]), 0.1)}[mean_id]
    h = so.SumHyper(MIXED[case], 2e-3, mean)
    fam = [c.family for c in h.comps]
    nls = [c.n_ls for c in h.comps]
    u = h.pack()
    f, g = so.neg_lml_and_grad(fam, nls, X, y, u, mean_id)
    assert f == pytest.approx(-so.lml(so.SumHyper.unpack(fam, nls, u, mean_id, d), X, y), rel=1e-12)
    assert g.size == u.size == h.theta().size
    for i in range(u.size):
        e = np.zeros_like(u)
        e[i] = 1e-6
        fd = (so.neg_lml_and_grad(fam, nls, X, y, u + e, mean_id)[0] - so.neg_lml_and_grad(fam, nls, X, y, u - e, mean_id)[0]) / 2e-6
        assert g[i] == pytest.approx(fd, rel=2e-5, abs=2e-6), i


@pytest.mark.parametrize("family", ["Matern12", "Matern52", "SquaredExponential", rq.KERNEL])
def test_two_halves_equal_the_bare_kernel(family):
    X, y = synthetic(25, 2)
    alpha = 1.3 if family == rq.KERNEL else None
    halves = so.SumHyper([so.Comp(family, 0.4, 0.6, alpha), so.Comp(family, 0.4, 0.6, alpha)], 1e-3, 0.1)
    whole = so.SumHyper([so.Comp(family, 0.4, 1.2, alpha)], 1e-3, 0.1)
    np.testing.assert_allclose(so.kern(halves, X, None), so.kern(whole, X, None), rtol=4e-16, atol=0.0)
    assert so.lml(halves, X, y) == pytest.approx(so.lml(whole, X, y), rel=1e-12)
    xc = np.random.default_rng(1).random((9, 2))
    for a, b in zip(so.predict_y(halves, X, y, xc), so.predict_y(whole, X, y, xc)):
        np.testing.assert_allclose(a, b, rtol=1e-10, atol=1e-12)
    # and the one-component sum is the family's own oracle (which expands the squared distance: a looser bar)
    bare = rq.RQHyper(1.3, 0.4, 1.2, 1e-3, 0.1) if alpha else go.Hyper(0.4, 1.2, 1e-3, 0.1)
    mb, vb = rq.predict_y(X, y, bare, xc) if alpha else go.predict_y(family, X, y, bare, xc)
    m, v = so.predict_y(whole, X, y, xc)
    np.testing.assert_allclose(m, mb, rtol=1e-6, atol=1e-6)
    np.testing.assert_allclose(v, vb, rtol=1e-6, atol=1e-6)


def test_full_cov_diagonal_is_the_marginal_variance():
    X, y = synthetic(25, 3)
    h = so.SumHyper(MIXED["four"], 1e-3, 0.0)
    xc = np.random.default_rng(2).random((11, 3))
    mf, cov = so.predict_f_full_cov(h, X, y, xc)
    m, v = so.predict_y(h, X, y, xc)
    np.testing.assert_allclose(mf, m[:, 0], rtol=1e-12)
    np.testing.assert_allclose(np.diag(cov), v[:, 0] - 1e-3, rtol=1e-9, atol=1e-13)


# ---- model layer ----------------------------------------------------------------------------------------------------
def model(kernel, mean=None, d=2):
    X, y = synthetic(20, d)
    return gpmodel.GPR((X, y), kernel, mean_function=mean, noise_variance=1e-3, backend=so.SumOracleBackend())


def test_add_builds_a_sum_and_flattens():
    a, b, c = gpmodel.SquaredExponential(), gpmodel.Matern12(), gpmodel.Matern32()
    s = a + b
    assert isinstance(s, gpmodel.Sum) and s.kernels == [a, b]
    left, right = (a + b) + c, a + (b + c)
    assert left.kernels == right.kernels == [a, b, c]
    assert gpmodel.kernels.Sum is gpmodel.Sum
    assert gpmodel.Sum([a]).kernels == [a]


def test_sum_limits_and_shared_objects():
    k = gpmodel.Matern52()
    with pytest.raises(ValueError, match="twice"):
        k + k
    with pytest.raises(ValueError, match="twice"):
        gpmodel.Sum([k, gpmodel.Matern12() + k])
    with pytest.raises(ValueError, match="1..4"):
        gpmodel.Sum([gpmodel.Matern52() for _ in range(5)])
    with pytest.raises(ValueError, match="1..4"):
        gpmodel.Sum([])
    with pytest.raises(TypeError):
        gpmodel.Sum([k, 3.0])


def test_packing_order_and_leaf_names():
    k0 = gpmodel.SquaredExponential(variance=0.8, lengthscales=[0.5, 0.6])
    k1 = gpmodel.RationalQuadratic(variance=0.3, lengthscales=0.2, alpha=2.0)
    m = model(k0 + k1, gpmodel.Linear(np.array([[0.3], [-0.2]]), np.array([0.1])))
    assert np.array_equal(m._theta(), [0.5, 0.6, 0.8, 2.0, 0.2, 0.3, 1e-3, 0.3, -0.2, 0.1])
    names = list(gpmodel.parameter_dict(m))
    assert names == [".kernel.kernels[0].lengthscales", ".kernel.kernels[0].variance", ".kernel.kernels[1].alpha",
                     ".kernel.kernels[1].lengthscales", ".kernel.kernels[1].variance", ".likelihood.variance",
                     ".mean_function.A", ".mean_function.b"]
    gpmodel.multiple_assign(m, {".kernel.kernels[1].alpha": 3.5, ".kernel.kernels[0].variance": 0.25})
    assert m._theta()[2] == 0.25 and m._theta()[3] == 3.5
    assert "GPR.kernel.kernels[1].alpha" in gpmodel.tabulate_module_summary(m)
    assert type(m._session) is so.SumOracleSession
    assert m._session.families == ["SquaredExponential", "RationalQuadratic"] and m._session.n_lss == [2, 1]


def test_ard_check_runs_per_component():
    with pytest.raises(ValueError, match="ARD"):
        model(gpmodel.Matern52(lengthscales=[0.1, 0.2, 0.3]) + gpmodel.Matern12(), d=2)
    with pytest.raises(TypeError):
        model(gpmodel.Sum([gpmodel.Matern52(), gpmodel.Kernel()]))


def test_training_loss_and_predict_are_the_oracle():
    m = model(gpmodel.Matern52(lengthscales=0.4) + gpmodel.RationalQuadratic(lengthscales=[0.2, 0.3], alpha=1.5),
              gpmodel.Constant(0.1))
    f, g = m.neg_log_marginal_likelihood_and_grad(m._pack())
    f_ref, g_ref = so.neg_lml_and_grad(["Matern52", rq.KERNEL], [1, 2], *m.data, m._pack(), 1)
    assert f == f_ref and np.array_equal(g, g_ref)
    xc = np.random.default_rng(0).random((7, 2))
    mean, var = m.predict_y(xc)
    mf, cov = m.predict_f(xc, full_cov=True)
    np.testing.assert_allclose(mf[:, 0], mean[:, 0], rtol=1e-12)
    np.testing.assert_allclose(np.diag(cov[0]), var[:, 0] - 1e-3, rtol=1e-10, atol=1e-14)


def test_frozen_component_parameter_is_left_alone():
    k0, k1 = gpmodel.SquaredExponential(lengthscales=0.5), gpmodel.Matern12(lengthscales=0.1, variance=0.3)
    m = model(k0 + k1, gpmodel.Constant(0.0))
    k1.lengthscales.trainable = False
    before = k1.lengthscales.numpy().copy()
    others = [p.numpy().copy() for p in (k0.lengthscales, k0.variance, k1.variance)]
    res = gpmodel.Scipy().minimize(m.training_loss, m.trainable_variables)
    assert res.success or res.nit > 0
    assert k1.lengthscales.numpy() == pytest.approx(before, rel=1e-15)  # only the softplus round trip of the packed vector
    assert any(not np.array_equal(p.numpy(), o) for p, o in zip((k0.lengthscales, k0.variance, k1.variance), others))


def _trained_surrogate(kernel, backend_):
    surr = GPRSurrogate(gp_kernel=kernel, gp_meanf=gpmodel.Constant(0.0), points=seeded_points(), backend=backend_)
    x, y = surr.current_training_data
    surr._gp_train(x=x, y=y[:, np.newaxis])
    return surr, x


def test_save_from_saved_round_trips_every_parameter(tmp_path):
    kernel = (gpmodel.SquaredExponential(lengthscales=[0.5, 0.4]) + gpmodel.RationalQuadratic(lengthscales=0.2, alpha=1.2)
              + gpmodel.Matern12(lengthscales=0.1, variance=0.2))
    surr, x = _trained_surrogate(kernel, so.SumOracleBackend())
    surr.save(str(tmp_path / "s"))
    with open(tmp_path / "s" / GPRSurrogate.GPR_INFO) as fh:
        info = json.load(fh)
    assert info["gpr_kernel"] == "Sum"
    assert info["gpr_kernel_components"] == [["SquaredExponential", [2]], ["RationalQuadratic", []], ["Matern12", []]]
    loaded = GPRSurrogate.from_saved(str(tmp_path / "s"), backend=so.SumOracleBackend())
    lk = loaded.gpflow_model.kernel
    assert [type(k) for k in lk.kernels] == [gpmodel.SquaredExponential, gpmodel.RationalQuadratic, gpmodel.Matern12]
    assert loaded.gpflow_model._theta().tobytes() == surr.gpflow_model._theta().tobytes()
    p, q = surr.gpflow_model.predict_y(x), loaded.gpflow_model.predict_y(x)
    assert np.array_equal(p[0], q[0]) and np.array_equal(p[1], q[1])


def test_non_sum_save_files_are_unchanged(tmp_path):
    from tests.oracle_backend import OracleBackend

    surr, _ = _trained_surrogate(gpmodel.Matern52(lengthscales=0.25), OracleBackend())
    surr.save(str(tmp_path / "s"))
    with open(os.path.join(tmp_path, "s", GPRSurrogate.GPR_INFO)) as fh:
        text = fh.read()
    model_ = surr.gpflow_model
    expected = json.dumps({
        "gpr_kernel": "Matern52", "gpr_kernel_shape": [], "gpr_meanf": "Constant", "gpr_meanf_shape": [],
        "gp_varsigma": surr.gp_varsigma, "gp_likelihood": surr.gp_lik_sigma, "optimiser": ["Scipy"],
    })
    assert text == expected
    import dill

    with open(os.path.join(tmp_path, "s", GPRSurrogate.GPR_FILE), "rb") as fh:
        params = dill.load(fh)
    assert list(params) == [".kernel.lengthscales", ".kernel.variance", ".likelihood.variance", ".mean_function.c"]
    assert params[".kernel.variance"].tobytes() == model_.kernel.variance.numpy().tobytes()


def test_optimiser_runs_with_the_sum_checker_backend():
    from tests.conftest import paper_objective

    opt = make_optimiser(backend=so.SumOracleBackend(), depth=3, budget=40)
    opt.gp_surr.gp_kernel = gpmodel.SquaredExponential(lengthscales=0.5) + gpmodel.Matern12(lengthscales=0.05, variance=0.1)
    best = opt.run(paper_objective)
    k = opt.gp_surr.gpflow_model.kernel
    assert isinstance(k, gpmodel.Sum) and type(opt.gp_surr.gpflow_model._session) is so.SumOracleSession
    assert opt.n_eval_counter >= 40 and np.isfinite(best.score_mu)


# ---- fp32 screening covariance: |k32 - k64| <= 2e-6 var_tot, the rounding of the additions included ----------------------
@pytest.mark.parametrize("case", sorted(MIXED) + ["rq_large_alpha", "tiny_plus_big"])
def test_cov32_of_a_sum_within_the_screen_contract(case):
    comps = {
        "rq_large_alpha": [so.Comp(rq.KERNEL, 0.3, 1.0, alpha=1e4), so.Comp("Matern52", 0.3, 1.0), so.Comp("Matern32", 0.2, 1.0)],
        "tiny_plus_big": [so.Comp("SquaredExponential", 0.5, 1e3), so.Comp("Matern12", 0.05, 1e-3)],
    }.get(case, MIXED.get(case))
    h = so.SumHyper(comps, 1e-3)
    rng = np.random.default_rng(3)
    d = 3
    Xa = rng.random((300, d))
    Xb = np.vstack([rng.random((400, d)), Xa[:50] + 1e-4 * rng.standard_normal((50, d)), Xa[:5]])
    k32 = so.cov32(h, Xa, Xb).astype(np.float64)
    k64 = so.kern(h, Xa, Xb)
    err = np.max(np.abs(k32 - k64))
    # half the contract: MUFU.EX2 / RSQ / LG2 and __fdividef are not emulated (a few ulp each)
    assert err <= 2e-6 * h.var_tot / 2.0, err / h.var_tot
    assert np.all(np.diag(so.cov32(h, Xa[:5], Xa[:5])) == np.float32(h.var_tot)) or case == "tiny_plus_big"


# ---- C argument checks that need no device ------------------------------------------------------------------------------
def test_create_sum_rejects_bad_arguments():
    lib = backend.load_library()
    h = ctypes.c_void_p()

    def create(n, ids, ards, mean=1):
        k = (ctypes.c_int * max(len(ids), 1))(*ids)
        a = (ctypes.c_int * max(len(ards), 1))(*ards)
        return lib.gpso_create_sum(0, n, k, a, mean, ctypes.byref(h))

    assert create(0, [], []) == -1   # GPSO_E_BADARG before any CUDA call
    assert b"components" in lib.gpso_last_error()
    assert create(5, [0] * 5, [0] * 5) == -1
    assert create(2, [2, 7], [0, 0]) == -1
    assert b"kernel id" in lib.gpso_last_error()
    assert create(2, [2, 5], [0, 0]) == -1    # a sum is not a component
    assert create(2, [2, 3], [0, 2]) == -1
    assert b"ard" in lib.gpso_last_error()
    assert create(2, [2, 3], [0, 1], mean=3) == -1
    assert lib.gpso_create(0, 5, 0, 1, ctypes.byref(h)) == -1   # the sum id has no components: gpso_create_sum
    assert not h.value
