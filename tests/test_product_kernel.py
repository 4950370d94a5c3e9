"""
Product kernel (gpflow.kernels.Product, k = prod_c k_c) without a GPU: the oracle's closed-form gradient, the model layer
(flattening, packing and leaf names, shared objects and sums of products refused, frozen factors, persistence, an optimiser run
through the checker backend), the fp32 screening covariance of a product against the contract of the screening error model,
and the C argument checks that need no device.
"""
import ctypes
import itertools
import json

import numpy as np
import pytest

from pygpso_b200 import GPRSurrogate, backend, gpmodel
from tests import product_oracle as po
from tests import rq_oracle as rq
from tests import sum_oracle as so
from tests.test_oracle_goldens import make_optimiser, seeded_points
from tests.test_sum_kernel import synthetic

MIXED = {
    "se*m12": [po.Comp("SquaredExponential", 0.5, 0.8), po.Comp("Matern12", 0.3, 1.5)],
    "m52*rq_ard": [po.Comp("Matern52", 0.4, 1.1), po.Comp(rq.KERNEL, [0.3, 0.6, 0.5], 0.4, alpha=1.7)],
    "four": [po.Comp("Matern32", [0.3, 0.5, 0.7], 0.5), po.Comp("SquaredExponential", 0.6, 1.7),
             po.Comp(rq.KERNEL, 0.4, 1.3, alpha=0.8), po.Comp("Matern12", [0.6, 0.9, 0.8], 1.1)],
}
FAMILIES = ["Matern12", "Matern32", "Matern52", "SquaredExponential", rq.KERNEL]


# ---- oracle ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("case", sorted(MIXED))
@pytest.mark.parametrize("mean_id", [0, 1, 2])
def test_oracle_gradient_matches_finite_differences(case, mean_id):
    N, d = 30, 3
    X, y = synthetic(N, d)
    mean = {0: None, 1: 0.2, 2: (np.array([0.3, -0.5, 0.2]), 0.1)}[mean_id]
    h = po.ProductHyper(MIXED[case], 2e-3, mean)
    fam = [c.family for c in h.comps]
    nls = [c.n_ls for c in h.comps]
    u = h.pack()
    f, g = po.neg_lml_and_grad(fam, nls, X, y, u, mean_id)
    assert f == pytest.approx(-po.lml(po.ProductHyper.unpack(fam, nls, u, mean_id, d), X, y), rel=1e-12)
    assert g.size == u.size == h.theta().size
    for i in range(u.size):
        e = np.zeros_like(u)
        e[i] = 1e-6
        fd = (po.neg_lml_and_grad(fam, nls, X, y, u + e, mean_id)[0] - po.neg_lml_and_grad(fam, nls, X, y, u - e, mean_id)[0]) / 2e-6
        assert g[i] == pytest.approx(fd, rel=2e-5, abs=2e-6), i


@pytest.mark.parametrize("family", FAMILIES)
def test_one_factor_is_the_bare_kernel(family):
    X, y = synthetic(25, 2)
    alpha = 1.3 if family == rq.KERNEL else None
    one = po.ProductHyper([po.Comp(family, 0.4, 1.2, alpha)], 1e-3, 0.1)
    as_sum = so.SumHyper(one.comps, 1e-3, 0.1)
    assert np.array_equal(po.kern(one, X, None), so.kern(as_sum, X, None))
    assert po.lml(one, X, y) == so.lml(as_sum, X, y)
    u = one.pack()
    fam, nls = [family], [1]
    for a, b in zip(po.neg_lml_and_grad(fam, nls, X, y, u, 1), so.neg_lml_and_grad(fam, nls, X, y, u, 1)):
        np.testing.assert_allclose(a, b, rtol=1e-13, atol=0)
    xc = np.random.default_rng(1).random((9, 2))
    for a, b in zip(po.predict_y(one, X, y, xc), so.predict_y(as_sum, X, y, xc)):
        assert np.array_equal(a, b)


def test_product_of_equal_se_factors_is_one_se():
    """SE(l) * SE(l) = SE(l / sqrt 2) with the variances multiplied: the product's closed form against a known kernel."""
    X, y = synthetic(25, 3)
    h = po.ProductHyper([po.Comp("SquaredExponential", 0.5, 0.6), po.Comp("SquaredExponential", 0.5, 2.0)], 1e-3, 0.1)
    whole = so.SumHyper([so.Comp("SquaredExponential", 0.5 / np.sqrt(2.0), 1.2)], 1e-3, 0.1)
    np.testing.assert_allclose(po.kern(h, X, None), so.kern(whole, X, None), rtol=1e-13, atol=1e-15)
    assert po.lml(h, X, y) == pytest.approx(so.lml(whole, X, y), rel=1e-11)


def test_full_cov_diagonal_is_the_marginal_variance():
    X, y = synthetic(25, 3)
    h = po.ProductHyper(MIXED["four"], 1e-3, 0.0)
    xc = np.random.default_rng(2).random((11, 3))
    mf, cov = po.predict_f_full_cov(h, X, y, xc)
    m, v = po.predict_y(h, X, y, xc)
    np.testing.assert_allclose(mf, m[:, 0], rtol=1e-12)
    np.testing.assert_allclose(np.diag(cov), v[:, 0] - 1e-3, rtol=1e-9, atol=1e-13)
    assert po.kern(h, xc, None)[3, 3] == h.var_prod


# ---- model layer ----------------------------------------------------------------------------------------------------
def model(kernel, mean=None, d=2):
    X, y = synthetic(20, d)
    return gpmodel.GPR((X, y), kernel, mean_function=mean, noise_variance=1e-3, backend=po.ProductOracleBackend())


def test_mul_builds_a_product_and_flattens():
    a, b, c = gpmodel.SquaredExponential(), gpmodel.Matern12(), gpmodel.Matern32()
    p = a * b
    assert isinstance(p, gpmodel.Product) and p.kernels == [a, b]
    left, right = (a * b) * c, a * (b * c)
    assert left.kernels == right.kernels == [a, b, c]
    assert gpmodel.kernels.Product is gpmodel.Product
    assert gpmodel.Product([a]).kernels == [a]
    assert (a * b + c).kernels[0].kernels == [a, b]   # a sum whose first term is a product: no flattening across kinds


def test_product_limits_and_shared_objects():
    k = gpmodel.Matern52()
    with pytest.raises(ValueError, match="twice in the product"):
        k * k
    with pytest.raises(ValueError, match="twice"):
        gpmodel.Product([k, gpmodel.Matern12() * k])
    with pytest.raises(ValueError, match="1..4"):
        gpmodel.Product([gpmodel.Matern52() for _ in range(5)])
    with pytest.raises(ValueError, match="1..4"):
        gpmodel.Product([])
    with pytest.raises(TypeError):
        gpmodel.Product([k, 3.0])


@pytest.mark.parametrize("build", [lambda a, b, c: a * b + c, lambda a, b, c: (a + b) * c, lambda a, b, c: gpmodel.Product([a + b])])
def test_sums_of_products_are_refused(build):
    a, b, c = gpmodel.Matern52(), gpmodel.SquaredExponential(), gpmodel.Matern12()
    with pytest.raises(TypeError, match="sums of products and products of sums are not supported"):
        model(build(a, b, c))


def test_packing_order_and_leaf_names():
    k0 = gpmodel.SquaredExponential(variance=0.8, lengthscales=[0.5, 0.6])
    k1 = gpmodel.RationalQuadratic(variance=0.3, lengthscales=0.2, alpha=2.0)
    m = model(k0 * k1, gpmodel.Linear(np.array([[0.3], [-0.2]]), np.array([0.1])))
    assert np.array_equal(m._theta(), [0.5, 0.6, 0.8, 2.0, 0.2, 0.3, 1e-3, 0.3, -0.2, 0.1])
    names = list(gpmodel.parameter_dict(m))
    assert names == [".kernel.kernels[0].lengthscales", ".kernel.kernels[0].variance", ".kernel.kernels[1].alpha",
                     ".kernel.kernels[1].lengthscales", ".kernel.kernels[1].variance", ".likelihood.variance",
                     ".mean_function.A", ".mean_function.b"]
    gpmodel.multiple_assign(m, {".kernel.kernels[1].alpha": 3.5, ".kernel.kernels[0].variance": 0.25})
    assert m._theta()[2] == 0.25 and m._theta()[3] == 3.5
    assert "GPR.kernel.kernels[1].alpha" in gpmodel.tabulate_module_summary(m)
    assert type(m._session) is po.ProductOracleSession
    assert m._session.families == ["SquaredExponential", "RationalQuadratic"] and m._session.n_lss == [2, 1]


def test_training_loss_and_predict_are_the_oracle():
    m = model(gpmodel.Matern52(lengthscales=0.4) * gpmodel.RationalQuadratic(lengthscales=[0.2, 0.3], alpha=1.5),
              gpmodel.Constant(0.1))
    f, g = m.neg_log_marginal_likelihood_and_grad(m._pack())
    f_ref, g_ref = po.neg_lml_and_grad(["Matern52", rq.KERNEL], [1, 2], *m.data, m._pack(), 1)
    assert f == f_ref and np.array_equal(g, g_ref)
    xc = np.random.default_rng(0).random((7, 2))
    mean, var = m.predict_y(xc)
    mf, cov = m.predict_f(xc, full_cov=True)
    np.testing.assert_allclose(mf[:, 0], mean[:, 0], rtol=1e-12)
    np.testing.assert_allclose(np.diag(cov[0]), var[:, 0] - 1e-3, rtol=1e-10, atol=1e-14)


def test_frozen_factor_parameter_is_left_alone():
    k0, k1 = gpmodel.SquaredExponential(lengthscales=0.5), gpmodel.Matern12(lengthscales=0.3, variance=0.7)
    m = model(k0 * k1, gpmodel.Constant(0.0))
    k1.variance.trainable = False
    before = k1.variance.numpy().copy()
    others = [p.numpy().copy() for p in (k0.lengthscales, k0.variance, k1.lengthscales)]
    res = gpmodel.Scipy().minimize(m.training_loss, m.trainable_variables)
    assert res.success or res.nit > 0
    assert k1.variance.numpy() == pytest.approx(before, rel=1e-15)  # only the softplus round trip of the packed vector
    assert any(not np.array_equal(p.numpy(), o) for p, o in zip((k0.lengthscales, k0.variance, k1.lengthscales), others))


def _trained_surrogate(kernel, backend_):
    surr = GPRSurrogate(gp_kernel=kernel, gp_meanf=gpmodel.Constant(0.0), points=seeded_points(), backend=backend_)
    x, y = surr.current_training_data
    surr._gp_train(x=x, y=y[:, np.newaxis])
    return surr, x


def test_save_from_saved_round_trips_every_parameter(tmp_path):
    kernel = (gpmodel.SquaredExponential(lengthscales=[0.5, 0.4]) * gpmodel.RationalQuadratic(lengthscales=0.2, alpha=1.2)
              * gpmodel.Matern12(lengthscales=0.5, variance=0.2))
    surr, x = _trained_surrogate(kernel, po.ProductOracleBackend())
    surr.save(str(tmp_path / "s"))
    with open(tmp_path / "s" / GPRSurrogate.GPR_INFO) as fh:
        info = json.load(fh)
    assert info["gpr_kernel"] == "Product"
    assert info["gpr_kernel_components"] == [["SquaredExponential", [2]], ["RationalQuadratic", []], ["Matern12", []]]
    loaded = GPRSurrogate.from_saved(str(tmp_path / "s"), backend=po.ProductOracleBackend())
    lk = loaded.gpflow_model.kernel
    assert isinstance(lk, gpmodel.Product)
    assert [type(k) for k in lk.kernels] == [gpmodel.SquaredExponential, gpmodel.RationalQuadratic, gpmodel.Matern12]
    assert loaded.gpflow_model._theta().tobytes() == surr.gpflow_model._theta().tobytes()
    p, q = surr.gpflow_model.predict_y(x), loaded.gpflow_model.predict_y(x)
    assert np.array_equal(p[0], q[0]) and np.array_equal(p[1], q[1])


@pytest.mark.parametrize("kind", ["Matern52", "Sum"])
def test_non_product_save_files_are_unchanged(tmp_path, kind):
    """A bare kernel's and a sum's saved info are the text the previous release wrote, byte for byte."""
    if kind == "Sum":
        kernel, be = gpmodel.SquaredExponential(lengthscales=0.5) + gpmodel.Matern12(lengthscales=0.1), so.SumOracleBackend()
        extra = {"gpr_kernel_components": [["SquaredExponential", []], ["Matern12", []]]}
    else:
        from tests.oracle_backend import OracleBackend

        kernel, be, extra = gpmodel.Matern52(lengthscales=0.25), OracleBackend(), {}
    surr, _ = _trained_surrogate(kernel, be)
    surr.save(str(tmp_path / "s"))
    with open(tmp_path / "s" / GPRSurrogate.GPR_INFO) as fh:
        text = fh.read()
    expected = json.dumps({
        "gpr_kernel": kind, "gpr_kernel_shape": [], "gpr_meanf": "Constant", "gpr_meanf_shape": [],
        "gp_varsigma": surr.gp_varsigma, "gp_likelihood": surr.gp_lik_sigma, "optimiser": ["Scipy"], **extra,
    })
    assert text == expected


def test_optimiser_runs_with_the_product_checker_backend():
    from tests.conftest import paper_objective

    opt = make_optimiser(backend=po.ProductOracleBackend(), depth=3, budget=40)
    opt.gp_surr.gp_kernel = gpmodel.SquaredExponential(lengthscales=0.5) * gpmodel.Matern32(lengthscales=0.8, variance=0.5)
    best = opt.run(paper_objective)
    k = opt.gp_surr.gpflow_model.kernel
    assert isinstance(k, gpmodel.Product) and type(opt.gp_surr.gpflow_model._session) is po.ProductOracleSession
    assert opt.n_eval_counter >= 40 and np.isfinite(best.score_mu)


# ---- fp32 screening covariance: |k32 - k64| <= 2e-6 var_prod, the rounding of the products included ---------------------
def _mixed_products():
    """Every multiset of 2..4 families, with short and long lengthscales."""
    out = []
    for n in (2, 3, 4):
        for combo in itertools.combinations_with_replacement(FAMILIES, n):
            for ls in (0.15, 0.5):
                out.append([po.Comp(f, ls * (1 + 0.3 * i), 0.5 + i, alpha=1.7 if f == rq.KERNEL else None)
                            for i, f in enumerate(combo)])
    return out


def test_cov32_of_mixed_products_within_the_screen_contract():
    rng = np.random.default_rng(3)
    d = 3
    Xa = rng.random((120, d))
    Xb = np.vstack([rng.random((200, d)), Xa[:40] + 1e-4 * rng.standard_normal((40, d)), Xa[:5]])
    worst = 0.0
    for comps in _mixed_products():
        h = po.ProductHyper(comps, 1e-3)
        k32 = po.cov32(h, Xa, Xb).astype(np.float64)
        k64 = po.kern(h, Xa, Xb)
        worst = max(worst, np.max(np.abs(k32 - k64)) / h.var_prod)
        assert np.all(np.diag(po.cov32(h, Xa[:5], Xa[:5])) == np.float32(h.var_prod))
        assert np.all(k64 >= 0.0) and np.all(k64 <= h.var_prod)   # each unit factor lies in [0, 1]
    # half the contract: MUFU.EX2 / RSQ / LG2 and __fdividef are not emulated (a few ulp each)
    assert worst <= 2e-6 / 2.0, worst


@pytest.mark.parametrize("case", ["rq_large_alpha", "var1e-8", "var1e8"])
def test_cov32_of_a_product_at_the_edges(case):
    comps = {
        "rq_large_alpha": [po.Comp(rq.KERNEL, 0.3, 1.0, alpha=1e4), po.Comp("Matern52", 0.3, 1.0), po.Comp("Matern32", 0.2, 1.0)],
        "var1e-8": [po.Comp(f, 0.4, 1e-2) for f in ("Matern52", "SquaredExponential", "Matern32", "Matern12")],
        "var1e8": [po.Comp(f, 0.4, 1e2) for f in ("Matern52", "SquaredExponential", "Matern32", "Matern12")],
    }[case]
    h = po.ProductHyper(comps, 1e-3)
    rng = np.random.default_rng(5)
    Xa = rng.random((200, 3))
    Xb = np.vstack([rng.random((300, 3)), Xa[:5]])
    err = np.max(np.abs(po.cov32(h, Xa, Xb).astype(np.float64) - po.kern(h, Xa, Xb)))
    assert err <= 2e-6 * h.var_prod / 2.0, err / h.var_prod


# ---- C argument checks that need no device ------------------------------------------------------------------------------
def test_create_product_rejects_bad_arguments():
    lib = backend.load_library()
    h = ctypes.c_void_p()

    def create(n, ids, ards, mean=1):
        k = (ctypes.c_int * max(len(ids), 1))(*ids)
        a = (ctypes.c_int * max(len(ards), 1))(*ards)
        return lib.gpso_create_product(0, n, k, a, mean, ctypes.byref(h))

    assert create(0, [], []) == -1   # GPSO_E_BADARG before any CUDA call
    assert b"gpso_create_product" in lib.gpso_last_error() and b"1..4" in lib.gpso_last_error()
    assert create(5, [0] * 5, [0] * 5) == -1
    assert create(2, [2, 7], [0, 0]) == -1
    assert b"kernel id" in lib.gpso_last_error()
    assert create(2, [2, 5], [0, 0]) == -1    # a sum is not a factor
    assert create(2, [2, 6], [0, 0]) == -1    # nor is a product
    assert create(2, [2, 3], [0, 2]) == -1
    assert b"ard" in lib.gpso_last_error()
    assert create(2, [2, 3], [0, 1], mean=3) == -1
    assert b"mean id" in lib.gpso_last_error()
    assert lib.gpso_create_product(0, 2, None, None, 1, ctypes.byref(h)) == -1
    assert b"null" in lib.gpso_last_error()
    for kid in (5, 6):   # the sum and product ids have components: gpso_create_sum / gpso_create_product
        assert lib.gpso_create(0, kid, 0, 1, ctypes.byref(h)) == -1
    assert not h.value
