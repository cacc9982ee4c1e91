"""GPU parity tests of the model-level path (GPR LML, SGPR ELBO, SVGP ELBO, posteriors, KL,
conditionals) against the CPU oracle and the committed golden fixtures, through the reference-shaped
Python API (which calls the C ABI)."""
import json
import os

import numpy as np
import pytest
from numpy.testing import assert_allclose

import gpflow_b200 as gpf
from gpflow_b200 import ops
from oracle import gp_oracle as O
from tests.golden.make_golden import c5_kernels, kernels_for
from tests.helpers import build, to_np

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))
GOLD = np.load(os.path.join(HERE, "golden", "golden_small.npz"))
F64 = dict(rtol=1e-8, atol=1e-8)


def product_kernel(c, D):
    s = np.sqrt(D)
    k = gpf.kernels
    return {1: lambda: k.RBF(variance=1.0, lengthscales=s), 2: lambda: k.Matern52(variance=1.0, lengthscales=s),
            3: lambda: k.RBF(variance=1.0, lengthscales=s),
            4: lambda: k.RBF(variance=1.0, lengthscales=s) + k.White(variance=0.1)}[c]()


def product_c5_kernels(D, P=4):
    s = np.sqrt(D)
    k = gpf.kernels
    return [(k.RBF(variance=1.0 + 0.1 * p, lengthscales=s * (1 + 0.05 * p)) + k.Matern32(variance=1.0, lengthscales=2 * s))
            * k.Linear(variance=1.0 / (1 + p)) for p in range(P)]


# ---- GPR --------------------------------------------------------------------------------------------
def test_c1_gpr_rbf_lml_and_predict_golden(cuda_device):
    """BASELINE config 1: GPR RBF fp64 N=512 D=2."""
    d = O.make_data(1, 512, 2, 1, n_new=64)
    m = gpf.models.GPR((d["X"], d["Y"]), product_kernel(1, 2), noise_variance=0.1)
    lml = float(m.log_marginal_likelihood())
    assert_allclose(lml, float(GOLD["c1_lml"]), rtol=1e-10)
    assert_allclose(lml, O.gpr_log_marginal_likelihood(d["X"], d["Y"], kernels_for(1, 2), 0.1), rtol=1e-10)
    assert m.cholesky_info() == 0
    mean, var = m.predict_f(d["Xnew"])
    assert_allclose(to_np(mean), GOLD["c1_mean"], **F64)
    assert_allclose(to_np(var), GOLD["c1_var"], **F64)
    assert_allclose(float(m.training_loss()), -lml, rtol=1e-12)
    assert float(m.training_loss_closure()()) == pytest.approx(-lml, rel=1e-12)


def test_c2_reduced_gpr_matern52_golden(cuda_device):
    d = O.make_data(2, 1024, 8, 1, n_new=32)
    m = gpf.models.GPR((d["X"], d["Y"]), product_kernel(2, 8), noise_variance=0.1)
    assert_allclose(float(m.log_marginal_likelihood()), float(GOLD["c2_lml"]), rtol=1e-9)
    mean, var = m.predict_f(d["Xnew"])
    assert_allclose(to_np(mean), GOLD["c2_mean"], **F64)
    assert_allclose(to_np(var), GOLD["c2_var"], **F64)
    post = m.posterior()                      # cached: posteriors.py:322-358
    m2, v2 = post.predict_f(d["Xnew"])
    assert_allclose(to_np(m2), to_np(mean), rtol=1e-12, atol=1e-13)
    assert_allclose(to_np(v2), to_np(var), rtol=1e-12, atol=1e-13)
    mf, vf = m.predict_f(d["Xnew"], full_cov=True)
    mo, vo = O.gpr_predict_f(d["X"], d["Y"], kernels_for(2, 8), 0.1, d["Xnew"], full_cov=True)
    assert_allclose(to_np(vf), vo, **F64)
    assert_allclose(np.diagonal(to_np(vf)[0]), to_np(var)[:, 0], rtol=1e-8, atol=1e-10)  # test_model_predict.py:137-153
    my, vy = m.predict_y(d["Xnew"])
    assert_allclose(to_np(vy), to_np(var) + 0.1, rtol=1e-12)
    # predictive log density on the device (models/model.py:332-343, scalar_continuous.py:133-136;
    # the reference checks it by hand in tests/gpflow/models/test_model_predict.py:119-135)
    Ynew = np.sin(d["Xnew"][:, :1]) + 0.05
    lpd = m.predict_log_density((d["Xnew"], Ynew))
    assert lpd.is_cuda and tuple(lpd.shape) == (32,)
    mo1, vo1 = O.gpr_predict_f(d["X"], d["Y"], kernels_for(2, 8), 0.1, d["Xnew"])
    assert_allclose(to_np(lpd), O.gaussian_predict_log_density(mo1, vo1, Ynew, 0.1), rtol=1e-9, atol=1e-11)
    with pytest.raises(NotImplementedError):
        m.predict_f(d["Xnew"], full_output_cov=True)


@pytest.mark.parametrize("N,P", [(1, 1), (7, 2), (128, 1), (129, 3), (777, 2)])
def test_gpr_lml_sizes_multi_output_and_mean_function(cuda_device, N, P):
    rng = np.random.default_rng(N)
    D = 3
    X, Y = rng.standard_normal((N, D)), rng.standard_normal((N, P))
    ko, kp = build(("sum", "m32", ("prod", "rbf", "lin")), D, [O, gpf.kernels])
    A, b = rng.standard_normal((D, P)), rng.standard_normal(P)
    m = gpf.models.GPR((X, Y), kp, mean_function=gpf.mean_functions.Linear(A, b), noise_variance=0.3)
    ref = O.gpr_log_marginal_likelihood(X, Y, ko, 0.3, O.LinearMean(A, b))
    assert_allclose(float(m.log_marginal_likelihood()), ref, rtol=1e-9)
    Xn = rng.standard_normal((5, D))
    mean, var = m.predict_f(Xn)
    mo, vo = O.gpr_predict_f(X, Y, ko, 0.3, Xn, O.LinearMean(A, b))
    assert_allclose(to_np(mean), mo, **F64)
    assert_allclose(to_np(var), vo, **F64)


def test_gpr_fp32_within_1e3(cuda_device):
    d = O.make_data(2, 1500, 8, 1)
    with gpf.config.as_context(gpf.config.Config(float=np.float32)):
        m = gpf.models.GPR((d["X"], d["Y"]), product_kernel(2, 8), noise_variance=0.1)
        lml = float(m.log_marginal_likelihood())
    ref = O.gpr_log_marginal_likelihood(d["X"], d["Y"], kernels_for(2, 8), 0.1)
    assert_allclose(lml, ref, rtol=1e-3)


def test_gpr_default_noise_and_not_pd(cuda_device):
    rng = np.random.default_rng(0)
    X, Y = rng.standard_normal((50, 2)), rng.standard_normal((50, 1))
    m = gpf.models.GPR((X, Y), gpf.kernels.RBF())
    assert float(m.likelihood.variance.numpy()) == 1.0  # gpr.py:75-78
    assert_allclose(float(m.log_marginal_likelihood()), O.gpr_log_marginal_likelihood(X, Y, O.RBF(), 1.0), rtol=1e-10)
    Xd = np.concatenate([X, X])  # duplicated inputs with tiny noise: numerically singular
    m = gpf.models.GPR((Xd, np.concatenate([Y, Y])), gpf.kernels.RBF(), likelihood=gpf.likelihoods.Gaussian(2e-6, variance_lower_bound=1e-6))
    # numerically singular but still positive definite in fp64 (pivots ~ 2 * 2e-6): evaluates, like LAPACK; the truly
    # non-positive-definite case (exception on the host read) is tests/test_gpu_edge.py
    assert np.isfinite(float(m.log_marginal_likelihood()))
    assert m.cholesky_info() == 0


def test_c5_reduced_separate_outputs_golden(cuda_device):
    d = O.make_data(5, 512, 32, 4)
    ks = product_c5_kernels(32)
    total = sum(float(gpf.models.GPR((d["X"], d["Y"][:, p:p + 1]), ks[p], noise_variance=0.1).log_marginal_likelihood())
                for p in range(4))
    assert_allclose(total, float(GOLD["c5_lml"]), rtol=1e-9)


# ---- SGPR -------------------------------------------------------------------------------------------
def test_c3_reduced_sgpr_elbo_and_predict_golden(cuda_device):
    gpf.config.set_default_jitter(1e-4)
    try:
        d = O.make_data(3, 5000, 16, 1, M=256, n_new=100)
        m = gpf.models.SGPR((d["X"], d["Y"]), product_kernel(3, 16), d["Z"], noise_variance=0.1)
        assert_allclose(float(m.elbo()), float(GOLD["c3_elbo_f64"]), rtol=1e-8)
        c, ld, q = (float(t) for t in m.elbo_terms())
        assert_allclose(c + ld + q, float(GOLD["c3_elbo_f64"]), rtol=1e-8)
        mean, var = m.predict_f(d["Xnew"])
        assert_allclose(to_np(mean), GOLD["c3_mean_f64"], rtol=1e-6, atol=1e-7)
        assert_allclose(to_np(var), GOLD["c3_var_f64"], rtol=1e-6, atol=1e-7)
        post = m.posterior()
        m2, v2 = post.predict_f(d["Xnew"])
        assert_allclose(to_np(m2), to_np(mean), rtol=1e-10, atol=1e-12)
        with gpf.config.as_context(gpf.config.Config(float=np.float32, jitter=1e-4)):   # the fp32 config proper
            m32 = gpf.models.SGPR((d["X"], d["Y"]), product_kernel(3, 16), d["Z"], noise_variance=0.1)
            assert_allclose(float(m32.elbo()), float(GOLD["c3_elbo_f64"]), rtol=1e-3)
            mean32, var32 = m32.predict_f(d["Xnew"])
            assert_allclose(to_np(mean32), GOLD["c3_mean_f64"], rtol=1e-3, atol=1e-3)
            assert_allclose(to_np(var32), GOLD["c3_var_f64"], rtol=1e-3, atol=1e-3)
    finally:
        gpf.config.set_default_jitter(1e-6)


def test_sgpr_multi_output_mean_function_full_cov(cuda_device):
    rng = np.random.default_rng(1)
    X, Y, Z, Xn = rng.standard_normal((300, 2)), rng.standard_normal((300, 2)), rng.standard_normal((37, 2)), rng.standard_normal((9, 2))
    ko, kp = build(("sum", "m52", "white"), 2, [O, gpf.kernels])
    mf_o, mf_p = O.ConstantMean([0.3, -0.2]), gpf.mean_functions.Constant([0.3, -0.2])
    m = gpf.models.SGPR((X, Y), kp, Z, mean_function=mf_p, noise_variance=0.2)
    assert_allclose(float(m.elbo()), O.sgpr_elbo(X, Y, ko, Z, 0.2, mf_o), rtol=1e-9)
    mean, var = m.predict_f(Xn, full_cov=True)
    mo, vo = O.sgpr_predict_f(X, Y, ko, Z, 0.2, Xn, mf_o, full_cov=True)
    assert_allclose(to_np(mean), mo, **F64)
    assert_allclose(to_np(var), vo, rtol=1e-7, atol=1e-8)
    mu, cov = m.compute_qu()
    muo, covo = O.sgpr_compute_qu(X, Y, ko, Z, 0.2, mf_o)
    assert_allclose(to_np(mu), muo, rtol=1e-6, atol=1e-8)
    assert_allclose(to_np(cov), covo, rtol=1e-6, atol=1e-8)
    common = m._common_calculation()
    co = O.sgpr_common(X, ko, Z, 0.2)
    assert_allclose(to_np(common.A), co.A, rtol=1e-7, atol=1e-9)
    assert_allclose(to_np(common.LB), co.LB, rtol=1e-7, atol=1e-9)


def test_sgpr_upper_bound_vs_oracle_and_brackets_gpr(cuda_device):
    """SGPR.upper_bound (sgpr.py:87-147): parity with the oracle, and the reference's own check
    elbo < GPR lml < upper_bound (tests/integration/test_method_equivalence.py:297-327) on its DatumUpper data."""
    rng = np.random.default_rng(123)
    X = rng.random((100, 1))
    Y = np.sin(1.5 * 2 * np.pi * X) + rng.standard_normal(X.shape) * 0.1 + 5.3
    Z = X[:10].copy()
    ko, kp = O.SquaredExponential(variance=1.3, lengthscales=0.3), gpf.kernels.SquaredExponential(variance=1.3, lengthscales=0.3)
    mf_o, mf_p = O.ConstantMean([5.0]), gpf.mean_functions.Constant([5.0])
    m = gpf.models.SGPR((X, Y), kp, Z, mean_function=mf_p, noise_variance=0.05)
    ub, elbo = float(m.upper_bound()), float(m.elbo())
    assert_allclose(ub, O.sgpr_upper_bound(X, Y, ko, Z, 0.05, mf_o), rtol=1e-9)
    lml = float(gpf.models.GPR((X, Y), kp, mean_function=mf_p, noise_variance=0.05).log_marginal_likelihood())
    assert elbo < lml < ub
    # two outputs, larger M (two diagonal blocks in each factorisation)
    X2, Y2, Z2 = rng.standard_normal((400, 3)), rng.standard_normal((400, 2)), rng.standard_normal((150, 3))
    ko2, kp2 = build("m32", 3, [O, gpf.kernels])
    m2 = gpf.models.SGPR((X2, Y2), kp2, Z2, noise_variance=0.3)
    assert_allclose(float(m2.upper_bound()), O.sgpr_upper_bound(X2, Y2, ko2, Z2, 0.3), rtol=1e-9)


@pytest.mark.parametrize("N,P", [(60, 1), (200, 2)])
def test_vgp_elbo_and_predict_vs_oracle(cuda_device, N, P):
    """VGP with a Gaussian likelihood (vgp.py:111-161) against the oracle; with q set to the exact whitened posterior
    the ELBO equals the GPR log marginal likelihood (the fixed point test_method_equivalence.py reaches by training)."""
    rng = np.random.default_rng(N + P)
    X, Xn = rng.standard_normal((N, 2)), rng.standard_normal((11, 2))
    Y = np.sin(X[:, :1]) + 0.1 * rng.standard_normal((N, P))
    ko, kp = build("m32", 2, [O, gpf.kernels])
    q_mu = 0.3 * rng.standard_normal((N, P))
    q_sqrt = np.stack([np.tril(0.1 * rng.standard_normal((N, N))) + np.eye(N) for _ in range(P)])
    mf_o, mf_p = O.ConstantMean([0.2] * P), gpf.mean_functions.Constant([0.2] * P)
    m = gpf.models.VGP((X, Y), kp, gpf.likelihoods.Gaussian(0.2), mean_function=mf_p)
    m.q_mu.assign(q_mu)
    m.q_sqrt.assign(q_sqrt)
    assert_allclose(float(m.elbo()), O.vgp_elbo(X, Y, ko, q_mu, q_sqrt, 0.2, mf_o), rtol=1e-9)
    assert_allclose(float(m.training_loss()), -float(m.elbo()), rtol=1e-12)
    mean, var = m.predict_f(Xn)
    mo, vo = O.vgp_predict_f(X, ko, q_mu, q_sqrt, Xn, mf_o)
    assert_allclose(to_np(mean), mo, **F64)
    assert_allclose(to_np(var), vo, **F64)
    mf, vf = m.predict_f(Xn, full_cov=True)
    mo2, vo2 = O.vgp_predict_f(X, ko, q_mu, q_sqrt, Xn, mf_o, full_cov=True)
    assert_allclose(to_np(vf), vo2, rtol=1e-7, atol=1e-8)
    if P == 1:  # exact posterior in whitened coordinates  =>  ELBO == GPR LML (jitter aside)
        s2 = 0.2
        K = ko(X) + 1e-6 * np.eye(N)
        L = np.linalg.cholesky(K)
        Ky = K + s2 * np.eye(N)
        mu = K @ np.linalg.solve(Ky, Y - 0.2)
        S = K - K @ np.linalg.solve(Ky, K)
        m.q_mu.assign(np.linalg.solve(L, mu))
        m.q_sqrt.assign(np.linalg.solve(L, np.linalg.cholesky(S + 1e-12 * np.eye(N)))[None])
        lml = float(gpf.models.GPR((X, Y), kp, mean_function=mf_p, noise_variance=s2).log_marginal_likelihood())
        assert_allclose(float(m.elbo()), lml, rtol=1e-5)


def test_method_equivalence_on_device(cuda_device):
    """tests/integration/test_method_equivalence.py:181-241 at fixed hyper-parameters, on the GPU path."""
    rng = np.random.RandomState(0)
    X = rng.rand(20, 1) * 10
    Y = np.tile(np.sin(X) + 0.9 * np.cos(X * 1.6) + rng.randn(*X.shape) * 0.8, 2)
    Xt = rng.rand(10, 1) * 10
    mk = lambda: gpf.kernels.RBF(variance=1.3, lengthscales=1.7)
    gpr = gpf.models.GPR((X, Y), mk(), noise_variance=0.4)
    sgpr = gpf.models.SGPR((X, Y), mk(), X.copy(), noise_variance=0.4)
    lml, elbo = float(gpr.log_marginal_likelihood()), float(sgpr.elbo())
    assert_allclose(elbo, lml, rtol=1e-5)
    assert elbo <= lml + 1e-9
    mu, cov = sgpr.compute_qu()
    q_sqrt = np.tile(np.linalg.cholesky(to_np(cov) + 1e-12 * np.eye(20))[None], (2, 1, 1))
    svgp = gpf.models.SVGP(mk(), gpf.likelihoods.Gaussian(0.4), X.copy(), q_mu=to_np(mu), q_sqrt=q_sqrt, whiten=False)
    assert_allclose(float(svgp.elbo((X, Y))), elbo, rtol=1e-4)
    mg, vg = gpr.predict_f(Xt)
    for model in (sgpr, svgp):
        mm, vv = model.predict_f(Xt)
        assert_allclose(to_np(mm), to_np(mg), rtol=1e-3, atol=1e-4)
        assert_allclose(to_np(vv), to_np(vg), rtol=1e-3, atol=1e-4)


# ---- SVGP -------------------------------------------------------------------------------------------
@pytest.mark.parametrize("whiten", [True, False])
def test_c4_reduced_svgp_elbo_golden(cuda_device, whiten):
    gpf.config.set_default_jitter(1e-4)
    try:
        d = O.make_data(4, 20000, 16, 4, M=128)
        q_mu, q_sqrt = O.make_q(4, 128, 4)
        Xb, Yb = d["X"][:512], d["Y"][:512]
        m = gpf.models.SVGP(product_kernel(4, 16), gpf.likelihoods.Gaussian(0.1), d["Z"], num_latent_gps=4, q_mu=q_mu,
                            q_sqrt=q_sqrt, whiten=whiten, num_data=20000)
        gold = float(GOLD["c4_elbo_f64" if whiten else "c4_elbo_nowhite_f64"])
        assert_allclose(float(m.elbo((Xb, Yb))), gold, rtol=1e-8)
        assert_allclose(float(m.elbo_unfused((Xb, Yb))), gold, rtol=1e-8)        # operator-by-operator path
        # latent sharding (SURVEY 8(e)): the shares of disjoint latent ranges sum to the ELBO
        parts = [float(m.elbo((Xb, Yb), latent_range=r)) for r in [(0, 1), (1, 3), (3, 4)]]
        assert_allclose(sum(parts), gold, rtol=1e-8)
        with gpf.config.as_context(gpf.config.Config(float=np.float32, jitter=1e-4)):
            m32 = gpf.models.SVGP(product_kernel(4, 16), gpf.likelihoods.Gaussian(0.1), d["Z"], num_latent_gps=4,
                                  q_mu=q_mu, q_sqrt=q_sqrt, whiten=whiten, num_data=20000)
            assert_allclose(float(m32.elbo((Xb, Yb))), gold, rtol=1e-3)
    finally:
        gpf.config.set_default_jitter(1e-6)


@pytest.mark.parametrize("whiten", [True, False])
@pytest.mark.parametrize("q_diag", [True, False])
def test_svgp_elbo_predict_kl_vs_oracle(cuda_device, whiten, q_diag):
    rng = np.random.default_rng(3)
    N, M, P, D = 200, 45, 3, 2
    X, Y, Z, Xn = rng.standard_normal((N, D)), rng.standard_normal((N, P)), rng.standard_normal((M, D)), rng.standard_normal((11, D))
    ko, kp = build(("sum", "m32", "white"), D, [O, gpf.kernels])
    q_mu = rng.standard_normal((M, P))
    q_sqrt = (rng.random((M, P)) + 0.2) if q_diag else np.stack([np.tril(rng.standard_normal((M, M))) * 0.2 + np.eye(M) for _ in range(P)])
    m = gpf.models.SVGP(kp, gpf.likelihoods.Gaussian(0.3), Z, num_latent_gps=P, q_diag=q_diag, q_mu=q_mu, q_sqrt=q_sqrt,
                        whiten=whiten, num_data=1000)
    ref = O.svgp_elbo(X, Y, Z, ko, q_mu, q_sqrt, 0.3, whiten=whiten, num_data=1000)
    assert_allclose(float(m.elbo((X, Y))), ref, rtol=1e-9)
    assert_allclose(float(m.elbo_unfused((X, Y))), ref, rtol=1e-9)
    assert_allclose(float(m.prior_kl()), O.prior_kl(Z, ko, q_mu, q_sqrt, whiten=whiten), rtol=1e-9)
    for full_cov in (False, True):
        mean, var = m.predict_f(Xn, full_cov=full_cov)
        mo, vo = O.svgp_predict_f(Xn, Z, ko, q_mu, q_sqrt, whiten=whiten, full_cov=full_cov)
        assert_allclose(to_np(mean), mo, **F64)
        assert_allclose(to_np(var), vo, rtol=1e-7, atol=1e-8)
    post = m.posterior()                                  # cached alpha / Qinv, posteriors.py:694-822
    mc, vc = post.predict_f(Xn)
    mo, vo = O.svgp_predict_f(Xn, Z, ko, q_mu, q_sqrt, whiten=whiten)
    assert_allclose(to_np(mc), mo, rtol=1e-7, atol=1e-8)
    assert_allclose(to_np(vc), vo, rtol=1e-6, atol=1e-7)
    # external-data closure with an iterator (training_mixins.py:127-137)
    it = iter([(X[:50], Y[:50]), (X[50:100], Y[50:100])])
    closure = m.training_loss_closure(it)
    l1, l2 = float(closure()), float(closure())
    assert_allclose(l1, -O.svgp_elbo(X[:50], Y[:50], Z, ko, q_mu, q_sqrt, 0.3, whiten=whiten, num_data=1000), rtol=1e-9)
    assert l1 != l2


def test_gauss_kl_variants_vs_oracle(cuda_device):
    rng = np.random.RandomState(0)
    M, L = 5, 4
    mu = rng.randn(M, L)
    A = rng.randn(M, M)
    K = A @ A.T + 1e-6 * np.eye(M)
    sq = np.array([np.tril(rng.randn(M, M)) for _ in range(L)])
    sqd = rng.randn(M, L)
    Kb = rng.randn(L, M, M)
    Kb = 0.1 * (Kb + Kb.transpose(0, 2, 1)) + np.eye(M)[None]
    kl = gpf.kullback_leiblers.gauss_kl
    for qs in (sq, sqd):
        for Kc in (None, K, Kb):
            assert_allclose(float(kl(mu, qs, Kc)), O.gauss_kl(mu, qs, Kc), rtol=1e-7, err_msg=f"{qs.ndim} {None if Kc is None else Kc.ndim}")
        assert_allclose(float(kl(mu, qs, K_cholesky=np.linalg.cholesky(K))), O.gauss_kl(mu, qs, K), rtol=1e-7)
    with pytest.raises(ValueError):
        kl(mu, sq, K, K_cholesky=K)


def test_conditional_and_base_conditional_vs_explicit_inverse(cuda_device):
    """tests/gpflow/conditionals/test_conditionals.py:168-214 on the device path."""
    rng = np.random.RandomState(123)
    Dy, N, M, Dx = 5, 4, 3, 2
    X, Z = rng.randn(N, Dx), rng.randn(M, Dx)
    q_mu = rng.randn(M, Dy)
    q_sqrt = np.tril(rng.randn(Dy, M, M), -1)
    ko = O.Matern52(lengthscales=0.5)
    Kmm = ko(Z, Z) + np.eye(M) * 1e-6
    Kmn, Knn = ko(Z, X), ko(X, X)
    S = q_sqrt @ q_sqrt.transpose(0, 2, 1)
    Ki = np.linalg.inv(Kmm)
    mean_np = Kmn.T @ Ki @ q_mu
    cov_np = Knn[None] + Kmn.T[None] @ Ki[None] @ (S - Kmm[None]) @ Ki[None] @ Kmn[None]
    kp = gpf.kernels.Matern52(lengthscales=0.5)
    for full_cov in (True, False):
        for iv in (Z, gpf.inducing_variables.InducingPoints(Z)):
            mean, cov = gpf.conditionals.conditional(X, iv, kp, q_mu, q_sqrt=q_sqrt, white=False, full_cov=full_cov)
            ref = cov_np if full_cov else np.diagonal(cov_np, axis1=-1, axis2=-2).T
            assert_allclose(to_np(mean), mean_np, rtol=1e-6, atol=1e-9)
            assert_allclose(to_np(cov), ref, rtol=1e-6, atol=1e-9)
    m2, v2 = gpf.conditionals.base_conditional(Kmn, Kmm, np.diag(Knn).copy(), q_mu, q_sqrt=q_sqrt, white=False)
    assert_allclose(to_np(m2), mean_np, rtol=1e-6, atol=1e-9)


def test_kuu_kuf_and_logdensity(cuda_device):
    rng = np.random.default_rng(5)
    Z, X = rng.standard_normal((30, 3)), rng.standard_normal((50, 3))
    ko, kp = build(("sum", "rbf", "white"), 3, [O, gpf.kernels])
    iv = gpf.inducing_variables.InducingPoints(Z)
    assert_allclose(to_np(gpf.covariances.Kuu(iv, kp, jitter=1e-3)), O.Kuu(Z, ko, jitter=1e-3), rtol=1e-12)
    assert_allclose(to_np(gpf.covariances.Kuf(iv, kp, X)), O.Kuf(Z, ko, X), rtol=1e-12, atol=1e-14)
    # Schur complement PSD (tests/gpflow/covariances/test_base_covariances.py:99-109)
    Kuu, Kuf, Kff = (to_np(gpf.covariances.Kuu(iv, kp, jitter=1e-6)), to_np(gpf.covariances.Kuf(iv, kp, X)), to_np(kp(X)))
    assert np.linalg.eigvalsh(Kff - Kuf.T @ np.linalg.solve(Kuu, Kuf)).min() > -1e-8
    x, mu = rng.standard_normal((30, 4)), rng.standard_normal((30, 4))
    L = np.linalg.cholesky(O.Kuu(Z, ko, jitter=1e-3))
    assert_allclose(to_np(gpf.logdensities.multivariate_normal(x, mu, L)), O.multivariate_normal(x, mu, L), rtol=1e-10)


# ---- full-size property checks (BASELINE sizes; no oracle run on the GPU box) ----------------------
def test_c2_full_size_lml_golden_scalar(cuda_device):
    path = os.path.join(HERE, "golden", "golden_full.json")
    if not os.path.exists(path):
        pytest.skip("golden_full.json not generated")
    gold = json.load(open(path))
    d = O.make_data(2, 8192, 8, 1)
    m = gpf.models.GPR((d["X"], d["Y"]), product_kernel(2, 8), noise_variance=0.1)
    assert_allclose(float(m.log_marginal_likelihood()), gold["c2_lml_N8192_D8_f64"], rtol=1e-5)


def test_c2_full_size_factor_residual(cuda_device):
    """Size-independent property at BASELINE size: ||L L^T - K||_F / ||K||_F and the log-det identity."""
    T = ops.torch()
    d = O.make_data(2, 8192, 8, 1)
    kp = product_kernel(2, 8)
    Xd = ops.to_device(d["X"])
    K = kp(Xd)
    ops.add_diag_(K, 0.1)
    L, _ = ops.cholesky(K)
    # residual through our own GEMM: R = K - L L^T
    R = ops.copy(K)
    ops.gemm(L, L, transb=True, alpha=-1.0, beta=1.0, out=R)
    num = float(ops.reduce(ops.SUMSQ, R, R.numel())) ** 0.5
    den = float(ops.reduce(ops.SUMSQ, K, K.numel())) ** 0.5
    # digit planes with STATIC row scales 2^ceil(log2 sqrt(K_ii)) (csrc/planes.cuh): rows of L are usually well below
    # sqrt(K_ii), so a few leading digit bits are unused -- measured 6e-13 here (4e-14 with per-update row maxima);
    # the parity bar on the objective is 1e-5
    assert num / den < 3e-12


def _gold_full():
    path = os.path.join(HERE, "golden", "golden_full.json")
    if not os.path.exists(path):
        pytest.skip("golden_full.json not generated")
    return json.load(open(path))


def test_c3_full_size_sgpr_elbo_golden(cuda_device):
    """BASELINE config 3 at full size (N=100000, M=1024, D=16): fp32 within 1e-3 and fp64 within 1e-8 of the
    fp64 golden scalar."""
    gold = _gold_full()["c3_elbo_N100000_M1024_D16_f64_jitter1e-4"]
    d = O.make_data(3, 100000, 16, 1, M=1024)
    with gpf.config.as_context(gpf.config.Config(float=np.float32, jitter=1e-4)):
        m = gpf.models.SGPR((d["X"], d["Y"]), product_kernel(3, 16), d["Z"], noise_variance=0.1)
        assert_allclose(float(m.elbo()), gold, rtol=1e-3)
    with gpf.config.as_context(gpf.config.Config(float=np.float64, jitter=1e-4)):
        m = gpf.models.SGPR((d["X"], d["Y"]), product_kernel(3, 16), d["Z"], noise_variance=0.1)
        assert_allclose(float(m.elbo()), gold, rtol=1e-8)


def test_c3_full_size_sgpr_predict_golden(cuda_device):
    """BASELINE config 3 "posterior predict" at full size: SGPR.predict_f at Xnew [10000, 16] (N = 100000, M = 1024) against
    the fp64 oracle fixture (tests/golden/golden_c3_predict.npz: first 256 rows + sums over all rows); fp32 within 1e-3 of
    the prior variance, fp64 within 1e-6.  Reference: gpflow/posteriors.py:479-551."""
    import os
    g = np.load(os.path.join(os.path.dirname(__file__), "golden", "golden_c3_predict.npz"))
    d = O.make_data(3, 100000, 16, 1, M=1024, n_new=10000)
    for dt, tol in ((np.float32, 1e-3), (np.float64, 1e-6)):
        with gpf.config.as_context(gpf.config.Config(float=dt, jitter=1e-4)):
            m = gpf.models.SGPR((d["X"], d["Y"]), product_kernel(3, 16), d["Z"], noise_variance=0.1)
            mean, var = m.predict_f(d["Xnew"])
        mean, var = mean.cpu().numpy().astype(np.float64), var.cpu().numpy().astype(np.float64)
        assert mean.shape == (10000, 1) and var.shape == (10000, 1)
        assert_allclose(mean[:256], g["mean"], rtol=tol, atol=tol)
        assert_allclose(var[:256], g["var"], rtol=tol, atol=tol)
        assert_allclose(mean.sum(), float(g["mean_sum"]), atol=tol * float(g["mean_abs_sum"]))
        assert_allclose(var.sum(), float(g["var_sum"]), rtol=tol)


def test_c4_full_size_svgp_elbo_golden(cuda_device):
    """BASELINE config 4 at full size (B=4096, M=2048, P=8, D=16, num_data=1e6), first minibatch."""
    gold = _gold_full()["c4_elbo_N1e6_B4096_M2048_P8_D16_f64_jitter1e-4_batch0"]
    d = O.make_data(4, 1000000, 16, 8, M=2048)
    q_mu, q_sqrt = O.make_q(4, 2048, 8)
    Xb, Yb = d["X"][:4096], d["Y"][:4096]
    for dtype, rtol in ((np.float32, 1e-3), (np.float64, 1e-8)):
        with gpf.config.as_context(gpf.config.Config(float=dtype, jitter=1e-4)):
            m = gpf.models.SVGP(product_kernel(4, 16), gpf.likelihoods.Gaussian(0.1), d["Z"], num_latent_gps=8, q_mu=q_mu,
                                q_sqrt=q_sqrt, whiten=True, num_data=1000000)
            assert_allclose(float(m.elbo((Xb, Yb))), gold, rtol=rtol)
            if dtype == np.float64:  # latent sharding over 8 "GPUs" at full size
                parts = [float(m.elbo((Xb, Yb), latent_range=(p, p + 1))) for p in range(8)]
                assert_allclose(sum(parts), gold, rtol=1e-8)


def test_c5_full_size_multi_output_lml_golden(cuda_device):
    gold = _gold_full()["c5_lml_N4096_D32_P4_f64"]
    d = O.make_data(5, 4096, 32, 4)
    ks = product_c5_kernels(32)
    total = sum(float(gpf.models.GPR((d["X"], d["Y"][:, p:p + 1]), ks[p], noise_variance=0.1).log_marginal_likelihood())
                for p in range(4))
    assert_allclose(total, gold, rtol=1e-8)
