"""Device backward pass of the SGPR ELBO (csrc/grad.cu, gpk_sgpr_elbo_grad) against the gradient oracle
(tests/sgpr_grad_oracle.py, pinned by finite differences in tests/test_oracle_sgpr_grad.py), against finite differences
of the device ELBO at BASELINE configs[2] size, and driving the Scipy optimiser.
Reference: TensorFlow autodiff through gpflow/models/sgpr.py:181-289, driven by gpflow/optimizers/scipy.py:78-228."""
import numpy as np
import pytest

import gpflow_b200 as gpf
from gpflow_b200 import ops
from oracle import gp_oracle as O
from tests import sgpr_grad_oracle as SG

pytestmark = pytest.mark.gpu

KERNELS = ["SquaredExponential", "Matern12", "Matern32", "Matern52", "Exponential"]


def _check(m, X, Y, Z, ko, s2, rtol, jitter=1e-6, mean=None):
    """Device gradients against the oracle; tolerance rtol with an absolute floor of rtol x the largest |gradient| of
    each group (kernel / noise parameters, inducing points)."""
    elbo, g = m.elbo_and_grad()
    ref_elbo, ref = SG.sgpr_elbo_and_grad(X, Y, ko, Z, s2, mean_function=mean, jitter=jitter)
    np.testing.assert_allclose(float(elbo), ref_elbo, rtol=max(rtol, 1e-9))
    k = m.kernel
    scale = max(abs(ref["variance"]), np.max(np.abs(ref["lengthscales"])), abs(ref["noise_variance"]))
    np.testing.assert_allclose(float(g[k.variance]), ref["variance"], rtol=rtol, atol=rtol * scale)
    np.testing.assert_allclose(np.asarray(g[k.lengthscales]), ref["lengthscales"], rtol=rtol, atol=rtol * scale)
    np.testing.assert_allclose(float(g[m.likelihood.variance]), ref["noise_variance"], rtol=rtol, atol=rtol * scale)
    zs = np.max(np.abs(ref["Z"]))
    np.testing.assert_allclose(g[m.inducing_variable.Z], ref["Z"], rtol=rtol, atol=rtol * zs)
    return g, ref


# (N, M, D, P, lengthscale mode): M = 130 and 300 cross the 128-block boundaries of the inverse recursion
CASES = [(600, 40, 3, 1, "scalar"), (1500, 130, 5, 2, "ard"), (3000, 300, 4, 1, "active")]


@pytest.mark.parametrize("name", KERNELS)
@pytest.mark.parametrize("N,M,D,P,mode", CASES)
def test_sgpr_grad_fp64_matches_oracle(cuda_device, name, N, M, D, P, mode):
    d = O.make_data(6, N, D, P, M=M)            # Z: a random subset of X (well spread, Kuu well conditioned)
    kw = {"variance": 1.2}
    if mode == "scalar":
        kw["lengthscales"] = 1.4
    elif mode == "ard":
        kw["lengthscales"] = np.linspace(0.9, 2.2, D)
    else:
        kw["lengthscales"], kw["active_dims"] = np.array([1.1, 1.8, 0.9]), [0, 2, 3]
    kp, ko = getattr(gpf.kernels, name)(**kw), getattr(O, name)(**kw)
    m = gpf.models.SGPR((d["X"], d["Y"]), kp, d["Z"], noise_variance=0.2)
    g, _ = _check(m, d["X"], d["Y"], d["Z"], ko, 0.2, 1e-6)
    if mode == "active":
        assert np.all(g[m.inducing_variable.Z][:, 1] == 0.0)


def test_sgpr_grad_fp64_constant_mean(cuda_device):
    """A (fixed) Constant mean function shifts E = Y - m(X) in every term of the gradient."""
    d = O.make_data(7, 900, 3, 2, M=60)
    mo, mp = O.ConstantMean([0.3, -0.2]), gpf.mean_functions.Constant([0.3, -0.2])
    mp.c.trainable = False
    m = gpf.models.SGPR((d["X"], d["Y"]), gpf.kernels.Matern32(lengthscales=1.3), d["Z"], mean_function=mp,
                        noise_variance=0.15)
    _check(m, d["X"], d["Y"], d["Z"], O.Matern32(lengthscales=1.3), 0.15, 1e-6, mean=mo)
    m.training_loss_and_gradients()   # every trainable parameter has a gradient


def test_sgpr_grad_fp32_reduced_c3(cuda_device):
    """BASELINE configs[2] (SGPR RBF, D = 16) at reduced size in float32 against the float64 oracle: within 1e-3 of each
    group's largest gradient, the project's fp32 bar."""
    d = O.make_data(3, 8000, 16, 1, M=256)
    s = float(np.sqrt(16.0))
    with gpf.config.as_context(gpf.config.Config(float=np.float32, jitter=1e-4)):
        m = gpf.models.SGPR((d["X"].astype(np.float32), d["Y"].astype(np.float32)),
                            gpf.kernels.SquaredExponential(lengthscales=s), d["Z"].astype(np.float32), noise_variance=0.1)
        elbo, g = m.elbo_and_grad()
    X, Y, Z = (d[k].astype(np.float32).astype(np.float64) for k in ("X", "Y", "Z"))
    ref_elbo, ref = SG.sgpr_elbo_and_grad(X, Y, O.SquaredExponential(lengthscales=s), Z, 0.1, jitter=1e-4)
    np.testing.assert_allclose(float(elbo), ref_elbo, rtol=1e-3)
    scale = max(abs(ref["variance"]), abs(ref["lengthscales"]), abs(ref["noise_variance"]))
    for p, key in ((m.kernel.variance, "variance"), (m.kernel.lengthscales, "lengthscales"),
                   (m.likelihood.variance, "noise_variance")):
        np.testing.assert_allclose(float(g[p]), ref[key], rtol=1e-3, atol=1e-3 * scale, err_msg=key)
    np.testing.assert_allclose(g[m.inducing_variable.Z], ref["Z"], rtol=1e-3, atol=1e-3 * np.max(np.abs(ref["Z"])))


def test_sgpr_grad_full_c3_fp64_finite_difference_of_device_elbo(cuda_device):
    """Size-independent check at BASELINE configs[2] size (N = 1e5, M = 1024, D = 16, RBF) in float64: the analytic
    device gradient against a central difference of the device elbo() along the lengthscale, the noise, the variance
    and three Z coordinates."""
    d = O.make_data(3, 100000, 16, 1, M=1024)
    s = float(np.sqrt(16.0))
    X, Y = ops.to_device(d["X"]), ops.to_device(d["Y"])

    def elbo(var=1.0, ell=s, s2=0.1, Z=d["Z"]):
        return float(gpf.models.SGPR((X, Y), gpf.kernels.SquaredExponential(variance=var, lengthscales=ell), Z,
                                     noise_variance=s2).elbo())

    m = gpf.models.SGPR((X, Y), gpf.kernels.SquaredExponential(lengthscales=s), d["Z"], noise_variance=0.1)
    e0, g = m.elbo_and_grad()
    e0 = float(e0)
    h = 1e-4
    np.testing.assert_allclose(float(g[m.kernel.lengthscales]), (elbo(ell=s + h) - elbo(ell=s - h)) / (2 * h), rtol=1e-5)
    np.testing.assert_allclose(float(g[m.likelihood.variance]), (elbo(s2=0.1 + h) - elbo(s2=0.1 - h)) / (2 * h),
                               rtol=1e-5)
    np.testing.assert_allclose(float(g[m.kernel.variance]), (elbo(var=1.0 + h) - elbo(var=1.0 - h)) / (2 * h), rtol=1e-5)
    # Z: single coordinates move the ELBO little; the floor is the evaluation noise (~1e-11 relative to the ELBO of a
    # float64 evaluation) over the step
    gz = g[m.inducing_variable.Z]
    atol = 1e-11 * abs(e0) / h
    for (i, j) in ((0, 0), (511, 7), (1023, 15)):
        Zp, Zm = d["Z"].copy(), d["Z"].copy()
        Zp[i, j] += h
        Zm[i, j] -= h
        np.testing.assert_allclose(gz[i, j], (elbo(Z=Zp) - elbo(Z=Zm)) / (2 * h), rtol=1e-5, atol=atol,
                                   err_msg=f"Z[{i},{j}]")


def test_sgpr_elbo_and_grad_value_and_not_pd(cuda_device):
    d = O.make_data(8, 2000, 4, 2, M=150)
    m = gpf.models.SGPR((d["X"], d["Y"]), gpf.kernels.Matern52(lengthscales=1.5), d["Z"], noise_variance=0.1)
    e1 = float(m.elbo_and_grad()[0])
    e0 = float(m.elbo())
    assert abs(e1 - e0) <= 1e-12 * abs(e0)
    # Kuu of 30 inducing points on 3 distinct locations has rank 3; with zero jitter 27 of its pivots are rounding noise
    # around zero, so one of them is non-positive (all positive: probability 2^-27)
    Zd = np.repeat(d["Z"][:3], 10, axis=0)
    with gpf.config.as_context(gpf.config.Config(jitter=0.0)):
        m = gpf.models.SGPR((d["X"], d["Y"]), gpf.kernels.Matern52(lengthscales=1.5), Zd, noise_variance=0.1)
        with pytest.raises(ops.NonPositiveDefiniteError):
            m.elbo_and_grad()


def _oracle_unconstrained(m, X, Y):
    k = m.kernel
    ko = O.SquaredExponential(float(k.variance.numpy()), float(k.lengthscales.numpy()))
    _, g = SG.sgpr_elbo_and_grad(X, Y, ko, m.inducing_variable.Z.numpy(), float(m.likelihood.variance.numpy()))
    return {id(k.variance): g["variance"], id(k.lengthscales): g["lengthscales"],
            id(m.likelihood.variance): g["noise_variance"], id(m.inducing_variable.Z): g["Z"]}


@pytest.mark.parametrize("train_z", [True, False])
def test_scipy_trains_sgpr_on_device_gradients(cuda_device, train_z):
    """gpflow/optimizers/scipy.py:78-228 contract with Z trainable (the GPflow default) and frozen: L-BFGS-B lowers the
    loss, res.fun is the loss at the final iterate, and the gradients there match the oracle chained through the
    bijectors."""
    d = O.make_data(9, 1000, 2, 1, M=30)
    m = gpf.models.SGPR((d["X"], d["Y"]), gpf.kernels.SquaredExponential(lengthscales=3.0), d["Z"], noise_variance=1.0)
    m.inducing_variable.Z.trainable = train_z
    assert (m.inducing_variable.Z in m.trainable_parameters) == train_z
    loss0 = -float(m.elbo())
    res = gpf.optimizers.Scipy().minimize(m.training_loss_closure(), m.trainable_variables, options={"maxiter": 30})
    loss1 = -float(m.elbo())
    assert loss1 < loss0 - 10.0, (loss0, loss1)
    np.testing.assert_allclose(loss1, res.fun, rtol=1e-8)
    loss, grads = m.training_loss_and_gradients()
    assert len(grads) == len(m.trainable_parameters) == (4 if train_z else 3)
    ref = _oracle_unconstrained(m, d["X"], d["Y"])
    for p, gu in zip(m.trainable_parameters, grads):
        want = -p.unconstrained_gradient(ref[id(p)])
        np.testing.assert_allclose(np.asarray(gu), np.asarray(want), rtol=1e-5, atol=1e-5 * max(1.0, np.max(np.abs(want))))


def test_sgpr_grad_unsupported_inputs_raise(cuda_device):
    d = O.make_data(1, 300, 2, 1, M=20)
    kern = gpf.kernels.SquaredExponential() + gpf.kernels.Matern32()
    m = gpf.models.SGPR((d["X"], d["Y"]), kern, d["Z"], noise_variance=0.1)
    with pytest.raises(NotImplementedError):
        m.elbo_and_grad()

    def noise_fn(X):
        return ops.full((X.shape[0], 1), 0.1, like=X)

    m = gpf.models.SGPR((d["X"], d["Y"]), gpf.kernels.SquaredExponential(), d["Z"],
                        likelihood=gpf.likelihoods.Gaussian(variance=noise_fn))
    with pytest.raises(NotImplementedError):
        m.elbo_and_grad()
    m = gpf.models.SGPR((d["X"], d["Y"]), gpf.kernels.SquaredExponential(), d["Z"],
                        mean_function=gpf.mean_functions.Constant([0.1]), noise_variance=0.1)
    with pytest.raises(NotImplementedError):
        m.training_loss_and_gradients()
    with pytest.raises(NotImplementedError):
        gpf.optimizers.Scipy().minimize(m.training_loss_closure(), m.trainable_variables, options={"maxiter": 2})
    f = gpf.models.GPRFITC((d["X"], d["Y"]), gpf.kernels.SquaredExponential(), d["Z"], noise_variance=0.1)
    assert not hasattr(f.training_loss_closure(), "value_and_gradients")
    assert hasattr(gpf.models.SGPR((d["X"], d["Y"]), gpf.kernels.SquaredExponential(), d["Z"],
                                   noise_variance=0.1).training_loss_closure(), "value_and_gradients")
