"""Pins the SGPR ELBO gradient oracle (tests/sgpr_grad_oracle.py) by central finite differences of the ELBO oracle, and
the host-side contract of the SGPR backward pass (workspace query, which closures offer value_and_gradients)."""
import numpy as np
import pytest

from oracle import gp_oracle as O
from tests import sgpr_grad_oracle as SG

KERNELS = [O.SquaredExponential, O.Matern12, O.Matern32, O.Matern52, O.Exponential]


def _setup(seed, N, M, D, P):
    rng = np.random.default_rng(seed)
    X = rng.standard_normal((N, D))
    Y = np.sin(X[:, :1]) + 0.1 * rng.standard_normal((N, P))
    Z = rng.standard_normal((M, D))        # not a subset of X: no zero distances for the sqrt-type kernels
    return X, Y, Z


def _exact(cls):
    """The oracle kernel with its scaled squared distance taken by direct differences.  The reference's norm expansion
    (utilities/ops.py:109-111) leaves rounding noise of ~1e-16 in r^2 on the diagonal of K(Z, Z), which moves with the
    lengthscale; for the sqrt-type kernels (Matern12, Exponential) a finite difference of the ELBO sees it at the 1e-4
    level.  With direct differences the diagonal distance is exactly 0, where the closed form has it."""

    class Exact(cls):
        def scaled_squared_euclid_dist(self, X, X2=None):
            A = self.scale(X)
            B = A if X2 is None else self.scale(X2)
            d = A[:, None, :] - B[None, :, :]
            return np.sum(d * d, axis=-1)

    return Exact


def _fd_check(X, Y, Z, make, var, ell, s2, mean=None, tol=2e-6):
    """Every gradient entry of the oracle against a central difference of gp_oracle.sgpr_elbo."""
    elbo, g = SG.sgpr_elbo_and_grad(X, Y, make(var, ell), Z, s2, mean_function=mean)
    assert abs(elbo - O.sgpr_elbo(X, Y, make(var, ell), Z, s2, mean_function=mean)) <= 1e-10 * abs(elbo)

    def f(v=var, l=ell, s=s2, z=Z):
        return O.sgpr_elbo(X, Y, make(v, l), z, s, mean_function=mean)

    h = 1e-6

    def close(got, fd, what):
        assert abs(got - fd) <= tol * max(1.0, abs(fd)), (what, got, fd)

    close(g["variance"], (f(v=var + h) - f(v=var - h)) / (2 * h), "variance")
    close(g["noise_variance"], (f(s=s2 + h) - f(s=s2 - h)) / (2 * h), "noise_variance")
    ell = np.asarray(ell, dtype=np.float64)
    if ell.ndim == 0:
        close(g["lengthscales"], (f(l=float(ell) + h) - f(l=float(ell) - h)) / (2 * h), "lengthscale")
    else:
        assert np.shape(g["lengthscales"]) == ell.shape
        for d in range(ell.size):
            e = np.zeros(ell.size)
            e[d] = h
            close(g["lengthscales"][d], (f(l=ell + e) - f(l=ell - e)) / (2 * h), ("lengthscale", d))
    assert g["Z"].shape == Z.shape
    for m in range(Z.shape[0]):
        for d in range(Z.shape[1]):
            e = np.zeros_like(Z)
            e[m, d] = h
            close(g["Z"][m, d], (f(z=Z + e) - f(z=Z - e)) / (2 * h), ("Z", m, d))
    return g


@pytest.mark.parametrize("cls", KERNELS)
@pytest.mark.parametrize("P", [1, 2])
@pytest.mark.parametrize("ard", [False, True])
def test_sgpr_elbo_gradient_matches_finite_differences(cls, P, ard):
    X, Y, Z = _setup(11 + P, 80, 9, 3, P)
    ell = np.array([0.9, 1.4, 2.0]) if ard else 1.3
    _fd_check(X, Y, Z, lambda v, l: _exact(cls)(variance=v, lengthscales=l), 1.3, ell, 0.3)


@pytest.mark.parametrize("cls", KERNELS)
def test_sgpr_elbo_gradient_constant_mean_and_active_dims(cls):
    """A Constant mean function, and a kernel on two of four input columns: the inactive Z columns get exactly 0."""
    X, Y, Z = _setup(5, 70, 8, 4, 2)
    mean = O.ConstantMean(np.array([0.3, -0.2]))
    for ell in (1.1, np.array([0.8, 1.6])):
        g = _fd_check(X, Y, Z, lambda v, l: _exact(cls)(variance=v, lengthscales=l, active_dims=[0, 2]), 0.9, ell, 0.25,
                      mean=mean)
        assert np.all(g["Z"][:, [1, 3]] == 0.0)
        assert np.any(g["Z"][:, [0, 2]] != 0.0)


def test_sgpr_noise_gradient_sign_at_extremes():
    """Sanity of the noise gradient away from the finite-difference check: shrinking a very large noise raises the
    ELBO (negative gradient), as does growing a very small one on noisy data (positive gradient)."""
    X, Y, Z = _setup(3, 120, 10, 2, 1)
    k = O.SquaredExponential(variance=1.0, lengthscales=1.0)
    assert SG.sgpr_elbo_and_grad(X, Y, k, Z, 50.0)[1]["noise_variance"] < 0.0
    assert SG.sgpr_elbo_and_grad(X, Y, k, Z, 1e-4)[1]["noise_variance"] > 0.0


def test_sgpr_elbo_grad_workspace_query():
    """The value + gradient workspace holds the forward's and grows with N and M."""
    from gpflow_b200 import _lib

    try:
        lib = _lib.load()
    except Exception as e:  # noqa: BLE001
        pytest.skip(f"libgpk.so not loadable here: {e}")
    for dc in (_lib.GPK_F32, _lib.GPK_F64):
        for N, M, P in [(100, 10, 1), (1000, 130, 2), (100000, 1024, 1)]:
            assert lib.gpk_sgpr_elbo_grad_ws(N, M, P, dc) >= lib.gpk_sgpr_elbo_ws(N, M, P, dc)
        assert lib.gpk_sgpr_elbo_grad_ws(2000, 100, 1, dc) > lib.gpk_sgpr_elbo_grad_ws(1000, 100, 1, dc)
        assert lib.gpk_sgpr_elbo_grad_ws(1000, 200, 1, dc) > lib.gpk_sgpr_elbo_grad_ws(1000, 100, 1, dc)


def test_closures_offer_value_and_gradients_for_sgpr_not_gprfitc():
    """SGPR's training closure carries value_and_gradients (the device backward pass); GPRFITC, which subclasses SGPR
    but optimises the FITC marginal likelihood, does not.  Checked on the classes: no device is touched."""
    from gpflow_b200.models import GPRFITC, SGPR
    from gpflow_b200.models.model import LossClosure

    class _Fake:
        pass

    sg = _Fake()
    sg.training_loss_and_gradients = SGPR.training_loss_and_gradients.__get__(sg)
    assert hasattr(LossClosure(sg, lambda: 0.0), "value_and_gradients")
    assert GPRFITC.training_loss_and_gradients is None
    fitc = _Fake()
    fitc.training_loss_and_gradients = GPRFITC.training_loss_and_gradients
    assert not hasattr(LossClosure(fitc, lambda: 0.0), "value_and_gradients")
    assert callable(SGPR.training_loss_and_gradients)
