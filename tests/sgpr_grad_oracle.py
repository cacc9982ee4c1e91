"""Gradient oracle of the SGPR ELBO (test infrastructure, NumPy; not imported by the product).

The reference obtains dELBO/d(theta) from TensorFlow autodiff through gpflow/models/sgpr.py:181-289.  The closed form
restated here is what the device backward pass (csrc/grad.cu, DESIGN.md section 4.9) computes.  With E = Y - m(X),
Kuu = K(Z, Z) + jitter I = L L^T, A' = L^-1 Kuf, B = A'A'^T / s2 + I = LB LB^T, c = LB^-1 A'E / s2, w~ = LB^-T c and
v = L^-T w~:

    dELBO/dKuf   = (L^-T C A' + v E^T) / s2,             C = P (I - B^-1) - w~ w~^T
    dELBO/dKuu   = L^-T (P I - P/2 (B + B^-1) - 1/2 w~ w~^T) L^-1
    dELBO/dKdiag = -P / (2 s2)
    dELBO/ds2    = (1/s2) [-NP/2 + sum E^2 / (2 s2) + P/2 (trace_k - trace_q) + P/2 (M - tr B^-1) - |c|^2/2 - |w~|^2/2]

chained into the kernel variance, the lengthscale(s) and Z through k(s), s = sum_d ((a_d - b_d) / l_d)^2.
tests/test_oracle_sgpr_grad.py pins it by central finite differences of gp_oracle.sgpr_elbo.
"""
from __future__ import annotations

from typing import Dict, Tuple

import numpy as np

from oracle import gp_oracle as O


def _k_and_dkds(kernel: O.Stationary, s: np.ndarray) -> Tuple[np.ndarray, np.ndarray]:
    """k(s) and dk/ds of a stationary kernel at scaled squared distances s (stationaries.py:209-210, 250-251, 270-271,
    290-292, 311-313).  The 1e-36 clip before the square root passes no gradient, as tf.maximum does."""
    var = float(np.asarray(kernel.variance))
    clipped = ~(s > 1e-36)
    r = np.sqrt(np.where(clipped, 1e-36, s))
    if isinstance(kernel, O.SquaredExponential):
        k = var * np.exp(-0.5 * s)
        return k, -0.5 * k
    if isinstance(kernel, O.Matern12):
        k = var * np.exp(-r)
        return k, np.where(clipped, 0.0, -k / (2.0 * r))
    if isinstance(kernel, O.Exponential):
        k = var * np.exp(-0.5 * r)
        return k, np.where(clipped, 0.0, -k / (4.0 * r))
    if isinstance(kernel, O.Matern32):
        s3 = np.sqrt(3.0)
        e = np.exp(-s3 * r)
        return var * (1.0 + s3 * r) * e, np.where(clipped, 0.0, -1.5 * var * e)
    if isinstance(kernel, O.Matern52):
        s5 = np.sqrt(5.0)
        e = np.exp(-s5 * r)
        return var * (1.0 + s5 * r + (5.0 / 3.0) * r * r) * e, np.where(clipped, 0.0, -(5.0 / 6.0) * var * (1.0 + s5 * r) * e)
    raise NotImplementedError(type(kernel).__name__)


def _active(kernel: O.Stationary, D: int) -> np.ndarray:
    return np.arange(D)[kernel.active_dims]


def _chain(kernel: O.Stationary, A: np.ndarray, B: np.ndarray, G: np.ndarray, dims: np.ndarray):
    """sum_ij G_ij dk(a_i, b_j)/d(variance, lengthscales) and sum_j G_ij dk(a_i, b_j)/da_i (active columns)."""
    ell = np.asarray(kernel.lengthscales, dtype=np.float64)
    ell_d = np.broadcast_to(ell, (dims.size,)) if ell.ndim else np.full(dims.size, float(ell))
    diff = (A[:, None, dims] - B[None, :, dims]) / ell_d                    # scaled differences [I, J, Da]
    s = np.sum(diff * diff, axis=-1)
    k, dkds = _k_and_dkds(kernel, s)
    W = G * dkds
    g_var = float(np.sum(G * k)) / float(np.asarray(kernel.variance))
    if ell.ndim:
        g_ell = np.einsum("ij,ijd->d", W, -2.0 * diff * diff) / ell_d
    else:
        g_ell = float(np.sum(W * -2.0 * s)) / float(ell)
    g_a = np.einsum("ij,ijd->id", W, 2.0 * diff) / ell_d                   # ds/da_d = 2 (a_d - b_d) / l_d^2
    return g_var, g_ell, g_a


def sgpr_elbo_and_grad(X: np.ndarray, Y: np.ndarray, kernel: O.Stationary, Z: np.ndarray, noise_variance: float,
                       mean_function=None, jitter: float = O.DEFAULT_JITTER) -> Tuple[float, Dict[str, np.ndarray]]:
    """ELBO (sgpr.py:214-289) and its gradient w.r.t. the kernel variance, the lengthscales (scalar or ARD vector), the
    likelihood variance and Z ([M, D], zero in the columns outside the kernel's active_dims)."""
    X, Y, Z = (np.asarray(a, dtype=np.float64) for a in (X, Y, Z))
    N, P = Y.shape
    M, D = Z.shape
    s2 = float(noise_variance)
    E = Y - O._mean(mean_function, X, P)
    Kuu = kernel(Z) + jitter * np.eye(M)
    Kuf = kernel(Z, X)
    L = O.cholesky(Kuu)
    Li = O.tri_solve(L, np.eye(M))
    Ap = Li @ Kuf
    B = Ap @ Ap.T / s2 + np.eye(M)
    LB = O.cholesky(B)
    LBi = O.tri_solve(LB, np.eye(M))
    Bi = LBi.T @ LBi
    c = LBi @ (Ap @ E) / s2
    wt = LBi.T @ c
    v = Li.T @ wt
    C = P * (np.eye(M) - Bi) - wt @ wt.T
    dKuf = (Li.T @ C @ Ap + v @ E.T) / s2
    dKuu = Li.T @ (P * np.eye(M) - 0.5 * P * (B + Bi) - 0.5 * wt @ wt.T) @ Li
    trace_k = float(np.sum(kernel(X, full_cov=False))) / s2
    trace_q = float(np.trace(Ap @ Ap.T)) / s2
    elbo = float(-0.5 * N * P * O.LOG2PI - P * (np.sum(np.log(np.diag(LB))) + 0.5 * N * np.log(s2)
                                                + 0.5 * (trace_k - trace_q))
                 - 0.5 * (np.sum(E * E) / s2 - np.sum(c * c)))
    dims = _active(kernel, D)
    gv_f, gl_f, gz_f = _chain(kernel, Z, X, dKuf, dims)
    gv_u, gl_u, gz_u = _chain(kernel, Z, Z, dKuu, dims)
    dZ = np.zeros((M, D))
    dZ[:, dims] = gz_f + 2.0 * gz_u       # k(z_i, z_j) depends on z_m through i = m and j = m alike
    grad = {
        "variance": gv_f + gv_u - P * N / (2.0 * s2),    # Kdiag = variance at every point
        "lengthscales": gl_f + gl_u,
        "noise_variance": (-0.5 * N * P + 0.5 * np.sum(E * E) / s2 + 0.5 * P * (trace_k - trace_q)
                           + 0.5 * P * (M - np.trace(Bi)) - 0.5 * np.sum(c * c) - 0.5 * np.sum(wt * wt)) / s2,
        "Z": dZ,
    }
    return elbo, grad
