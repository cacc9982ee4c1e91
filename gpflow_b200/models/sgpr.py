"""Sparse GP regression, Titsias bound (mirrors gpflow/models/sgpr.py:40-289, 346-377, 535-581)."""
from __future__ import annotations

from typing import Any, NamedTuple, Optional, Tuple

import numpy as np

from .. import _lib, config, covariances, ops, posteriors
from ..inducing_variables import InducingPoints, inducingpoint_wrapper
from ..kernels import Kernel, compile_kernel
from ..likelihoods import Gaussian
from ..mean_functions import MeanFunction, Zero
from .model import GPModel, InternalDataTrainingLossMixin, data_input_to_tensor

def _sgpr_fused(X, Y, kernel, inducing_variable, likelihood, mean_function, cache=None, jitter=None, owner=None):
    """One gpk_sgpr_elbo call; returns the device fp64 vector
    [elbo, const, logdet, quad, trace_k, trace_q, half_logdet_b, info]."""
    lib = _lib.load()
    N, D = X.shape
    P = Y.shape[1]
    Z = ops.to_device(inducing_variable.Z)
    M = Z.shape[0]
    dc = ops.dtype_code(X)
    need = lib.gpk_sgpr_elbo_ws(N, M, P, dc)
    # the scratch workspace belongs to the calling model / posterior instance (`owner`): evaluations of different
    # instances on different streams never share it
    ws = getattr(owner, "_sgpr_ws", None) if owner is not None else None
    if ws is None or ws.numel() < need or ws.device != X.device:
        ws = ops.scratch_bytes(need)
        if owner is not None:
            owner._sgpr_ws = ws
    out = ops.torch().empty((8,), dtype=ops.torch().float64, device=X.device)
    if mean_function is None or isinstance(mean_function, Zero):
        Yc = Y
    else:
        Yc = ops.axpby(-1.0, mean_function(X), 1.0, ops.copy(Y))
    nodes, n_nodes, dims, ard = compile_kernel(kernel, D)
    cL, cLB, cc = cache if cache is not None else (None, None, None)
    _lib.check(lib.gpk_sgpr_elbo(nodes, n_nodes, dims, ard, ops._p(X), N, ops._ld(X), D, ops._p(Yc), P, ops._p(Z), M,
                                 ops._ld(Z), likelihood._variance_value(),
                                 config.default_jitter() if jitter is None else jitter, dc, ops._p(out), ops._p(cL),
                                 ops._p(cLB), ops._p(cc), ops._p(ws), ops._stream()), "gpk_sgpr_elbo")
    return out


class SGPR(GPModel, InternalDataTrainingLossMixin):
    class CommonTensors(NamedTuple):
        sigma_sq: Any
        sigma: Any
        A: Any
        B: Any
        LB: Any
        AAT: Any
        L: Any

    def __init__(self, data, kernel: Kernel, inducing_variable, *, mean_function: Optional[MeanFunction] = None,
                 num_latent_gps: Optional[int] = None, noise_variance: Any = None,
                 likelihood: Optional[Gaussian] = None):
        assert (noise_variance is None) or (likelihood is None), "Cannot set both `noise_variance` and `likelihood`."
        if likelihood is None:
            if noise_variance is None:
                noise_variance = 1.0  # sgpr.py:71-74
            likelihood = Gaussian(noise_variance)
        X_data, Y_data = data_input_to_tensor(data)
        num_latent_gps = Y_data.shape[-1] if num_latent_gps is None else num_latent_gps
        super().__init__(kernel, likelihood, mean_function, num_latent_gps=num_latent_gps)
        self.data = X_data, Y_data
        self.num_data = X_data.shape[0]
        self.inducing_variable: InducingPoints = inducingpoint_wrapper(inducing_variable)
        self._last = None

    def maximum_log_likelihood_objective(self):  # sgpr.py:170-171
        return self.elbo()

    def elbo(self):
        """sgpr.py:276-289 in one fused call; device fp64 scalar."""
        X, Y = self.data
        self._last = _sgpr_fused(X, Y, self.kernel, self.inducing_variable, self.likelihood, self.mean_function,
                                 owner=self)
        return ops.objective(self._last, 0, 7)

    def elbo_and_grad(self):
        """Value and gradient in ONE fused call (gpk_sgpr_elbo_grad): the backward pass the reference gets from TensorFlow
        autodiff through sgpr.py:181-289.  Returns (elbo, grads): `elbo` as elbo(); `grads` a dict
        {Parameter: dELBO/d(constrained value)} for the kernel variance, the lengthscale(s), the likelihood variance and
        the inducing points Z ([M, D], zero outside the kernel's active dims), NumPy after one device->host read.
        Covers a single stationary leaf kernel, a constant Gaussian noise variance and InducingPoints, float32 / float64."""
        from ..kernels.stationaries import Stationary

        k = self.kernel
        if not isinstance(k, Stationary) or k._op not in (_lib.K_RBF, _lib.K_MATERN12, _lib.K_MATERN32,
                                                          _lib.K_MATERN52, _lib.K_EXPONENTIAL):
            raise NotImplementedError("the device backward pass covers a single SquaredExponential / Matern12 / "
                                      "Matern32 / Matern52 / Exponential kernel")
        if self.likelihood.heteroskedastic or self.likelihood.variance is None:
            raise NotImplementedError("the device backward pass covers Gaussian(variance=...)")
        iv = self.inducing_variable
        if not isinstance(iv, InducingPoints):
            raise NotImplementedError("the device backward pass covers InducingPoints")
        lib = _lib.load()
        X, Y = self.data
        N, D = X.shape
        P = Y.shape[1]
        Z = ops.to_device(iv.Z)
        M = Z.shape[0]
        dc = ops.dtype_code(X)
        need = lib.gpk_sgpr_elbo_grad_ws(N, M, P, dc)
        if getattr(self, "_sgpr_gws", None) is None or self._sgpr_gws.numel() < need or self._sgpr_gws.device != X.device:
            self._sgpr_gws = ops.scratch_bytes(need)
        nl = int(k.lengthscales.numpy().size) if k.ard else 1
        n_out = 10 + nl
        # one fp64 buffer holds the scalars and dZ [M, D], so the host reads both in one transfer
        buf = ops.torch().empty((n_out + M * D,), dtype=ops.torch().float64, device=X.device)
        out, dZ = buf[:n_out], buf[n_out:]
        if isinstance(self.mean_function, Zero):
            Yc = Y
        else:
            Yc = ops.axpby(-1.0, self.mean_function(X), 1.0, ops.copy(Y))
        nodes, n_nodes, dims, ard = compile_kernel(k, D)
        _lib.check(lib.gpk_sgpr_elbo_grad(nodes, n_nodes, dims, ard, ops._p(X), N, ops._ld(X), D, ops._p(Yc), P,
                                          ops._p(Z), M, ops._ld(Z), self.likelihood._variance_value(),
                                          config.default_jitter(), dc, ops._p(out), n_out, ops._p(dZ), D,
                                          ops._p(self._sgpr_gws), ops._stream()), "gpk_sgpr_elbo_grad")
        self._last = out
        h = buf.cpu().numpy()
        if int(h[7]) != 0:
            raise ops.NonPositiveDefiniteError(f"Cholesky decomposition was not successful (pivot {int(h[7])} <= 0)")
        grads = {k.variance: np.asarray(h[8]), self.likelihood.variance: np.asarray(h[9]),
                 k.lengthscales: (h[10:10 + nl].copy() if k.ard else np.asarray(h[10])),
                 iv.Z: h[n_out:].reshape(M, D).copy()}
        return ops.objective(out, 0, 7), grads

    def training_loss_and_gradients(self):
        """(loss, gradients) for the optimiser contract of gpflow/optimizers/scipy.py:322-331: loss = -ELBO (float) and
        one gradient per TRAINABLE parameter w.r.t. its UNCONSTRAINED variable, in `trainable_parameters` order."""
        elbo, grads = self.elbo_and_grad()
        out = []
        for p in self.trainable_parameters:
            if p not in grads:
                raise NotImplementedError("a trainable parameter has no device gradient (mean-function parameters, "
                                          "priors and data gradients are outside the hot path)")
            out.append(-p.unconstrained_gradient(grads[p]))
        return -float(elbo), out

    def elbo_terms(self):
        """(const, logdet_term, quad_term) of the last evaluation as device scalars (sgpr.py:214-271)."""
        if self._last is None:
            self.elbo()
        return self._last[1], self._last[2], self._last[3]

    def _common_calculation(self) -> "SGPR.CommonTensors":
        """sgpr.py:181-209 built from the individual operators (kept for API parity / testing)."""
        X, _ = self.data
        iv = self.inducing_variable
        s2 = self.likelihood._variance_value()
        sigma_sq = ops.full((X.shape[0],), s2, like=X)
        sigma = ops.full((X.shape[0],), s2 ** 0.5, like=X)
        kuf = covariances.Kuf(iv, self.kernel, X)
        kuu = covariances.Kuu(iv, self.kernel, jitter=config.default_jitter())
        L, dinv = ops.cholesky(kuu)
        A = ops.scale_cols_(kuf, sigma, invert=True)
        ops.trsm(L, A, dinv=dinv)
        AAT = ops.gemm(A, A, transb=True)
        B = ops.add_diag_(ops.copy(AAT), 1.0)
        LB, _ = ops.cholesky(B)
        return self.CommonTensors(sigma_sq, sigma, A, B, LB, AAT, L)

    def upper_bound(self):
        """sgpr.py:87-147: Titsias' (2014) upper bound on the GPR log marginal likelihood, built from the individual
        operators; device fp64 scalar.  (Scalar noise variance: L^-1 (Kuf / s) = (L^-1 Kuf) / s column-wise, so the
        reference's three triangular solves share one.)"""
        X, Y = self.data
        N, P = Y.shape
        s2 = self.likelihood._variance_value()
        iv = self.inducing_variable
        kdiag = self.kernel(X, full_cov=False)
        kuu = covariances.Kuu(iv, self.kernel, jitter=config.default_jitter())
        kuf = covariances.Kuf(iv, self.kernel, X)
        M = kuu.shape[0]
        L, dinv = ops.cholesky(kuu)
        A = ops.trsm(L, kuf, dinv=dinv)                                                   # :118
        # trace bound c = sum Kdiag - sum A^2 (:126): a scalar that enters cn_std = sqrt(s2 + c) below
        c_dev = ops.reduce(ops.SUM, kdiag, N)
        ops.reduce(ops.SUM, ops.colsumsq(A), N, scale=-1.0, out=c_dev, accumulate=True)
        c = float(c_dev.item())
        cn_std = (s2 + c) ** 0.5                                                           # :129-130
        acc = ops.zeros_scalar(1)
        B = ops.gemm(A, A, transb=True, alpha=1.0 / s2)                                   # AAT_sigma (:121)
        ops.add_diag_(B, 1.0)
        LB, _ = ops.cholesky(B)                                                            # :123
        ops.reduce(ops.SUMLOG, LB, M, ops._ld(LB) + 1, scale=-1.0, out=acc, accumulate=True)   # logdet (:133)
        Bc = ops.gemm(A, A, transb=True, alpha=1.0 / (cn_std * cn_std))                    # AAT_cn (:136)
        ops.add_diag_(Bc, 1.0)
        LC, dinvC = ops.cholesky(Bc)                                                       # :139
        err = Y if isinstance(self.mean_function, Zero) else ops.axpby(-1.0, self.mean_function(X), 1.0, ops.copy(Y))
        v = ops.gemm(A, err, alpha=1.0 / (cn_std * cn_std))                                # A_cn (err / cn_std) (:141)
        ops.trsm(LC, v, dinv=dinvC)
        ops.reduce(ops.SUMSQ, err, N * P, 1, scale=-0.5 / (cn_std * cn_std), out=acc, accumulate=True)   # :143
        ops.reduce(ops.SUMSQ, v, M * P, 1, scale=0.5, out=acc, accumulate=True)
        import math
        const = -0.5 * N * math.log(2.0 * math.pi * s2)                                    # :132
        ops.axpby(1.0, ops.full((1,), const, dtype="float64"), 1.0, acc)
        return acc[0]

    def compute_qu(self) -> Tuple[Any, Any]:
        """sgpr.py:346-377: mean [M, P] and covariance [M, M] of q(u)."""
        X, Y = self.data
        s2 = self.likelihood._variance_value()
        kuf = covariances.Kuf(self.inducing_variable, self.kernel, X)
        kuu = covariances.Kuu(self.inducing_variable, self.kernel, jitter=config.default_jitter())
        sig = ops.copy(kuu)
        ops.gemm(kuf, kuf, transb=True, alpha=1.0 / s2, beta=1.0, out=sig)      # kuu + kuf kuf^T / s2
        sig_sqrt, dinv = ops.cholesky(sig)
        sig_sqrt_kuu = ops.trsm(sig_sqrt, ops.copy(kuu), dinv=dinv)
        cov = ops.gemm(sig_sqrt_kuu, sig_sqrt_kuu, transa=True)
        err = Y if isinstance(self.mean_function, Zero) else ops.axpby(-1.0, self.mean_function(X), 1.0, ops.copy(Y))
        rhs = ops.gemm(kuf, err, alpha=1.0 / s2)                                # scaled_kuf @ scaled_err
        ops.trsm(sig_sqrt, rhs, dinv=dinv)
        mu = ops.gemm(sig_sqrt_kuu, rhs, transa=True)
        return mu, cov

    def posterior(self, precompute_cache=posteriors.PrecomputeCacheType.TENSOR) -> posteriors.SGPRPosterior:
        """sgpr.py:535-566."""
        return posteriors.SGPRPosterior(kernel=self.kernel, data=self.data, inducing_variable=self.inducing_variable,
                                        likelihood=self.likelihood, num_latent_gps=self.num_latent_gps,
                                        mean_function=self.mean_function,
                                        precompute_cache=posteriors._validate_precompute_cache_type(precompute_cache))

    def predict_f(self, Xnew, full_cov: bool = False, full_output_cov: bool = False):  # sgpr.py:568-581
        return self.posterior(posteriors.PrecomputeCacheType.NOCACHE).fused_predict_f(
            Xnew, full_cov=full_cov, full_output_cov=full_output_cov)


class GPRFITC(SGPR):
    """GP regression with the FITC approximation (mirrors gpflow/models/sgpr.py:380-523; Snelson & Ghahramani 2006), a
    re-composition of the same device operators: K-build (Kdiag, Kuf, Kuu), two Cholesky factorisations, triangular
    solves, and fp64 reductions.  Same constructor as SGPR."""

    def common_terms(self):
        """sgpr.py:399-432 -> (err [N, R], nu [N], Luu [M, M], L [M, M], alpha [M, R], beta [N, R], gamma [M, R]) plus the
        block inverses of the two factors (for the solves of predict_f)."""
        X, Y = self.data
        iv = self.inducing_variable
        M = iv.num_inducing
        err = Y if isinstance(self.mean_function, Zero) else ops.axpby(-1.0, self.mean_function(X), 1.0, ops.copy(Y))
        Kdiag = self.kernel(X, full_cov=False)
        kuf = covariances.Kuf(iv, self.kernel, X)
        kuu = covariances.Kuu(iv, self.kernel, jitter=config.default_jitter())
        sigma_sq = self.likelihood.variance_at(X).reshape(-1)
        Luu, dinv_uu = ops.potrf(kuu)
        ops.tril_(Luu)
        V = ops.trsm(Luu, kuf, dinv=dinv_uu)                                  # V^T V = Qff
        nu = ops.copy(Kdiag)                                                    # nu = Kdiag - diagQff + sigma_sq
        ops.colsumsq(V, scale=-1.0, out=nu, accumulate=True)
        ops.axpby(1.0, sigma_sq, 1.0, nu)
        Vn = ops.scale_cols_(ops.copy(V), nu, invert=True)                      # V / nu
        B = ops.gemm(Vn, V, transb=True)
        ops.add_diag_(B, 1.0)
        L, dinv_b = ops.potrf(B)
        ops.tril_(L)
        beta = ops.scale_rows_(ops.copy(err), nu, invert=True)                  # err / nu[:, None]
        alpha = ops.gemm(V, beta)
        gamma = ops.trsm(L, ops.copy(alpha), dinv=dinv_b)
        self._dinvs = (dinv_uu, dinv_b)
        return err, nu, Luu, L, alpha, beta, gamma

    def maximum_log_likelihood_objective(self):  # sgpr.py:434-435
        return self.fitc_log_marginal_likelihood()

    # GPRFITC optimises fitc_log_marginal_likelihood(), which has no device backward pass: its training closure offers
    # no value_and_gradients
    training_loss_and_gradients = None

    def elbo(self):
        raise NotImplementedError("GPRFITC optimises fitc_log_marginal_likelihood(), not an ELBO")

    def elbo_and_grad(self):
        raise NotImplementedError("GPRFITC optimises fitc_log_marginal_likelihood(), not an ELBO")

    def fitc_log_marginal_likelihood(self):
        """sgpr.py:440-480; device fp64 scalar."""
        import math

        err, nu, _Luu, L, _alpha, beta, gamma = self.common_terms()
        N, R = err.shape
        M = L.shape[0]
        acc = ops.zeros_scalar(1)
        # mahalanobis: -1/2 sum err^2 / nu + 1/2 sum gamma^2   (err^2 / nu = err * beta)
        prod = ops.hadamard_(ops.copy(err), beta)
        ops.reduce(ops.SUM, prod, N * R, 1, scale=-0.5, out=acc, accumulate=True)
        ops.reduce(ops.SUMSQ, gamma, M * R, 1, scale=0.5, out=acc, accumulate=True)
        # (constant + log-determinant) * num_latent_gps
        P = float(self.num_latent_gps)
        ops.reduce(ops.SUMLOG, nu, N, 1, scale=-0.5 * P, out=acc, accumulate=True)
        ops.reduce(ops.SUMLOG, L, M, ops._ld(L) + 1, scale=-P, out=acc, accumulate=True)
        ops.axpby(1.0, ops.full((1,), -0.5 * self.num_data * math.log(2.0 * math.pi) * P, dtype="float64"), 1.0, acc)
        return acc[0]

    def predict_f(self, Xnew, full_cov: bool = False, full_output_cov: bool = False):  # sgpr.py:482-523
        if full_output_cov:
            raise NotImplementedError("GPRFITC.predict_f does not support full_output_cov=True")
        _, _, Luu, L, _, _, gamma = self.common_terms()
        dinv_uu, dinv_b = self._dinvs
        Xnew = ops.to_device(Xnew)
        Kus = covariances.Kuf(self.inducing_variable, self.kernel, Xnew)       # [M, N]
        w = ops.trsm(Luu, Kus, dinv=dinv_uu)
        tmp = ops.trsm(L, ops.copy(gamma), trans=True, dinv=dinv_b)             # L^-T gamma
        mean = ops.gemm(w, tmp, transa=True)
        if not isinstance(self.mean_function, Zero):
            ops.axpby(1.0, self.mean_function(Xnew), 1.0, mean)
        iA = ops.trsm(L, ops.copy(w), dinv=dinv_b)
        P = self.num_latent_gps
        if full_cov:
            v = ops.copy(self.kernel(Xnew))
            ops.gemm(w, w, transa=True, alpha=-1.0, beta=1.0, out=v)
            ops.gemm(iA, iA, transa=True, alpha=1.0, beta=1.0, out=v)
            var = ops.empty((P,) + tuple(v.shape), like=v)
            for p in range(P):
                ops.axpby(1.0, v, 0.0, var[p])
            return mean, var
        v = ops.copy(self.kernel(Xnew, full_cov=False))
        ops.colsumsq(w, scale=-1.0, out=v, accumulate=True)
        ops.colsumsq(iA, scale=1.0, out=v, accumulate=True)
        var_t = ops.empty((P, v.shape[0]), like=v)
        for p in range(P):
            ops.axpby(1.0, v, 0.0, var_t[p])
        return mean, ops.transpose(var_t)
