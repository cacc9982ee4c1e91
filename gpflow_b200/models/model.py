"""Model base classes (mirrors gpflow/models/model.py:29-343, training_mixins.py:43-147, util.py:31-107)."""
from __future__ import annotations

import abc
from typing import Any, Callable, Optional, Tuple

import numpy as np

from .. import ops
from ..base import Module
from ..kernels import Kernel
from ..likelihoods import Likelihood
from ..mean_functions import MeanFunction, Zero


def data_input_to_tensor(data):  # models/util.py:91-107
    return tuple(ops.to_device(d) for d in data)


class BayesianModel(Module, metaclass=abc.ABCMeta):
    def log_prior_density(self) -> float:  # model.py:47-60 (priors are outside the hot path)
        if any(p.prior is not None for p in self.parameters):
            raise NotImplementedError("parameter priors are outside the hot path")
        return 0.0

    def log_posterior_density(self, *args: Any, **kwargs: Any):
        return self.maximum_log_likelihood_objective(*args, **kwargs)

    def _training_loss(self, *args: Any, **kwargs: Any):  # model.py:71-76
        obj = self.maximum_log_likelihood_objective(*args, **kwargs)
        out = ops.copy(obj)
        return ops.axpby(-1.0, obj, 0.0, out)

    @abc.abstractmethod
    def maximum_log_likelihood_objective(self, *args: Any, **kwargs: Any):
        raise NotImplementedError


class GPModel(BayesianModel):
    def __init__(self, kernel: Kernel, likelihood: Likelihood, mean_function: Optional[MeanFunction] = None,
                 num_latent_gps: Optional[int] = None) -> None:
        assert num_latent_gps is not None, "GPModel requires specification of num_latent_gps"
        self.num_latent_gps = num_latent_gps
        self.mean_function = mean_function if mean_function is not None else Zero(output_dim=num_latent_gps)
        self.kernel = kernel
        self.likelihood = likelihood

    @staticmethod
    def calc_num_latent_gps_from_data(data, kernel: Kernel, likelihood: Likelihood) -> int:  # model.py:146-160
        _, Y = data
        return Y.shape[-1]

    @abc.abstractmethod
    def predict_f(self, Xnew, full_cov: bool = False, full_output_cov: bool = False):
        raise NotImplementedError

    def predict_f_samples(self, Xnew, num_samples: Optional[int] = None, full_cov: bool = True,
                          full_output_cov: bool = False, *, eps=None, generator=None):
        """model.py:232-288: samples of the posterior latent function(s) at Xnew, [N, P] or [S, N, P].  `eps` injects the
        standard-normal draws (shapes of conditionals.sample_mvn)."""
        from ..conditionals import sample_mvn

        if full_cov and full_output_cov:
            raise NotImplementedError("The combination of both `full_cov` and `full_output_cov` is not supported.")
        Xnew = ops.to_device(Xnew)
        mean, cov = self.predict_f(Xnew, full_cov=full_cov, full_output_cov=full_output_cov)
        if full_cov:                                                       # model.py:273-279
            samples = sample_mvn(ops.transpose(mean), cov, True, num_samples, eps=eps, generator=generator)  # [(S), P, N]
            if num_samples is None:
                return ops.transpose(samples)
            out = ops.empty((samples.shape[0], samples.shape[2], samples.shape[1]), like=samples)
            for s_ in range(samples.shape[0]):
                ops.transpose(samples[s_], out=out[s_])
            return out
        return sample_mvn(mean, cov, full_output_cov, num_samples, eps=eps, generator=generator)       # model.py:281-284

    def predict_y(self, Xnew, full_cov: bool = False, full_output_cov: bool = False):  # model.py:290-325
        if full_cov or full_output_cov:
            raise NotImplementedError("The predict_y method currently supports only the argument values "
                                      "full_cov=False and full_output_cov=False")
        Xnew = ops.to_device(Xnew)
        f_mean, f_var = self.predict_f(Xnew, full_cov=full_cov, full_output_cov=full_output_cov)
        return self.likelihood.predict_mean_and_var(Xnew, f_mean, f_var)

    def predict_log_density(self, data, full_cov: bool = False, full_output_cov: bool = False):  # :332-343
        if full_cov or full_output_cov:
            raise NotImplementedError("The predict_log_density method currently supports only the argument values "
                                      "full_cov=False and full_output_cov=False")
        X, Y = data
        X = ops.to_device(X)
        f_mean, f_var = self.predict_f(X, full_cov=full_cov, full_output_cov=full_output_cov)
        return self.likelihood.predict_log_density(X, f_mean, f_var, Y)


class LossClosure:
    """What `training_loss_closure()` returns: calling it evaluates the loss (as in the reference); models with a device
    backward pass also give the optimiser `value_and_gradients(variables)` -> (loss, [d loss / d unconstrained variable])
    in the order of `variables` (the pair gpflow/optimizers/scipy.py:300-316 obtains from a GradientTape)."""

    def __init__(self, model, loss_fn: Callable[[], Any]):
        self._model, self._loss_fn = model, loss_fn
        # a subclass that optimises another objective sets the attribute to None (GPRFITC under SGPR)
        if getattr(model, "training_loss_and_gradients", None) is not None:
            self.value_and_gradients = self._value_and_gradients

    def __call__(self):
        return self._loss_fn()

    def _value_and_gradients(self, variables=None):
        loss, grads = self._model.training_loss_and_gradients()
        params = self._model.trainable_parameters
        if variables is None:
            return loss, grads
        by_id = {id(p): g for p, g in zip(params, grads)}
        missing = [v for v in variables if id(v) not in by_id]
        if missing:
            raise ValueError("a variable passed to the optimiser is not a trainable parameter of the model")
        return loss, [by_id[id(v)] for v in variables]


class InternalDataTrainingLossMixin:
    """training_mixins.py:43-78."""

    def training_loss(self):
        return self._training_loss()

    def training_loss_closure(self, *, compile: bool = True) -> Callable[[], Any]:
        return LossClosure(self, self.training_loss)


class ExternalDataTrainingLossMixin:
    """training_mixins.py:81-147."""

    def training_loss(self, data):
        return self._training_loss(data)

    def training_loss_closure(self, data, *, compile: bool = True) -> Callable[[], Any]:
        if hasattr(data, "__next__"):
            it = data

            def closure():
                return self._training_loss(next(it))

            return closure

        def closure():
            return self._training_loss(data)

        return closure
