# The interface pieces of this module that a drop-in must keep word for word -- the ValueError messages of
# `validate_meta_data`, the prior-name -> parameter-name rule of `sample_all_priors` -- are derived from
# scamlgp/utils.py of boschresearch/Scalable-Meta-Learning-with-Gaussian-Processes,
# Copyright (c) 2024 Robert Bosch GmbH, AGPL-3.0.
"""Mirror of the reference's scamlgp/utils.py: restart driver, prior sampling, meta-data
conversion/validation and the UCB acquisition, on the B200 engine.

  sample_all_priors              scamlgp/utils.py:31-69
  metadata_to_numerical          scamlgp/utils.py:72-109
  validate_meta_data             scamlgp/utils.py:112-136
  optimize_marginal_likelihood   scamlgp/utils.py:139-212
  UpperConfidenceBound           scamlgp/utils.py:215-224
plus the batch (q > 1) acquisitions qUpperConfidenceBound / qExpectedImprovement (botorch's MC semantics).
"""
from __future__ import annotations

import logging
import math
import warnings
from typing import Dict, Hashable, Iterable, Optional, Union

import torch

from .modules import DT, ModelFittingError, SupervisedDataset

logger = logging.getLogger("scamlgp_b200")


def sample_all_priors(model, num_retries: int = 5, generator: Optional[torch.Generator] = None) -> None:
    r"""Sample every registered prior in place (reference utils.py:31-69): a draw is rejected when the
    constraint's inverse transform is not finite; more than `num_retries` rejections raise RuntimeError."""
    for prior_name, module, prior, closure, setting_closure in model.named_priors():
        if prior is None:
            continue
        if setting_closure is None:
            raise RuntimeError("Must provide inverse transform to be able to sample from prior.")
        parameter_name = "_".join(prior_name.split(".")[-1].split("_")[:-1])
        constraint = getattr(module, "raw_" + parameter_name + "_constraint")
        for i in range(num_retries + 1):
            sample = prior.sample(closure(module).shape, generator=generator)
            if bool(constraint.inverse_transform(sample).isfinite().all()):
                setting_closure(module, sample)
                break
        else:
            raise RuntimeError(f"Sampling of {prior_name} failed {num_retries} times. Please check the compatibility "
                               "between prior support and the constraint.")
        if i > 0:
            logger.warning(f"Sampling from {prior_name} failed {i} times in a row.")


def metadata_to_numerical(meta_data: Dict[Hashable, Iterable], search_space, objective,
                          batch_shape: torch.Size = torch.Size(), torch_dtype: torch.dtype = torch.float32
                          ) -> Dict[Hashable, SupervisedDataset]:
    """Meta evaluations -> tensors; evaluations are sorted first so runs do not depend on their order, NaNs of
    inactive (conditional) parameters are imputed (reference utils.py:72-109)."""
    from .space import impute_nans_with_constant, sort_numerical, to_numerical

    out = {}
    for task_id, task_data in meta_data.items():
        # the reference sorts the evaluations first (utils.py:99) so that runs do not depend on their order; the
        # same order independence is obtained by sorting the numerical rows (see space.sort_numerical)
        X_raw, Y = to_numerical(task_data, search_space, [objective], batch_shape=batch_shape, torch_dtype=torch_dtype)
        X_raw, Y = sort_numerical(X_raw, Y)
        out[task_id] = SupervisedDataset(impute_nans_with_constant(X_raw), Y)
    return out


def validate_meta_data(meta_data: Dict[Hashable, SupervisedDataset]):
    """Shape checks of the meta-data (reference utils.py:112-136; same messages)."""
    if len(meta_data) == 0:
        raise ValueError("Empty meta data. Needs at least one source task.")
    task_id_source_0, data_source_0 = list(meta_data.items())[0]
    X_shape = data_source_0.X.shape
    Y_shape = data_source_0.Y.shape
    if X_shape[:-2] != Y_shape[:-2]:
        raise ValueError(f"The X and Y batch sizes of task {task_id_source_0} are not equal.")
    for task_id, task_data in meta_data.items():
        if (task_data.X.shape[:-2] != X_shape[:-2] or task_data.Y.shape[:-2] != Y_shape[:-2]
                or task_data.X.shape[-1] != X_shape[-1]):
            raise ValueError(f"Dimensions of tasks {task_id_source_0} and {task_id} do not match.")
        if task_data.Y.shape[-1] != 1:
            raise ValueError(f"The output dimension of task {task_id} is {task_data.Y.shape[-1]} but must be one")


def optimize_marginal_likelihood(model, num_restarts: int = 0, generator: Optional[torch.Generator] = None,
                                 **fit_options):
    """Refit the ScaML-GP target model by maximising (LML + log priors)/n_t (reference utils.py:139-212).

    1 warm start from the current parameters + `num_restarts` prior-sampled starts, all optimised together
    (one batched objective launch per L-BFGS round); the best final value wins, failed rows are skipped
    with a warning, all failed -> ModelFittingError."""
    from .fit import fit_target
    from .model import ScaMLGP, SourceGP
    from .modules import set_theta_raw

    if isinstance(model, SourceGP):
        # the reference calls this on every source GP (model.py:187); here meta_fit_scamlgp batches those fits, and
        # this is the single-model form of the same driver (refit of one task, e.g. after its data changed)
        return _optimize_source_gp(model, num_restarts, generator, **fit_options)
    if not isinstance(model, ScaMLGP):
        raise TypeError("optimize_marginal_likelihood expects a ScaMLGP or a SourceGP of meta_fit_scamlgp, got "
                        f"{type(model).__name__}")
    if model.num_train == 0:
        raise ValueError("cannot optimise the marginal likelihood of a model without training data")
    fit_options.pop("max_attempts", None)
    fit_options.pop("caught_exception_types", None)
    state0 = model.state_dict()
    rows_w, rows_t = [model.weights.clone()], [model.theta_raw()]
    for _ in range(num_restarts):
        sample_all_priors(model, generator=generator)
        rows_w.append(model.weights.clone())
        rows_t.append(model.theta_raw())
    model.load_state_dict(state0)
    eng, dev = model.engine, model.engine.device
    ot = model.outcome_transform
    fit = fit_target(eng, model.source_means, model.source_covs, model._Xt,
                     model.train_targets.to(dev, DT).contiguous(), float(ot.means), float(ot.stdvs), model.hyper_spec(),
                     torch.stack(rows_w), torch.stack(rows_t), w_prior=model.weights_prior.spec(),
                     w_lower=model.raw_weights_constraint.lower_bound, fit_options=fit_options or None)
    nfail = int(torch.isinf(fit.all_lml).sum())
    if nfail:
        logger.warning(f"Error occurred while optimizing the model hyperparameters: {nfail} restart(s) skipped.")
    model.raw_weights = fit.weights.detach().cpu().clone()
    set_theta_raw(model.likelihood, model.covar_module, fit.theta_raw)
    model._tstate = None
    model.last_fit = fit
    return fit


def _optimize_source_gp(gp, num_restarts: int, generator: Optional[torch.Generator], **fit_options):
    """(LML + log priors)/n of ONE source GP maximised from its current parameters + `num_restarts` prior draws
    (reference utils.py:139-212 on a SingleTaskGP, as called at model.py:187); the winner is written back to the
    GP's modules and to its slice of the owner's packed device state (factor, alpha, parameters)."""
    from .engine import SourceBatch
    from .fit import fit_sources, sample_theta_raw
    from .modules import hyper_spec_of, set_theta_raw, theta_raw_of

    fit_options.pop("max_attempts", None)
    fit_options.pop("caught_exception_types", None)
    owner = gp._owner
    eng = owner.engine
    X, Y = gp.train_inputs[0], gp._raw_Y
    d = X.shape[-1]
    spec = hyper_spec_of(gp.likelihood, gp.covar_module)
    theta0 = theta_raw_of(gp.likelihood, gp.covar_module, d)
    rows = [theta0.reshape(1, 1, -1)]
    if num_restarts > 0:
        rows.append(sample_theta_raw(spec, theta0, 1, int(num_restarts), generator))
    sh = getattr(owner, "sharded", None)
    fitted = getattr(owner, "fitted", None)
    local = fitted is not None and (sh is None or sh.lo <= gp._index < sh.hi)
    n_max = fitted.batch.n_max if local else None
    batch = SourceBatch.from_ragged([(X, Y)], eng.device, n_max=n_max)
    fit = fit_sources(eng, batch, spec, torch.cat(rows, dim=1), fit_options or None)
    nfail = int(torch.isinf(fit.all_lml).sum())
    if nfail:
        logger.warning(f"Error occurred while optimizing the model hyperparameters: {nfail} restart(s) skipped.")
    set_theta_raw(gp.likelihood, gp.covar_module, fit.theta_raw[0].cpu())
    if local:
        i = gp._index - (sh.lo if sh is not None else 0)
        one = eng.factorize(batch, fit.theta_raw, spec)
        fitted.theta_raw[i], fitted.theta[i] = one.theta_raw[0], one.theta[0]
        fitted.linv[i], fitted.alpha[i], fitted.info[i] = one.linv[0], one.alpha[0], one.info[0]
        if sh is not None:
            sh._invalidate()
    return fit


class UpperConfidenceBound:
    """UCB with default beta = 9.0, always minimising (reference utils.py:215-224): botorch's UCB with
    maximize=False returns -mu + sqrt(beta * sigma^2), to be maximised."""

    def __init__(self, model, beta: Union[float, torch.Tensor] = 9.0, posterior_transform=None, **kwargs):
        if kwargs.get("maximize", False):
            raise ValueError("Only acquisition functions to be minimized are supported")
        self.model = model
        self.beta = float(beta)
        self.maximize = False

    def __call__(self, X: torch.Tensor) -> torch.Tensor:
        return self.forward(X)

    def forward(self, X: torch.Tensor) -> torch.Tensor:
        post = self.model.posterior(X)
        mean = post.mean.reshape(-1)
        var = post.variance.reshape(-1).clamp_min(1e-9)  # botorch: sigma = variance.clamp_min(1e-9).sqrt()
        return -mean + torch.sqrt(self.beta * var)

    def value_and_grad(self, X: torch.Tensor):
        """Acquisition value [B] and its gradient wrt the candidates [B, d] from the analytic posterior gradients
        (the reference differentiates the same expression by autograd inside botorch's optimize_acqf)."""
        mean, var, dmean, dvar = self.model.posterior_with_grad(X)
        live = var > 1e-9  # clamp_min(1e-9): zero variance gradient below the clamp
        sig = torch.sqrt(self.beta * var.clamp_min(1e-9))
        grad = -dmean + (0.5 * self.beta / sig * live.to(sig.dtype)).unsqueeze(-1) * dvar
        return -mean + sig, grad


def psd_safe_cholesky(A: torch.Tensor) -> torch.Tensor:
    """Cholesky factor of a batch of matrices [..., q, q] with linear_operator's psd_safe_cholesky jitter ladder: a
    matrix whose factorisation fails is retried with 1e-8, 1e-7, 1e-6 added to its diagonal (differentiable)."""
    from ._capi import NotPSDError
    from .engine import JITTER_LADDER

    L, info = torch.linalg.cholesky_ex(A)
    if not bool((info > 0).any()):
        return L
    eye = torch.eye(A.shape[-1], dtype=A.dtype, device=A.device)
    for jit in JITTER_LADDER:
        bad = (info > 0).to(A.dtype)[..., None, None]
        L, info = torch.linalg.cholesky_ex(A + bad * jit * eye)
        if not bool((info > 0).any()):
            return L
    raise NotPSDError(f"Matrix not positive definite after repeatedly adding jitter up to {JITTER_LADDER[-1]:.1e}")


def sobol_normal_samples(num_samples: int, q: int, seed: int) -> torch.Tensor:
    """[num_samples, q] scrambled-Sobol standard normal draws (botorch's draw_sobol_normal_samples: inverse CDF of
    the Sobol points pulled in by one ulp so that no draw is infinite)."""
    u = torch.quasirandom.SobolEngine(dimension=q, scramble=True, seed=seed).draw(num_samples, dtype=DT)
    u = 0.5 + (1.0 - torch.finfo(DT).eps) * (u - 0.5)
    return torch.erfinv(2.0 * u - 1.0) * math.sqrt(2.0)


class _MCBatchAcquisition:
    """Monte-Carlo acquisition over blocks of q points X [b, q, d] (botorch's MCAcquisitionFunction with a
    SobolQMCNormalSampler): samples xi = mu + L z of the joint posterior of every block, L its Cholesky factor, z a
    fixed scrambled-Sobol draw taken once per object (and q) so that an optimiser sees a deterministic function.
    Values and gradients come from `ScaMLGP.posterior_blocks`; the gradient is autograd on the small (mu, Sigma)
    leaves followed by the model's vector-Jacobian product (csrc/scaml_qblock.cuh)."""

    maximize = False

    def __init__(self, model, num_samples: int = 128, seed: int = 0):
        self.model = model
        self.num_samples = int(num_samples)
        self.seed = int(seed)
        self._z: Dict[int, torch.Tensor] = {}

    def base_samples(self, q: int) -> torch.Tensor:
        if q not in self._z:
            self._z[q] = sobol_normal_samples(self.num_samples, q, self.seed)
        return self._z[q]

    def from_moments(self, mean: torch.Tensor, cov: torch.Tensor) -> torch.Tensor:
        """Acquisition value [b] of blocks with posterior mean [b, q] and covariance [b, q, q] (differentiable)."""
        z = self.base_samples(mean.shape[-1]).to(mean.device)
        L = psd_safe_cholesky(cov)
        samples = mean.unsqueeze(-2) + torch.einsum("bik,sk->bsi", L, z)  # [b, num_samples, q]
        return self._reduce(mean, samples)

    def _reduce(self, mean: torch.Tensor, samples: torch.Tensor) -> torch.Tensor:
        raise NotImplementedError

    def __call__(self, X: torch.Tensor) -> torch.Tensor:
        return self.forward(X)

    def forward(self, X: torch.Tensor) -> torch.Tensor:
        """Values [b] of the blocks X [b, q, d]; evaluated 128 points at a time (each launch's U is freed before the
        next one is built)."""
        step = max(1, 128 // X.shape[-2])
        vals = []
        for lo in range(0, X.shape[0], step):
            mean, cov, _ = self.model.posterior_blocks(X[lo:lo + step])
            vals.append(self.from_moments(mean, cov))
        return torch.cat(vals)

    def value_and_grad(self, X: torch.Tensor):
        """Values [b] and their gradients wrt the blocks [b, q, d]."""
        mean, cov, vjp = self.model.posterior_blocks(X)
        m, c = mean.detach().requires_grad_(True), cov.detach().requires_grad_(True)
        with torch.enable_grad():
            val = self.from_moments(m, c)
            g_mean, g_cov = torch.autograd.grad(val.sum(), (m, c))
        return val.detach(), vjp(g_mean, g_cov)


class qUpperConfidenceBound(_MCBatchAcquisition):
    """botorch's qUpperConfidenceBound turned into minimisation like `UpperConfidenceBound`:
    mean over the samples of max_i ( -mu_i + sqrt(beta pi / 2) |xi_i - mu_i| ).  At q = 1 its expectation is the
    analytic -mu + sqrt(beta sigma^2)."""

    def __init__(self, model, beta: Union[float, torch.Tensor] = 9.0, num_samples: int = 128, seed: int = 0):
        super().__init__(model, num_samples, seed)
        self.beta = float(beta)

    def _reduce(self, mean, samples):
        scale = math.sqrt(self.beta * math.pi / 2.0)
        return (-mean.unsqueeze(-2) + scale * (samples - mean.unsqueeze(-2)).abs()).max(dim=-1).values.mean(dim=-1)


class qExpectedImprovement(_MCBatchAcquisition):
    """botorch's qExpectedImprovement for a loss to be minimised: mean over the samples of max_i max(best_f - xi_i, 0).
    best_f defaults to the smallest observed loss of the model's training data."""

    def __init__(self, model, best_f: Optional[Union[float, torch.Tensor]] = None, num_samples: int = 128,
                 seed: int = 0):
        super().__init__(model, num_samples, seed)
        if best_f is None:
            Y = model._train_Y.reshape(-1)
            Y = Y[~torch.isnan(Y)]
            if Y.numel() == 0:
                raise ValueError("qExpectedImprovement needs best_f when the model has no observations")
            best_f = Y.min()
        self.best_f = float(best_f)

    def _reduce(self, mean, samples):
        return (self.best_f - samples).clamp_min(0.0).max(dim=-1).values.mean(dim=-1)
