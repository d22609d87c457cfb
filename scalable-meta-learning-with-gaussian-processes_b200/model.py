# The interface pieces a drop-in must keep -- `significant_weights_mask` (a four-line formula), the default
# constraints / priors of the `_get_default_*` helpers and the argument lists -- are derived from scamlgp/model.py of
# boschresearch/Scalable-Meta-Learning-with-Gaussian-Processes, Copyright (c) 2024 Robert Bosch GmbH, AGPL-3.0.
"""ScaML-GP model API -- mirror of the reference's scamlgp/model.py on the B200 engine.

Same names, arguments and error behaviour as the reference:
  meta_fit_scamlgp            scamlgp/model.py:138-189
  ScaMLGP                     scamlgp/model.py:218-384
  significant_weights_mask    scamlgp/model.py:192-215
  _compute_target_prior       scamlgp/model.py:108-135
  _get_default_likelihood / _get_kernel_source_gp / _get_default_kernel   model.py:25-105
What changes is where the arithmetic runs: the per-task Python loops (model.py:128,176,281) become
single batched kernel launches through `engine.Engine` (C ABI: include/scaml_b200.h).
"""
from __future__ import annotations

import copy
from typing import Dict, Hashable, List, Optional, Tuple

import torch

from ._capi import PRIOR_GAMMA, HyperSpec
from .engine import Engine, FittedSources, SourceBatch, TargetState, default_engine
from .fit import fit_sources, sample_theta_raw
from .modules import (DT, GammaPrior, GaussianLikelihood, GreaterThan, Interval, LogNormalPrior, MaternKernel,
                      MultivariateNormal, Posterior, RBFKernel, ScaleKernel, Standardize, SupervisedDataset,
                      hyper_spec_of, set_theta_raw, theta_raw_of)
from .utils import validate_meta_data


# gpytorch is exact (Cholesky) up to max_cholesky_size = 800 training points and switches to CG / Lanczos
# approximations beyond (SURVEY A.5): parity is defined up to 800, and so is this implementation
MAX_TARGET_POINTS = 800


def max_target_points(engine: Engine, d: int) -> int:
    """Largest n_t whose target-GP kernels keep the n_t x n_t system in 227 KB of shared memory at input dimension d
    (the footprint grows with d * n_t: 117 at d = 2, 113 at d = 16; `scaml_target_max_points`).  Larger n_t (up to
    MAX_TARGET_POINTS) run on the global-memory variants of the same kernels: slower per evaluation, same results."""
    return int(engine.lib.target_max_points(int(d)))


# ---- defaults (reference model.py:25-105) ---------------------------------------------------- #
def _get_default_likelihood(batch_shape: torch.Size = torch.Size()) -> GaussianLikelihood:
    return GaussianLikelihood(noise_prior=LogNormalPrior(-8.0, 2.0), noise_constraint=Interval(1e-8, 1e-2, 1e-3),
                              batch_shape=batch_shape)


def _get_kernel_source_gp(base_kernel=RBFKernel, ard_num_dims: Optional[int] = None,
                          batch_shape: torch.Size = torch.Size()) -> ScaleKernel:
    return ScaleKernel(
        base_kernel=base_kernel(ard_num_dims=ard_num_dims, batch_shape=batch_shape,
                                lengthscale_prior=GammaPrior(3.0, 6.0),
                                lengthscale_constraint=Interval(1e-4, 1e2, 0.5)),
        batch_shape=batch_shape, outputscale_prior=GammaPrior(2.0, 0.15),
        outputscale_constraint=Interval(1e-4, 1e2, 1.0))


def _get_default_kernel(base_kernel=RBFKernel, ard_num_dims: Optional[int] = None,
                        batch_shape: torch.Size = torch.Size()) -> ScaleKernel:
    return ScaleKernel(
        base_kernel=base_kernel(ard_num_dims=ard_num_dims, batch_shape=batch_shape,
                                lengthscale_prior=LogNormalPrior(0.5, 1.5),
                                lengthscale_constraint=Interval(1e-4, 1e2, 1.0)),
        batch_shape=batch_shape, outputscale_prior=LogNormalPrior(-2.0, 3.0),
        outputscale_constraint=Interval(1e-4, 1e2, 0.1))


# ---- fitted source GP (stand-in for the botorch SingleTaskGP the reference returns) ---------- #
class SourceGP:
    """One fitted source task.  Holds its data, fitted modules and Standardize state; predictions go
    through the shared device batch (`owner.fitted`, index `index`).

    The per-task module objects (`likelihood`, `covar_module`, `outcome_transform`) and `train_targets` are
    materialised on first access from the fitted parameter row: deep-copying the kernel / likelihood templates for
    every one of 4096 tasks was 0.56 s of a 1.7 s meta-fit, and the BO loop itself never looks at them."""

    def __init__(self, train_X, train_Y, likelihood, covar_module, outcome_transform, owner: "SourceGPDict",
                 index: int, theta_raw: Optional[torch.Tensor] = None, ybar=None, ystd=None):
        """Either fully materialised modules (theta_raw None), or templates + (theta_raw, ybar, ystd) to build from."""
        self.train_inputs = (train_X,)
        self._raw_Y = train_Y
        self._owner = owner
        self._index = index
        self._lazy = None
        self._train_targets = None
        if theta_raw is None:
            self._likelihood, self._covar_module, self._outcome_transform = likelihood, covar_module, outcome_transform
        else:
            self._likelihood = self._covar_module = self._outcome_transform = None
            self._lazy = (likelihood, covar_module, theta_raw, ybar, ystd)

    def _materialise(self) -> None:
        if self._lazy is None:
            return
        lk_t, cm_t, theta_raw, ybar, ystd = self._lazy
        self._lazy = None
        lk, cm = copy.deepcopy(lk_t), copy.deepcopy(cm_t)
        set_theta_raw(lk, cm, theta_raw)
        tf = Standardize(1)
        tf.means, tf.stdvs, tf._is_trained = ybar.reshape(1, 1), ystd.reshape(1, 1), True
        tf.eval()
        self._likelihood, self._covar_module, self._outcome_transform = lk, cm, tf

    @property
    def likelihood(self):
        self._materialise()
        return self._likelihood

    @likelihood.setter
    def likelihood(self, value):
        self._materialise()
        self._likelihood = value

    @property
    def covar_module(self):
        self._materialise()
        return self._covar_module

    @covar_module.setter
    def covar_module(self, value):
        self._materialise()
        self._covar_module = value

    @property
    def outcome_transform(self):
        self._materialise()
        return self._outcome_transform

    @property
    def train_targets(self):
        if self._train_targets is None:
            ot = self.outcome_transform
            self._train_targets = (self._raw_Y.reshape(-1) - ot.means.reshape(())) / ot.stdvs.reshape(())
        return self._train_targets

    def posterior(self, X: torch.Tensor) -> Posterior:
        """Posterior of this source GP at X [n, d] (un-standardised, noise-free), full covariance."""
        sh = getattr(self._owner, "sharded", None)
        if sh is not None and not (sh.lo <= self._index < sh.hi):
            raise NotImplementedError(f"source task {self._index} lives on another rank (this rank owns tasks "
                                      f"[{sh.lo}, {sh.hi})); query it there or use the weighted ScaMLGP posterior")
        fs = self._owner.fitted.task_slice(self._index - (sh.lo if sh is not None else 0))
        eng = self._owner.engine
        Xd = X.reshape(-1, X.shape[-1]).to(eng.device, DT).contiguous()
        mean, cov = eng.predict_cross(fs, Xd)
        mean, cov = mean[:, 0].to(X.device), cov[:, :, 0].to(X.device)
        return Posterior(mean, cov.diagonal(), cov)


class SourceGPDict(dict):
    """Dict[task_id, SourceGP] that also carries the device-resident batch of all fitted tasks -- or, after a
    task-sharded meta-fit (`meta_fit_scamlgp(..., group=...)`), this rank's block of them plus the collectives
    (`sharded`: scamlgp_b200.sharded.ShardedSources)."""

    engine: Engine
    fitted: FittedSources
    sharded = None


def _batch_from_sources(source_gps: Dict[Hashable, SourceGP], engine: Engine) -> FittedSources:
    """Re-assemble (and re-factorise) a device batch from individual SourceGP objects, in dict order."""
    gps = list(source_gps.values())
    d = gps[0].train_inputs[0].shape[-1]
    batch = SourceBatch.from_ragged([(g.train_inputs[0], g._raw_Y) for g in gps], engine.device)
    spec = hyper_spec_of(gps[0].likelihood, gps[0].covar_module)
    theta = torch.stack([theta_raw_of(g.likelihood, g.covar_module, d) for g in gps]).to(engine.device).contiguous()
    return engine.factorize(batch, theta, spec)


def fitted_sources_of(source_gps: Dict[Hashable, SourceGP], engine: Optional[Engine] = None) -> FittedSources:
    """The device batch behind a dict of source GPs, in the dict's iteration order."""
    if getattr(source_gps, "sharded", None) is not None:
        raise NotImplementedError("task-sharded source GPs are queried through their ShardedSources "
                                  "(ScaMLGP does this); there is no single device batch of all tasks")
    if (isinstance(source_gps, SourceGPDict) and len(source_gps) == source_gps.fitted.batch.M
            and [g._index for g in source_gps.values()] == list(range(len(source_gps)))):
        return source_gps.fitted  # untouched dict: the device batch as fitted (a dict with tasks deleted re-selects)
    eng = engine or (source_gps.engine if isinstance(source_gps, SourceGPDict) else default_engine())
    owner = next(iter(source_gps.values()))._owner
    idx = [g._index for g in source_gps.values()]
    if all(g._owner is owner for g in source_gps.values()):
        return owner.fitted.select(torch.tensor(idx, device=owner.fitted.theta.device))
    return _batch_from_sources(source_gps, eng)


def meta_fit_scamlgp(meta_data: Dict[Hashable, SupervisedDataset], likelihood: Optional[GaussianLikelihood] = None,
                     covar_module: Optional[ScaleKernel] = None, num_restarts_log_likelihood: int = 5,
                     seed: Optional[int] = None, *, engine: Optional[Engine] = None,
                     fit_options: Optional[dict] = None, group=None) -> Dict[Hashable, SourceGP]:
    """Train the source GPs on the given meta-data (reference scamlgp/model.py:138-189).

    All tasks and all restarts are optimised together on the GPU; returns {task_id: SourceGP} in the
    order of `meta_data` (a SourceGPDict, which also owns the packed device state used for prediction).

    group: a torch.distributed process group (or True for the default group) -> the tasks are block-partitioned
    over its ranks (one process per GPU; the reference's loop over independent tasks, model.py:176-188, fans out):
    every rank fits and factorises only its block, one all_gather shares the fitted rows, and the returned dict
    carries `sharded` (ShardedSources) through which `ScaMLGP` / `ScaMLGPBO` predict with one all_reduce per call.
    Every rank must pass the same meta-data and seed and gets the same dict back."""
    generator = None
    if seed is not None:
        torch.manual_seed(seed)
        generator = torch.Generator().manual_seed(seed)
    validate_meta_data(meta_data)
    first = list(meta_data.values())[0]
    d = first.X.shape[-1]
    batch_shape = first.X.shape[:-2]
    if len(batch_shape) != 0:
        raise NotImplementedError("batched meta-data (batch_shape != ()) is not supported; the reference optimizer "
                                  "always uses torch.Size() (scamlgp/optimizer.py:121)")
    if likelihood is None:
        likelihood = _get_default_likelihood(batch_shape=batch_shape)
    if covar_module is None:
        covar_module = _get_kernel_source_gp(base_kernel=RBFKernel, ard_num_dims=d, batch_shape=batch_shape)
    eng = engine or default_engine()
    spec = hyper_spec_of(likelihood, covar_module)
    theta0 = theta_raw_of(likelihood, covar_module, d)
    tasks = [(ds.X(), ds.Y()) for ds in meta_data.values()]
    M, R = len(tasks), 1 + int(num_restarts_log_likelihood)
    rows = [theta0.reshape(1, 1, -1).expand(M, 1, -1)]
    if R > 1:
        rows.append(sample_theta_raw(spec, theta0, M, R - 1, generator))  # positional: identical on every rank
    out = SourceGPDict()
    if group is not None:
        from .sharded import ShardedSources

        src = ShardedSources(eng, tasks, group=None if group is True else group)
        sfit = src.fit(spec, torch.cat(rows, dim=1), fit_options)
        out.engine, out.fitted, out.fit, out.sharded = eng, src.fitted, sfit, src
        theta_host, ybar, ystd = sfit.theta_raw.cpu(), src.ybar_all.cpu(), src.ystd_all.cpu()
    else:
        batch = SourceBatch.from_ragged(tasks, eng.device)
        fit = fit_sources(eng, batch, spec, torch.cat(rows, dim=1), fit_options)
        fitted = eng.factorize(batch, fit.theta_raw, spec)
        out.engine, out.fitted, out.fit = eng, fitted, fit
        theta_host = fit.theta_raw.cpu()
        ybar, ystd = batch.ybar.cpu(), batch.ystd.cpu()
    for i, (task_id, (X, Y)) in enumerate(zip(meta_data.keys(), tasks)):
        # modules are built from (templates, fitted row) on first access: see SourceGP
        out[task_id] = SourceGP(X, Y, likelihood, covar_module, None, out, i, theta_raw=theta_host[i], ybar=ybar[i],
                                ystd=ystd[i])
    return out


def significant_weights_mask(weights: torch.Tensor, std_Y_vals: torch.Tensor, threshold: float) -> torch.Tensor:
    r"""Mask of weights with w_i sigma_i n_w / sum_j w_j sigma_j >= threshold (reference model.py:192-215)."""
    num_weights = len(weights)
    w_times_sigma = weights * std_Y_vals
    norm_weights = w_times_sigma * num_weights / w_times_sigma.sum()
    return norm_weights >= threshold


def _compute_target_prior(x: torch.Tensor, source_gps: List[SourceGP], weights: torch.Tensor,
                          engine: Optional[Engine] = None) -> Tuple[torch.Tensor, torch.Tensor]:
    """Prior of the target GP at x [n, d]: mean [n, 1] = sum_i w_i mu_i(x), cov [n, n] = sum_i w_i^2 Sigma_i(x, x)
    (reference model.py:108-135) -- one launch reduced over the tasks instead of a Python loop."""
    if len(source_gps) != len(weights):
        raise ValueError(f"The number of source GPs, {len(source_gps)}, does not equal the number of weights, "
                         f"{len(weights)}")
    fs = fitted_sources_of(dict(enumerate(source_gps)), engine)
    eng = engine or source_gps[0]._owner.engine
    mean, cov = eng.predict_cross(fs, x.to(eng.device, DT).contiguous(), None, w=weights.to(eng.device, DT))
    return mean.unsqueeze(-1), cov


class ScaMLGP:
    """Scalable and Modular Kernel for Transfer Learning with Gaussian Processes (reference model.py:218-384)."""

    def __init__(self, train_X: torch.Tensor, train_Y: torch.Tensor, source_gps: Dict[Hashable, SourceGP],
                 likelihood: Optional[GaussianLikelihood] = None, covar_module: Optional[ScaleKernel] = None,
                 weight_pruning_threshold: float = 1e-3, *, engine: Optional[Engine] = None) -> None:
        self._weight_pruning_threshold = weight_pruning_threshold
        if len(train_Y.shape[:-2]) != 0:
            raise NotImplementedError("batch_shape must be ()")
        n_source_tasks = len(source_gps)
        gps = list(source_gps.values())
        self.engine = engine or (source_gps.engine if isinstance(source_gps, SourceGPDict) else gps[0]._owner.engine)
        dev = self.engine.device
        # task-sharded source GPs (meta_fit_scamlgp(..., group=)): this rank holds a block of the tasks; caches are
        # all_gathered, predictions all_reduced (sharded.py).  Every rank builds the same model object.
        self._sharded = getattr(source_gps, "sharded", None)
        if self._sharded is not None and len(source_gps) != self._sharded.M:
            raise NotImplementedError("a task-sharded SourceGPDict must be used whole (all tasks, original order)")
        self._fitted = self._sharded.fitted if self._sharded is not None else fitted_sources_of(source_gps, self.engine)
        d = train_X.shape[-1]
        # all-data normaliser (model.py:264-276): every source task's raw Y + the target Y, frozen
        if self._sharded is not None:
            Y_all = torch.cat([self._sharded.all_Y.to(dev, DT), train_Y.reshape(-1).to(dev, DT)])
        else:
            b = self._fitted.batch
            mask = torch.arange(b.n_max, device=dev).unsqueeze(0) < b.n_valid.unsqueeze(1)
            Y_all = torch.cat([b.Y_raw[mask], train_Y.reshape(-1).to(dev, DT)])
        outcome_transform = Standardize(1)
        outcome_transform(Y_all.cpu())
        outcome_transform.eval()
        self.train_inputs = (train_X,)
        self._train_Y = train_Y
        n_t = train_Y.shape[-2]
        if n_t > MAX_TARGET_POINTS:
            raise NotImplementedError(
                f"{n_t} target observations: exact inference is defined for n_t <= {MAX_TARGET_POINTS} (beyond that the "
                "reference's gpytorch stack switches to CG / Lanczos approximations, SURVEY A.5)")
        if n_t > 128 and self._fitted.batch.n_max > 256:
            raise NotImplementedError(
                f"{n_t} target observations with {self._fitted.batch.n_max} points per source task: the fused "
                "conditioning kernels cover n_t <= 128 and the stand-alone cross-covariance kernel n <= 256")
        if n_t > 0 and not (self.engine.cond_supported(self._fitted, n_t) or self.engine.cross_supported(self._fitted)):
            raise NotImplementedError(f"{n_t} target observations with {self._limits_text()}: the source caches at "
                                      "the target inputs need the fused conditioning kernels (n_t <= 128, d <= 16 and "
                                      "the prediction kernel's n) or the cross-covariance kernel")
        self._Xt = train_X.reshape(n_t, d).to(dev, DT).contiguous()
        # cache the source posteriors at the target inputs (model.py:278-289): one launch for all tasks
        self._condA: Optional[torch.Tensor] = None  # K_m^-1 K_m(X_m, X_t) of every source task
        if n_t > 0:
            if self._sharded is not None:
                self.source_means, self.source_covs = self._sharded.target_caches(self._Xt)
            elif self.engine.cond_supported(self._fitted, n_t):
                # A_m once per model; the caches and every later posterior call are contractions with it
                self._condA = self.engine.cond_prepare(self._fitted, self._Xt)
                self.source_means, self.source_covs = self.engine.cond_caches(self._fitted, self._Xt, self._condA)
            else:
                self.source_means, self.source_covs = self.engine.predict_cross(self._fitted, self._Xt)
        if covar_module is None:
            covar_module = _get_default_kernel(base_kernel=RBFKernel, ard_num_dims=d)
        self.source_gps = source_gps
        if likelihood is None:
            likelihood = _get_default_likelihood()
        self.likelihood, self.covar_module = likelihood, covar_module
        if train_Y.nelement() == 0:  # empty input: do not standardise (model.py:307-308)
            self.outcome_transform = None
            self.train_targets = train_Y.reshape(-1).to(DT)
        else:
            self.outcome_transform = outcome_transform
            self.train_targets = outcome_transform(train_Y.to(DT))[0].reshape(-1)
        self.raw_weights = torch.full((n_source_tasks,), 1.0 / n_source_tasks, dtype=DT)
        self.weights_prior = GammaPrior(1.0, 1.0)
        self.raw_weights_constraint = GreaterThan(1e-10, transform=None)
        self.training = True
        self._tstate: Optional[TargetState] = None

    # ---- parameters ------------------------------------------------------------------------- #
    @property
    def weights(self) -> torch.Tensor:
        return self.raw_weights_constraint.transform(self.raw_weights)

    @weights.setter
    def weights(self, value):
        self._set_weights(value)

    def _set_weights(self, value):
        if not torch.is_tensor(value):
            value = torch.as_tensor(value)
        self.raw_weights = self.raw_weights_constraint.inverse_transform(value.detach().to("cpu", DT)).clone()
        self._tstate = None

    def train(self, mode: bool = True):
        self.training = mode
        return self

    def eval(self):
        return self.train(False)

    def state_dict(self) -> Dict[str, torch.Tensor]:
        sd = {"raw_weights": self.raw_weights.clone()}
        sd.update(self.likelihood.state_dict("likelihood.noise_covar."))
        sd.update(self.covar_module.state_dict("covar_module."))
        return sd

    def load_state_dict(self, sd: Dict[str, torch.Tensor]) -> None:
        self.raw_weights = sd["raw_weights"].clone()
        self.likelihood.load_state_dict(sd, "likelihood.noise_covar.")
        self.covar_module.load_state_dict(sd, "covar_module.")
        self._tstate = None

    def named_priors(self):
        """(name, module, prior, closure, setting_closure) like gpytorch's Module.named_priors."""
        bk = self.covar_module.base_kernel
        yield ("covar_module.base_kernel.lengthscale_prior", bk, bk.lengthscale_prior, lambda m: m.lengthscale,
               lambda m, v: setattr(m, "lengthscale", v))
        yield ("covar_module.outputscale_prior", self.covar_module, self.covar_module.outputscale_prior,
               lambda m: m.outputscale, lambda m, v: setattr(m, "outputscale", v))
        yield ("likelihood.noise_covar.noise_prior", self.likelihood, self.likelihood.noise_prior,
               lambda m: m.noise, lambda m, v: setattr(m, "noise", v))
        yield ("weights_prior", self, self.weights_prior, lambda m: m.weights, lambda m, v: m._set_weights(v))

    # ---- internals ---------------------------------------------------------------------------- #
    def _limits_text(self) -> str:
        b, lib = self._fitted.batch, self.engine.lib
        return (f"{b.n_max} points per source task at d = {b.d} (the prediction kernel covers n <= "
                f"{lib.predict_max_points(b.d)}, the cross-covariance kernel n <= {lib.predict_cross_max_points(b.d)})")

    def _require_predict(self) -> None:
        if not self.engine.predict_supported(self._fitted):
            raise NotImplementedError(f"posterior with {self._limits_text()}: outside the prediction kernel")

    def _require_cross(self, what: str) -> None:
        if not self.engine.cross_supported(self._fitted):
            raise NotImplementedError(f"{what} with {self._limits_text()}: outside the cross-covariance kernel")

    @property
    def num_train(self) -> int:
        return self._Xt.shape[0]

    def hyper_spec(self) -> HyperSpec:
        return hyper_spec_of(self.likelihood, self.covar_module)

    def theta_raw(self) -> torch.Tensor:
        return theta_raw_of(self.likelihood, self.covar_module, self._Xt.shape[1])

    def _std_Y_vals(self) -> torch.Tensor:
        if self._sharded is not None:
            return self._sharded.ystd_all.to(self.engine.device, DT)
        return self._fitted.batch.ystd

    def pruned_weights(self) -> torch.Tensor:
        """Device weights with the insignificant ones zeroed (the kernels skip w == 0), model.py:365-372."""
        w = self.weights.to(self.engine.device, DT)
        mask = significant_weights_mask(w, self._std_Y_vals(), self._weight_pruning_threshold)
        return torch.where(mask, w, torch.zeros_like(w)).contiguous()

    def _target_state(self) -> TargetState:
        if self._tstate is None:
            dev = self.engine.device
            ot = self.outcome_transform
            # conditioning uses the CACHED train-branch prior (all weights), exactly as gpytorch's prediction
            # strategy is built from forward(train_X) in ... eval mode -> pruned weights (model.py:364-375)
            w = self.pruned_weights()
            self._tstate = self.engine.target_factorize(
                self.source_means, self.source_covs, self._Xt, self.train_targets.to(dev, DT).contiguous(), w,
                self.theta_raw().to(dev).contiguous(), float(ot.means), float(ot.stdvs), self.hyper_spec())
        return self._tstate

    # ---- forward / posterior ------------------------------------------------------------------ #
    def forward(self, x: torch.Tensor) -> MultivariateNormal:
        """Prior of the target process at x [n, d] (or batch_shape x n x d: one joint prior per batch element) in the
        (all-data) standardised space (model.py:359-384)."""
        if x.dim() > 2:
            lead = x.shape[:-2]
            parts = [self.forward(xi) for xi in x.reshape(-1, x.shape[-2], x.shape[-1])]
            return MultivariateNormal(torch.stack([p.mean for p in parts]).reshape(*lead, -1),
                                      torch.stack([p.covariance_matrix for p in parts]).reshape(
                                          *lead, x.shape[-2], x.shape[-2]))
        eng, dev = self.engine, self.engine.device
        xd = x.reshape(-1, x.shape[-1]).to(dev, DT).contiguous()
        if self.training:
            w = self.weights.to(dev, DT)
            mean = self.source_means @ w
            cov = self.source_covs @ w ** 2
        elif self._sharded is not None:
            self._require_cross("joint prior (eval mode)")
            mean, cov = self._sharded.predict_cross(self.pruned_weights(), xd)
        elif eng.cross_supported(self._fitted):
            mean, cov = eng.predict_cross(self._fitted, xd, None, w=self.pruned_weights())
        elif eng.cond_supported(self._fitted, xd.shape[0]):  # the points as their own "target inputs"
            w = self.pruned_weights()
            U = eng.cond_prepare(self._fitted, xd, w)
            mean, _, cov = eng.predict_conditioned(self._fitted, w, xd, xd, U)
            cov = 0.5 * (cov + cov.t())
        else:
            self._require_cross("joint prior (eval mode)")
        if self.outcome_transform is not None:
            mu, sd = float(self.outcome_transform.means), float(self.outcome_transform.stdvs)
            mean = (mean - mu) / sd
            cov = cov / sd ** 2
        spec = self.hyper_spec()
        kt = eng.kernel_matrix(xd.unsqueeze(0), self._target_kernel_theta(xd.shape[1]), spec.kernel)[0]
        return MultivariateNormal(mean, cov + kt)

    def posterior(self, X: torch.Tensor, observation_noise: bool = False) -> Posterior:
        """Posterior at X, un-standardised (botorch `Model.posterior` shapes, reference model.py:359-384).

        X [B, d] or [B, 1, d]: B independent candidates (q = 1, the acquisition path) -> mean / variance [B, 1].
        X [b..., q, d] with q > 1: joint posterior over the q points of every batch element -> mean / variance
        [b..., q, 1] and `.mvn.covariance_matrix` [b..., q, q]."""
        if observation_noise:
            raise NotImplementedError("observation_noise=True is not used on the reference path")
        eng, dev = self.engine, self.engine.device
        if X.dim() >= 3 and X.shape[-2] != 1:
            return self._posterior_joint(X)
        if X.dim() >= 3:
            lead = X.shape[:-2]
            X = X.reshape(-1, X.shape[-1])
        else:
            lead = None
        self._require_predict()
        Xc = X.to(dev, DT).contiguous()
        w = self.pruned_weights()
        if self._sharded is not None:
            ts = self._target_state() if self.num_train > 0 else None
            mean, var = self._sharded.posterior(w, Xc, ts, float(self.covar_module.outputscale))
        elif self.num_train > 0 and eng.cond_supported(self._fitted, self.num_train):
            mean, var = self._posterior_fused(Xc, w)
        else:
            pm, pv = eng.predict_weighted(self._fitted, w, Xc)
            if self.num_train == 0:
                # prior-only model (optimizer.py:135-141): no outcome transform, var + s_t
                mean, var = pm, pv + float(self.covar_module.outputscale)
            else:
                _, cross = eng.predict_cross(self._fitted, Xc, self._Xt, w=w)
                mean, var = eng.target_posterior(self._target_state(), pm, pv, cross, Xc)
        mean, var = mean.to(X.device), var.to(X.device)
        if lead is not None and len(lead) > 1:
            return Posterior(mean.reshape(*lead, 1), var.reshape(*lead, 1))
        return Posterior(mean, var)

    def _target_kernel_theta(self, d: int) -> torch.Tensor:
        dev = self.engine.device
        ls = self.covar_module.base_kernel.lengthscale.reshape(-1).to(dev)
        if ls.numel() == 1:
            ls = ls.expand(d)
        return torch.cat([ls, self.covar_module.outputscale.reshape(1).to(dev),
                          torch.zeros(1, dtype=DT, device=dev)]).reshape(1, -1).contiguous()

    def _posterior_joint(self, X: torch.Tensor) -> Posterior:
        """q > 1: the joint blocks of the eval branch (model.py:364-375 evaluates every source posterior at
        [X_t; X*] jointly).  The weighted source blocks Sigma(X*, X*) and Sigma(X*, X_t) come from the fused
        prediction kernel -- the candidates of a chunk of batch elements play the role of the "target inputs" of
        `cond_prepare` / `predict_conditioned`, so one launch gives all their pair covariances, n <= 512 -- and the
        n_t-dimensional conditioning (q x n_t blocks against the cached L_t^-1, alpha_t) is torch on the device."""
        eng, dev = self.engine, self.engine.device
        lead, q, d = X.shape[:-2], X.shape[-2], X.shape[-1]
        if q > 128:
            raise NotImplementedError("joint posteriors are supported for q <= 128 points per batch element")
        Xall = X.reshape(-1, q, d).to(dev, DT)
        nb_all, n_t = Xall.shape[0], self.num_train
        w = self.pruned_weights()
        ts = self._target_state() if n_t > 0 else None
        spec = self.hyper_spec()
        theta_t = self._target_kernel_theta(d)
        means, covs = [], []
        step = max(1, 128 // q)
        for lo in range(0, nb_all, step):
            Xf = Xall[lo:lo + step].reshape(-1, d).contiguous()  # [nb * q, d]
            nb = Xf.shape[0] // q
            pm, cqq, cqt = self._weighted_blocks(Xf, w)
            Z = torch.cat([self._Xt, Xf]) if n_t > 0 else Xf
            kt = eng.kernel_matrix(Z.unsqueeze(0).contiguous(), theta_t, spec.kernel)[0]
            kqq = kt[n_t:, n_t:]
            idx = torch.arange(nb * q, device=dev).reshape(nb, q)
            blk = lambda A: A[idx.unsqueeze(2), idx.unsqueeze(1)]  # noqa: E731  [nb, q, q] diagonal blocks
            if n_t == 0:  # prior-only model (optimizer.py:135-141): no outcome transform
                mean, cov = pm.reshape(nb, q), blk(cqq) + blk(kqq)
            else:
                mu, sd = ts.mu_all, ts.s_all
                cst = cqt / sd ** 2 + kt[n_t:, :n_t]  # [nb q, n_t] standardised cross-covariance with X_t
                V = ts.linv @ cst.t()  # [n_t, nb q]
                mean_s = (pm - mu) / sd + cst @ ts.alpha
                cov_s = blk(cqq) / sd ** 2 + blk(kqq) - blk(V.t() @ V)
                mean, cov = (mu + sd * mean_s).reshape(nb, q), sd ** 2 * cov_s
            means.append(mean)
            covs.append(cov)
        mean = torch.cat(means).reshape(*lead, q).to(X.device)
        cov = torch.cat(covs).reshape(*lead, q, q).to(X.device)
        return Posterior(mean, cov.diagonal(dim1=-2, dim2=-1), cov)

    def _weighted_blocks(self, Xf: torch.Tensor, w: torch.Tensor):
        """Weighted source prior at the points Xf [B, d] (raw-Y units): mean [B], Sigma(Xf, Xf) [B, B] and
        Sigma(Xf, X_t) [B, n_t] (None without target data), summed over ALL tasks."""
        eng, n_t = self.engine, self.num_train
        if self._sharded is not None:
            self._require_cross("joint posterior")
            mean, cqq = self._sharded.predict_cross(w, Xf)
            cqt = self._sharded.predict_cross(w, Xf, self._Xt)[1] if n_t > 0 else None
            return mean, cqq, cqt
        fs = self._fitted
        if eng.cond_supported(fs, Xf.shape[0]):
            U = eng.cond_prepare(fs, Xf, w)  # K_m^-1 K_m(X_m, Xf): the points are their own "target inputs"
            mean, _, cqq = eng.predict_conditioned(fs, w, Xf, Xf, U)
            cqq = 0.5 * (cqq + cqq.t())
            cqt = None
            if n_t > 0 and eng.cond_supported(fs, n_t):
                if self._condA is None:
                    self._condA = eng.cond_prepare(fs, self._Xt)
                cqt = eng.predict_conditioned(fs, w, Xf, self._Xt, self._condA)[2]
            elif n_t > 0:  # n_t > 128: the constructor made sure the cross-covariance kernel covers the tasks
                cqt = eng.predict_cross(fs, Xf, self._Xt, w=w)[1]
            return mean, cqq, cqt
        self._require_cross("joint posterior")
        mean, cqq = eng.predict_cross(fs, Xf, None, w=w)
        cqt = eng.predict_cross(fs, Xf, self._Xt, w=w)[1] if n_t > 0 else None
        return mean, cqq, cqt

    @property
    def supports_candidate_gradients(self) -> bool:
        """Shapes the analytic-gradient kernels cover (n <= 512 points per task and what the prediction kernel
        covers, d <= 16, n_t <= 128); outside them the optimizer falls back to its zeroth-order acquisition search."""
        b = self._fitted.batch
        return b.n_max <= 512 and b.d <= 16 and self.num_train <= 128 and self.engine.predict_supported(self._fitted)

    def posterior_with_grad(self, X: torch.Tensor):
        """Posterior mean / variance [B] and their gradients wrt the candidates [B, d] (q = 1), un-standardised.

        What botorch's `optimize_acqf` gets by autograd through `ScaMLGP.forward` (eval branch, model.py:364-375) and
        the exact prediction strategy; here analytic: K_m^-1 k*_m on the tensor cores (`cond_prepare` at the
        candidates), the values from it (`csrc/scaml_gradval.cuh`), then the gradient contraction over all tasks
        (`csrc/scaml_grad.cuh`)."""
        eng, dev = self.engine, self.engine.device
        if X.dim() == 3:
            if X.shape[-2] != 1:
                raise NotImplementedError("candidate gradients cover q = 1 batches (the acquisition path)")
            X = X[:, 0, :]
        b = self._fitted.batch
        if not self.supports_candidate_gradients:
            raise NotImplementedError("candidate gradients need n <= 512 points per task (and within the prediction "
                                      f"kernel), d <= 16 and n_t <= 128; the model has {self._limits_text()} and "
                                      f"n_t = {self.num_train}")
        Xall = X.to(dev, DT).contiguous()
        w = self.pruned_weights()
        n_t = self.num_train
        if n_t > 0 and self._condA is None and self._sharded is None:
            self._condA = eng.cond_prepare(self._fitted, self._Xt)
        outs = []
        for lo in range(0, Xall.shape[0], 128):
            Xc = Xall[lo:lo + 128].contiguous()
            if self._sharded is not None:
                outs.append(self._sharded.posterior_with_grad(w, Xc, self._target_state() if n_t > 0 else None,
                                                              float(self.covar_module.outputscale)))
                continue
            U = eng.cond_prepare(self._fitted, Xc, w)  # pruned tasks skipped
            if n_t > 0:
                ts = self._target_state()
                pm, pv, cross = eng.prior_values(self._fitted, w, Xc, U, self._Xt, self._condA)
                mean, var, beta = eng.target_posterior_beta(ts, pm, pv, cross, Xc)
                dm, dv = eng.posterior_grad(self._fitted, w, Xc, U, ts, self._condA, beta)
            else:
                mean, pv, _ = eng.values_from_u(self._fitted, w, Xc, U)
                var = pv + float(self.covar_module.outputscale)
                dm, dv = eng.posterior_grad(self._fitted, w, Xc, U)
            outs.append((mean, var, dm, dv))
        return tuple(torch.cat([o[i] for o in outs]).to(X.device) for i in range(4))

    def posterior_blocks(self, X: torch.Tensor):
        """Joint posterior of b blocks of q points, X [b, q, d], 1 <= q <= 16, and its vector-Jacobian product.

        Returns mean [b, q], cov [b, q, q] (un-standardised, the blocks `posterior(X)` returns for q > 1) and
        `vjp(g_mean [b, q], g_cov [b, q, q]) -> dX [b, q, d]`, the gradient wrt X of sum(g_mean mean) + sum(g_cov cov):
        what a batch acquisition (qUCB, qEI) hands back from autograd on the small (mean, cov) leaves.  The blocks
        come from U = K_m^-1 k*_m on the tensor cores (`cond_prepare` at the points) and `csrc/scaml_qblock.cuh`,
        in launches of <= 128 points that never split a block.  `vjp` may be called once: it consumes the U of every
        launch, which stay allocated until then (one [M, n_pad, 128] array per 128 points)."""
        eng, dev = self.engine, self.engine.device
        if X.dim() != 3:
            raise ValueError(f"posterior_blocks expects X [b, q, d], got shape {tuple(X.shape)}")
        nb_all, q, d = X.shape
        if self._sharded is not None:
            raise NotImplementedError("q-point blocks are not available for task-sharded source GPs (group=)")
        if not 1 <= q <= 16:
            raise NotImplementedError(f"q-point blocks cover 1 <= q <= 16 points per block, got q = {q}")
        if not self.supports_candidate_gradients:
            raise NotImplementedError("q-point blocks need n <= 512 points per task (and within the prediction "
                                      f"kernel), d <= 16 and n_t <= 128; the model has {self._limits_text()} and "
                                      f"n_t = {self.num_train}")
        fs, n_t = self._fitted, self.num_train
        Xall = X.reshape(-1, d).to(dev, DT).contiguous()
        w = self.pruned_weights()
        kernel_t = self.hyper_spec().kernel
        if n_t > 0:
            ts = self._target_state()
            theta_t = ts.theta.clone()
            theta_t[d + 1] = 0.0  # noise-free kernel values
            if self._condA is None:
                self._condA = eng.cond_prepare(fs, self._Xt)
        else:
            ts, theta_t = None, self._target_kernel_theta(d).reshape(-1)
        step = (128 // q) * q
        idx = torch.arange(step, device=dev).reshape(-1, q)
        means, covs, launches = [], [], []
        for lo in range(0, Xall.shape[0], step):
            Xc = Xall[lo:lo + step].contiguous()
            nb = Xc.shape[0] // q
            U = eng.cond_prepare(fs, Xc, w)  # pruned tasks skipped
            cov = eng.qblock_cov(fs, w, Xc, U, q)
            Z = torch.cat([self._Xt, Xc]) if n_t > 0 else Xc
            kt = eng.kernel_matrix(Z.unsqueeze(0).contiguous(), theta_t.reshape(1, -1), kernel_t)[0]
            ib = idx[:nb]
            kqq = kt[n_t:, n_t:][ib.unsqueeze(2), ib.unsqueeze(1)]  # [nb, q, q] diagonal blocks
            beta = None
            if n_t > 0:
                pm, pv, cross = eng.prior_values(fs, w, Xc, U, self._Xt, self._condA)
                mean, _, beta = eng.target_posterior_beta(ts, pm, pv, cross, Xc)
                S2 = ts.s_all ** 2
                ks = (cross / S2 + kt[n_t:, :n_t]).reshape(nb, q, n_t)  # standardised cross-covariance with X_t
                cov = cov + S2 * (kqq - ks @ beta[:, :n_t].reshape(nb, q, n_t).transpose(1, 2))
                cov = 0.5 * (cov + cov.transpose(1, 2))
            else:  # prior-only model (optimizer.py:135-141): no outcome transform
                mean = eng.values_from_u(fs, w, Xc, U)[0]
                cov = cov + kqq
            means.append(mean.reshape(nb, q))
            covs.append(cov)
            launches.append((lo, Xc, U, beta))
        consumed = []

        def vjp(g_mean: torch.Tensor, g_cov: torch.Tensor) -> torch.Tensor:
            if consumed:
                raise RuntimeError("the vjp of posterior_blocks can be called once (it consumes the cached U)")
            consumed.append(True)
            gm = g_mean.reshape(-1).to(dev, DT)
            gc = g_cov.reshape(-1, q, q).to(dev, DT)
            outs = []
            for lo, Xc, U, beta in launches:
                B = Xc.shape[0]
                outs.append(eng.qblock_vjp(fs, w, Xc, U, q, gm[lo:lo + B], gc[lo // q:(lo + B) // q], theta_t, kernel_t,
                                           ts, self._condA if n_t > 0 else None, beta))
            launches.clear()
            return torch.cat(outs).reshape(nb_all, q, d).to(X.device)

        return torch.cat(means).to(X.device), torch.cat(covs).to(X.device), vjp

    def _posterior_fused(self, Xc: torch.Tensor, w: torch.Tensor):
        """n_t > 0, q = 1: prior mean / variance and the cross-covariance with the target inputs in ONE prediction
        launch (the k*^T A_m contraction rides on the k* tiles), then the n_t-dimensional conditioning."""
        eng = self.engine
        if self._condA is None:
            self._condA = eng.cond_prepare(self._fitted, self._Xt)
        pm, pv, cross = eng.predict_conditioned(self._fitted, w, Xc, self._Xt, self._condA)
        return eng.target_posterior(self._target_state(), pm, pv, cross, Xc)
