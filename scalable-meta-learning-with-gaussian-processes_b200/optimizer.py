# The constructor signature and the `report` skeleton are derived from scamlgp/optimizer.py of
# boschresearch/Scalable-Meta-Learning-with-Gaussian-Processes, Copyright (c) 2024 Robert Bosch GmbH, AGPL-3.0.
"""ScaMLGPBO -- mirror of the reference optimizer (scamlgp/optimizer.py:27-185) on the B200 engine.

The reference derives from blackboxopt's `SingleObjectiveBOTorchOptimizer` (not in its tree, not
installable here); the few behaviours of that base class the reference relies on and its tests assert
(SURVEY A.9: `X`, `losses`, `pending_specifications`, `report`, `generate_evaluation_specification`,
`OptimizerNotReady`) are restated in `_SingleObjectiveBase`.  Two acquisition optimisers: `optimize_acqf_lbfgsb`
(default; botorch's recipe -- raw-sample screening, then L-BFGS-B over all restarts with the analytic posterior
gradients of `csrc/scaml_grad.cuh`) and `optimize_acqf_batched` (zeroth order: shrinking-box refinement rounds, each
one posterior launch over every start x every perturbation; `af_optimizer_kwargs={"method": "batched"}`).
"""
from __future__ import annotations

import logging
from typing import Any, Callable, Dict, Hashable, Iterable, List, Optional, Union

import numpy as np
import torch

from .model import ScaMLGP, meta_fit_scamlgp
from .space import (Evaluation, EvaluationsError, EvaluationSpecification, Objective, OptimizerNotReady,
                    ParameterSpace, filter_y_nans, impute_nans_with_constant, to_numerical)
from .utils import UpperConfidenceBound, metadata_to_numerical, optimize_marginal_likelihood, qUpperConfidenceBound


def optimize_acqf_batched(af: Callable[[torch.Tensor], torch.Tensor], bounds: np.ndarray, generator: torch.Generator,
                          raw_samples: int = 4096, num_restarts: int = 8, rounds: int = 8,
                          perturbations: int = 128) -> torch.Tensor:
    """Maximise af over the box `bounds` [d, 2] (q = 1).  Returns the best point [d]."""
    lo = torch.tensor(bounds[:, 0], dtype=torch.float64)
    hi = torch.tensor(bounds[:, 1], dtype=torch.float64)
    d = lo.numel()
    X0 = lo + (hi - lo) * torch.rand(raw_samples, d, dtype=torch.float64, generator=generator)
    v0 = af(X0).reshape(-1).cpu()
    top = torch.topk(v0, min(num_restarts, raw_samples))
    starts, best = X0[top.indices].clone(), top.values.clone()
    radius = 0.25 * (hi - lo)
    for _ in range(rounds):
        S = starts.shape[0]
        noise = (2.0 * torch.rand(S, perturbations, d, dtype=torch.float64, generator=generator) - 1.0) * radius
        cand = torch.minimum(torch.maximum(starts.unsqueeze(1) + noise, lo), hi)
        vals = af(cand.reshape(-1, d)).reshape(S, perturbations).cpu()
        bv, bi = vals.max(dim=1)
        better = bv > best
        pick = cand[torch.arange(S), bi]
        starts = torch.where(better.unsqueeze(1), pick, starts)
        best = torch.where(better, bv, best)
        radius = radius * 0.5
    return starts[int(torch.argmax(best))]


def optimize_acqf_lbfgsb(af, bounds: np.ndarray, generator: torch.Generator, raw_samples: int = 1024,
                         num_restarts: int = 32, maxiter: int = 60, q: int = 1) -> torch.Tensor:
    """Maximise af over the box `bounds` [d, 2] the way botorch's `optimize_acqf` does for the reference:
    raw-sample screening, then scipy L-BFGS-B on the SUM of the acquisition values of all restarts (they are
    independent, so one optimiser run drives them in lock-step; botorch gen_candidates_scipy) with the analytic
    gradient of `af.value_and_grad` -- one posterior-with-gradient launch sequence per function evaluation.

    q = 1: af takes candidates [B, d]; returns the best point [d].  q > 1: af is a batch acquisition over blocks
    [b, q, d] (qUpperConfidenceBound, qExpectedImprovement); `raw_samples` random q-batches are screened and the
    q points of every restart are optimised jointly (num_restarts x q x d variables); returns the best batch [q, d]."""
    from scipy.optimize import minimize

    lo = torch.tensor(bounds[:, 0], dtype=torch.float64)
    hi = torch.tensor(bounds[:, 1], dtype=torch.float64)
    d = lo.numel()
    if q > 1:
        return optimize_acqf_lbfgsb_blocks(af, bounds, generator, raw_samples, num_restarts, maxiter, q)
    X0 = lo + (hi - lo) * torch.rand(raw_samples, d, dtype=torch.float64, generator=generator)
    v0 = af(X0).reshape(-1).cpu()
    top = torch.topk(v0, min(num_restarts, raw_samples))
    starts = X0[top.indices].clone()
    S = starts.shape[0]

    def fun(xflat: np.ndarray):
        X = torch.from_numpy(xflat.reshape(S, d).copy())
        val, grad = af.value_and_grad(X)
        return -float(val.sum()), -grad.cpu().numpy().reshape(-1).astype(np.float64)

    res = minimize(fun, starts.numpy().reshape(-1), jac=True, method="L-BFGS-B",
                   bounds=[(float(lo[k]), float(hi[k])) for _ in range(S) for k in range(d)],
                   options=dict(maxiter=int(maxiter)))
    Xo = torch.minimum(torch.maximum(torch.from_numpy(res.x.reshape(S, d).copy()), lo), hi)
    # never worse than the best raw sample: score the refined points and the starts together
    cand = torch.cat([Xo, starts])
    vals = af(cand).reshape(-1).cpu()
    return cand[int(torch.argmax(vals))]


def optimize_acqf_lbfgsb_blocks(af, bounds: np.ndarray, generator: torch.Generator, raw_samples: int = 1024,
                                num_restarts: int = 32, maxiter: int = 60, q: int = 1) -> torch.Tensor:
    """`optimize_acqf_lbfgsb` for a batch acquisition over blocks [b, q, d], any q >= 1; returns the best batch [q, d]."""
    from scipy.optimize import minimize

    lo = torch.tensor(bounds[:, 0], dtype=torch.float64)
    hi = torch.tensor(bounds[:, 1], dtype=torch.float64)
    d = lo.numel()
    X0 = lo + (hi - lo) * torch.rand(raw_samples, q, d, dtype=torch.float64, generator=generator)
    v0 = af(X0).reshape(-1).cpu()
    top = torch.topk(v0, min(num_restarts, raw_samples))
    starts = X0[top.indices].clone()
    S = starts.shape[0]

    def fun(xflat: np.ndarray):
        X = torch.from_numpy(xflat.reshape(S, q, d).copy())
        val, grad = af.value_and_grad(X)
        return -float(val.sum()), -grad.cpu().numpy().reshape(-1).astype(np.float64)

    res = minimize(fun, starts.numpy().reshape(-1), jac=True, method="L-BFGS-B",
                   bounds=[(float(lo[k]), float(hi[k])) for _ in range(S * q) for k in range(d)],
                   options=dict(maxiter=int(maxiter)))
    Xo = torch.minimum(torch.maximum(torch.from_numpy(res.x.reshape(S, q, d).copy()), lo), hi)
    cand = torch.cat([Xo, starts])
    vals = af(cand).reshape(-1).cpu()
    return cand[int(torch.argmax(vals))]


class _SingleObjectiveBase:
    """The slice of blackboxopt's SingleObjectiveBOTorchOptimizer the reference uses (SURVEY A.9)."""

    def __init__(self, search_space: ParameterSpace, objective: Objective, model, acquisition_function_factory,
                 af_optimizer_kwargs: Optional[dict], num_initial_random_samples: int,
                 max_pending_evaluations: Optional[int], batch_shape, logger: Optional[logging.Logger],
                 seed: Optional[int], torch_dtype: torch.dtype):
        self.search_space = search_space
        self.objective = objective
        self.objectives = [objective]
        self.model = model
        self.acquisition_function_factory = acquisition_function_factory
        self.af_opt_kwargs = dict(af_optimizer_kwargs or {})
        self.num_initial_random = num_initial_random_samples
        self.max_pending_evaluations = max_pending_evaluations
        self.batch_shape = batch_shape
        self.logger = logger or logging.getLogger("scamlgp_b200")
        self.seed = seed
        self.torch_dtype = torch_dtype
        self.X = torch.empty((0, len(search_space)), dtype=torch_dtype)
        self.losses = torch.empty((0, 1), dtype=torch_dtype)
        self.pending_specifications: Dict[int, EvaluationSpecification] = {}
        self._next_id = 0
        self._gen = torch.Generator().manual_seed(0 if seed is None else int(seed))
        if seed is not None:
            search_space.seed(seed)

    # -- bookkeeping ------------------------------------------------------------------------------- #
    def _validate(self, evaluation: Evaluation) -> None:
        if self.objective.name not in evaluation.objectives:
            raise EvaluationsError(f"Evaluation does not report the objective '{self.objective.name}': "
                                   f"{list(evaluation.objectives)}")
        unknown = set(evaluation.configuration) - set(self.search_space.parameter_names)
        if unknown:
            raise EvaluationsError(f"Configuration has parameters outside the search space: {sorted(unknown)}")

    def _update_internal_evaluation_data(self, evaluations: Iterable[Evaluation]) -> None:
        evaluations = list(evaluations)
        for e in evaluations:
            self._validate(e)
        X, Y = to_numerical(evaluations, self.search_space, self.objectives, self.batch_shape, self.torch_dtype)
        self.X = torch.cat([self.X, impute_nans_with_constant(X)], dim=0)
        self.losses = torch.cat([self.losses, Y], dim=0)
        for e in evaluations:
            self.pending_specifications.pop(e.optimizer_info.get("evaluation_id"), None)

    # -- suggestions ------------------------------------------------------------------------------- #
    def _spec(self, configuration: Dict[str, Any]) -> EvaluationSpecification:
        eval_id = self._next_id
        self._next_id += 1
        spec = EvaluationSpecification(configuration=configuration, optimizer_info={"evaluation_id": eval_id})
        self.pending_specifications[eval_id] = spec
        return spec

    def _model_for_acquisition(self):
        """The model the acquisition function sees.  With evaluations pending (max_pending_evaluations > 1) the
        reference's base class conditions a fantasy model on the pending points (SURVEY A.9); here the pending
        points are fantasised at the posterior mean ("kriging believer"): the mean is unchanged, the variance
        collapses around them, so concurrent suggestions spread out.  Hyper-parameters are not refitted."""
        if not self.pending_specifications or getattr(self.model, "num_train", 0) == 0:
            return self.model
        Xp = torch.tensor(np.stack([self.search_space.to_numerical(s.configuration)
                                    for s in self.pending_specifications.values()]), dtype=self.torch_dtype)
        Xp = impute_nans_with_constant(Xp)
        base = self.model
        yp = base.posterior(Xp).mean.reshape(-1, 1).to(self.torch_dtype).cpu()
        X_all = torch.cat([base.train_inputs[0].to(self.torch_dtype), Xp], dim=0)
        Y_all = torch.cat([base._train_Y.to(self.torch_dtype), yp], dim=0)
        fantasy = ScaMLGP(X_all, Y_all, self.source_gps, likelihood=base.likelihood, covar_module=base.covar_module,
                          **self.model_kwargs)
        fantasy.raw_weights = base.raw_weights.clone()
        return fantasy.eval()

    def generate_evaluation_specification(self) -> EvaluationSpecification:
        if (self.max_pending_evaluations is not None
                and len(self.pending_specifications) >= self.max_pending_evaluations):
            raise OptimizerNotReady(f"{len(self.pending_specifications)} evaluations are pending "
                                    f"(max_pending_evaluations = {self.max_pending_evaluations})")
        n_valid = int((~torch.isnan(self.losses)).sum())
        if len(self.X) < self.num_initial_random or (self.num_initial_random > 0 and n_valid == 0):
            return self._spec(self.search_space.sample())
        af = self.acquisition_function_factory(self._model_for_acquisition())
        if getattr(af, "maximize", False):
            raise ValueError("Only acquisition functions to be minimized are supported")
        d = len(self.search_space)
        kw = self.af_opt_kwargs
        has_grad = hasattr(af, "value_and_grad") and bool(getattr(getattr(af, "model", None),
                                                                 "supports_candidate_gradients", False))
        method = str(kw.get("method", "lbfgsb" if has_grad else "batched"))
        if self.search_space.is_all_continuous and method == "lbfgsb":
            x = optimize_acqf_lbfgsb(af, self.search_space.numerical_bounds(), self._gen,
                                     raw_samples=int(kw.get("raw_samples", 1024)),
                                     num_restarts=int(kw.get("num_restarts", 32)), maxiter=int(kw.get("maxiter", 60)))
            configuration = self.search_space.from_numerical(x.numpy())
        elif self.search_space.is_all_continuous:
            x = optimize_acqf_batched(af, self.search_space.numerical_bounds(), self._gen,
                                      raw_samples=int(kw.get("raw_samples", 4096)),
                                      num_restarts=int(kw.get("num_restarts", 8)), rounds=int(kw.get("rounds", 8)),
                                      perturbations=int(kw.get("perturbations", 128)))
            configuration = self.search_space.from_numerical(x.numpy())
        else:
            # discrete / conditional spaces: score a few thousand sampled configurations (optimize_acqf_discrete)
            n_choices = int(kw.get("num_random_choices", 5000))
            configs = [self.search_space.sample() for _ in range(n_choices)]
            Xn = torch.tensor(np.stack([self.search_space.to_numerical(c) for c in configs]), dtype=torch.float64)
            vals = af(impute_nans_with_constant(Xn)).reshape(-1).cpu()
            configuration = configs[int(torch.argmax(vals))]
        return self._spec(configuration)


class ScaMLGPBO(_SingleObjectiveBase):
    def __init__(self, search_space: ParameterSpace, objective: Objective,
                 meta_data: Dict[Hashable, Iterable[Evaluation]], gp_likelihood=None, gp_kernel=None,
                 base_gp_kernel=None, acquisition_function_factory: Optional[Callable] = None,
                 af_optimizer_kwargs: Optional[dict] = None, num_initial_random_samples: int = 0,
                 max_pending_evaluations: Optional[int] = 1, num_restarts_log_likelihood: int = 5,
                 model_kwargs: Optional[Dict[str, Any]] = None, logger: Optional[logging.Logger] = None,
                 seed: Optional[int] = None, torch_dtype: torch.dtype = torch.float64, *, engine=None,
                 fit_options: Optional[dict] = None, group=None,
                 batch_acquisition_function_factory: Optional[Callable] = None):
        """Single objective meta-learning BO optimizer with ScaML-GP as surrogate
        (reference scamlgp/optimizer.py:28-154: same arguments; `engine` / `fit_options` / `group` are additions).

        group: torch.distributed process group (True = default group): the meta-tasks are block-partitioned over its
        ranks -- the meta-fit (optimizer.py:128-133), the per-report caches (model.py:278-289) and every posterior
        (model.py:364-375) fan out over the GPUs with one all_gather / all_reduce each (sharded.py).  Every rank
        runs the same optimizer with the same seed and proposes the same configurations.

        batch_acquisition_function_factory: model -> batch acquisition over q-point blocks, used by
        `generate_evaluation_specifications(q)`; default qUpperConfidenceBound (beta = 9)."""
        n_features = len(search_space)
        self.batch_acquisition_function_factory = batch_acquisition_function_factory or qUpperConfidenceBound
        batch_shape = torch.Size()
        if acquisition_function_factory is None:
            acquisition_function_factory = UpperConfidenceBound
        metadata_numerical = metadata_to_numerical(meta_data, search_space, objective, batch_shape, torch_dtype)
        self.num_restarts_log_likelihood = num_restarts_log_likelihood
        self.fit_options = fit_options
        # NOTE: like the reference (optimizer.py:128-133) the meta-fit always uses the default 5 restarts
        self.source_gps = meta_fit_scamlgp(metadata_numerical, likelihood=gp_likelihood, covar_module=base_gp_kernel,
                                           seed=seed, engine=engine, fit_options=fit_options, group=group)
        self.model_kwargs = {} if model_kwargs is None else model_kwargs
        model = ScaMLGP(train_X=torch.empty((*batch_shape, 0, n_features), dtype=torch_dtype),
                        train_Y=torch.empty((*batch_shape, 0, 1), dtype=torch_dtype), source_gps=self.source_gps,
                        likelihood=gp_likelihood, covar_module=gp_kernel)
        super().__init__(search_space=search_space, objective=objective, model=model,
                         acquisition_function_factory=acquisition_function_factory,
                         af_optimizer_kwargs=af_optimizer_kwargs,
                         num_initial_random_samples=num_initial_random_samples,
                         max_pending_evaluations=max_pending_evaluations, batch_shape=batch_shape, logger=logger,
                         seed=seed, torch_dtype=torch_dtype)

    def generate_evaluation_specifications(self, q: int) -> List[EvaluationSpecification]:
        """q configurations chosen jointly, for q concurrent workers; all are registered as pending.

        The batch acquisition (`batch_acquisition_function_factory`) sees the model conditioned on the evaluations
        already pending (the kriging-believer fantasy of `generate_evaluation_specification`) and L-BFGS-B optimises
        the q points together.  Before `num_initial_random_samples` observations exist the q points are random
        samples.  Raises OptimizerNotReady when pending + q exceeds `max_pending_evaluations`, NotImplementedError
        for search spaces that are not all continuous and for q > 16."""
        q = int(q)
        if q < 1:
            raise ValueError(f"q must be at least 1, got {q}")
        if not self.search_space.is_all_continuous:
            raise NotImplementedError("batch proposals (q points at once) cover all-continuous search spaces")
        if (self.max_pending_evaluations is not None
                and len(self.pending_specifications) + q > self.max_pending_evaluations):
            raise OptimizerNotReady(f"{len(self.pending_specifications)} evaluations are pending, {q} more requested "
                                    f"(max_pending_evaluations = {self.max_pending_evaluations})")
        n_valid = int((~torch.isnan(self.losses)).sum())
        if len(self.X) < self.num_initial_random or (self.num_initial_random > 0 and n_valid == 0):
            return [self._spec(self.search_space.sample()) for _ in range(q)]
        af = self.batch_acquisition_function_factory(self._model_for_acquisition())
        if getattr(af, "maximize", False):
            raise ValueError("Only acquisition functions to be minimized are supported")
        kw = self.af_opt_kwargs
        X = optimize_acqf_lbfgsb_blocks(af, self.search_space.numerical_bounds(), self._gen,
                                        raw_samples=int(kw.get("raw_samples", 1024)),
                                        num_restarts=int(kw.get("num_restarts", 32)),
                                        maxiter=int(kw.get("maxiter", 60)), q=q)
        return [self._spec(self.search_space.from_numerical(x.numpy())) for x in X.reshape(q, -1)]

    def report(self, evaluations: Union[Evaluation, Iterable[Evaluation]]):
        """Book-keep the evaluations and refit the ScaML-GP target model (reference optimizer.py:156-185)."""
        _evals = evaluations if isinstance(evaluations, list) else [evaluations]
        from .model import MAX_TARGET_POINTS

        if int((~torch.isnan(self.losses)).sum()) + len(_evals) > MAX_TARGET_POINTS:  # before any book-keeping changes
            raise NotImplementedError(f"more than {MAX_TARGET_POINTS} target observations: exact inference is defined "
                                      "up to that size (SURVEY A.5); the optimizer state is unchanged")
        super()._update_internal_evaluation_data(_evals)
        if len(self.X) < self.num_initial_random:
            return
        x_filtered, y_filtered = filter_y_nans(self.X, self.losses)
        if x_filtered.numel() == 0:
            return
        self.model = ScaMLGP(x_filtered, y_filtered, self.source_gps, likelihood=self.model.likelihood,
                             covar_module=self.model.covar_module, **self.model_kwargs)
        optimize_marginal_likelihood(self.model, self.num_restarts_log_likelihood, generator=self._gen,
                                     **(self.fit_options or {}))
        self.model.eval()
