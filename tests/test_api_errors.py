"""Error behaviour of the public API at the same points as the reference (no GPU needed: the checks run before
any kernel is launched, or through the emulation engine)."""
import pytest
import torch

from scamlgp_b200._capi import HyperSpec, ScamlError, load_cuda_library
from scamlgp_b200.model import ScaMLGP, _compute_target_prior, meta_fit_scamlgp, significant_weights_mask
from scamlgp_b200.modules import (GammaPrior, GaussianLikelihood, Interval, MaternKernel, ModelFittingError, RBFKernel,
                                  ScaleKernel, SupervisedDataset)
from scamlgp_b200.utils import UpperConfidenceBound, sample_all_priors, validate_meta_data

DT = torch.float64


@pytest.fixture(scope="module")
def emu_engine(emu_lib):
    from tests.emu_engine import EmuEngine

    return EmuEngine(emu_lib)


def _ds(n, d, ydim=1):
    g = torch.Generator().manual_seed(n + d)
    return SupervisedDataset(torch.rand(n, d, dtype=DT, generator=g), torch.rand(n, ydim, dtype=DT, generator=g))


def test_validate_meta_data_messages_match_reference():
    """scamlgp/utils.py:112-136."""
    with pytest.raises(ValueError, match="Empty meta data"):
        validate_meta_data({})
    with pytest.raises(ValueError, match="Dimensions of tasks a and b do not match"):
        validate_meta_data({"a": _ds(4, 2), "b": _ds(4, 3)})
    with pytest.raises(ValueError, match="output dimension of task b is 2 but must be one"):
        validate_meta_data({"a": _ds(4, 2), "b": _ds(4, 2, ydim=2)})
    validate_meta_data({"a": _ds(4, 2), "b": _ds(7, 2)})  # ragged n is fine


def test_significant_weights_mask_matches_reference_formula():
    """scamlgp/model.py:192-215: w_i sigma_i M / sum_j w_j sigma_j >= tau."""
    w = torch.tensor([0.5, 1e-6, 0.2, 0.0], dtype=DT)
    s = torch.tensor([1.0, 2.0, 0.5, 3.0], dtype=DT)
    m = significant_weights_mask(w, s, 1e-3)
    assert m.tolist() == [True, False, True, False]
    assert significant_weights_mask(torch.ones(3, dtype=DT), torch.ones(3, dtype=DT), 1e-3).all()


def test_engine_refuses_to_run_without_cuda_and_library_must_exist(tmp_path):
    from scamlgp_b200._capi import ScamlLib
    from scamlgp_b200.engine import Engine

    if not torch.cuda.is_available():
        with pytest.raises(ScamlError, match="no CPU fallback"):
            Engine()
    with pytest.raises(ScamlError, match="not found"):
        ScamlLib(str(tmp_path / "libmissing.so"))
    assert load_cuda_library().version().endswith("sm_100a")  # the product library is built in-tree


def test_kernel_family_checks():
    with pytest.raises(ValueError):
        MaternKernel(nu=1.0, ard_num_dims=2)
    with pytest.raises(TypeError):
        from scamlgp_b200.modules import hyper_spec_of

        hyper_spec_of(GaussianLikelihood(), RBFKernel(ard_num_dims=2))  # must be ScaleKernel(base)
    k = ScaleKernel(MaternKernel(nu=2.5, ard_num_dims=3, lengthscale_constraint=Interval(1e-3, 10.0, 0.7)))
    assert abs(float(k.base_kernel.lengthscale[0, 0]) - 0.7) < 1e-12
    k.base_kernel.lengthscale = 0.3
    assert torch.allclose(k.base_kernel.lengthscale, torch.full((1, 3), 0.3, dtype=DT))


def test_sample_all_priors_rejects_incompatible_prior_and_constraint():
    """utils.py:47-69: a prior whose support misses the constraint interval fails after num_retries."""

    class M:
        def __init__(self):
            self.likelihood = GaussianLikelihood(noise_prior=GammaPrior(400.0, 1.0),  # mass around 400 >> 1e-2
                                                 noise_constraint=Interval(1e-8, 1e-2, 1e-3))

        def named_priors(self):
            yield ("likelihood.noise_covar.noise_prior", self.likelihood, self.likelihood.noise_prior,
                   lambda m: m.noise, lambda m, v: setattr(m, "noise", v))

    with pytest.raises(RuntimeError, match="failed 5 times"):
        sample_all_priors(M(), generator=torch.Generator().manual_seed(0))


def test_model_errors_through_emulation(emu_engine):
    md = {"a": _ds(6, 2), "b": _ds(5, 2)}
    gps = meta_fit_scamlgp(md, num_restarts_log_likelihood=0, seed=0, engine=emu_engine, fit_options=dict(maxiter=2))
    # number of weights must equal the number of source GPs (model.py:123-127)
    with pytest.raises(ValueError, match="does not equal the number of weights"):
        _compute_target_prior(torch.rand(3, 2, dtype=DT), list(gps.values()), torch.ones(3, dtype=DT), emu_engine)
    # batched meta-data are not supported (the reference optimizer never produces them)
    with pytest.raises(NotImplementedError):
        meta_fit_scamlgp({"a": SupervisedDataset(torch.rand(2, 4, 2, dtype=DT), torch.rand(2, 4, 1, dtype=DT))},
                         engine=emu_engine)
    model = ScaMLGP(torch.empty(0, 2, dtype=DT), torch.empty(0, 1, dtype=DT), gps, engine=emu_engine)
    assert model.outcome_transform is None and model.num_train == 0  # empty input: no standardisation (model.py:307-308)
    assert torch.allclose(model.weights, torch.full((2,), 0.5, dtype=DT))
    pj = model.posterior(torch.rand(4, 2, 2, dtype=DT))  # q > 1: joint posterior per batch element
    assert pj.mean.shape == (4, 2, 1) and pj.mvn.covariance_matrix.shape == (4, 2, 2)
    with pytest.raises(NotImplementedError, match="q <= 128"):
        model.posterior(torch.rand(1, 129, 2, dtype=DT))
    with pytest.raises(TypeError, match="ScaMLGP or a SourceGP"):
        from scamlgp_b200.utils import optimize_marginal_likelihood

        optimize_marginal_likelihood(object())
    from scamlgp_b200.model import max_target_points

    assert max_target_points(emu_engine, 2) == 117 and max_target_points(emu_engine, 16) == 113  # 227 KB, grows with d
    with pytest.raises(NotImplementedError, match="n_t <= 800"):
        ScaMLGP(torch.rand(801, 2, dtype=DT), torch.rand(801, 1, dtype=DT), gps, engine=emu_engine)
    with pytest.raises(ValueError):
        UpperConfidenceBound(model, maximize=True)
    # all restarts failing -> ModelFittingError (utils.py:207-212): NaN targets poison every row
    bad = {"a": SupervisedDataset(torch.rand(5, 2, dtype=DT), torch.full((5, 1), float("nan"), dtype=DT))}
    with pytest.raises(ModelFittingError, match="failed for all attempts"):
        meta_fit_scamlgp(bad, num_restarts_log_likelihood=1, seed=0, engine=emu_engine, fit_options=dict(maxiter=2))


def test_target_entry_points_reject_an_unknown_kernel_family(emu_engine):
    """The target-GP objective, its in-kernel jitter ladder and the target factorisation refuse a kernel family id
    outside 0..3, like every other entry point, instead of running some other family."""
    M, nt, d = 2, 3, 2
    g = torch.Generator().manual_seed(3)
    sm, sc = torch.rand(nt, M, dtype=DT, generator=g), torch.rand(nt, nt, M, dtype=DT, generator=g)
    Xt, yt = torch.rand(nt, d, dtype=DT, generator=g), torch.rand(nt, dtype=DT, generator=g)
    w, th = torch.ones(1, M, dtype=DT), torch.zeros(1, d + 2, dtype=DT)
    spec = HyperSpec.target(kernel=4)
    with pytest.raises(ScamlError, match="scaml_target_lml_grad: bad argument"):
        emu_engine.target_lml_grad(sm, sc, Xt, yt, w, th, 0.0, 1.0, spec)
    with pytest.raises(ScamlError, match="scaml_target_lml_grad_ladder: bad argument"):
        emu_engine.target_lml_grad_safe(sm, sc, Xt, yt, w, th, 0.0, 1.0, spec)
    with pytest.raises(ScamlError, match="scaml_target_factorize: bad argument"):
        emu_engine.target_factorize(sm, sc, Xt, yt, w[0], th[0], 0.0, 1.0, spec)


def test_acquisition_optimiser_falls_back_without_gradient_support():
    """Models outside the shapes of the analytic-gradient kernels (or custom acquisition functions without
    `value_and_grad`) take the zeroth-order search: the default method follows `supports_candidate_gradients`."""
    import numpy as np
    import torch

    from scamlgp_b200 import optimizer as opt_mod

    calls = []

    class _Model:
        supports_candidate_gradients = False

    class _AF:
        maximize = False
        model = _Model()

        def __call__(self, X):
            return -((X - 0.5) ** 2).sum(-1)

        def value_and_grad(self, X):  # must not be used
            raise AssertionError("gradient path taken for a model without gradient support")

    class _Space:
        is_all_continuous = True
        parameter_names = ["x"]

        def __len__(self):
            return 1

        def numerical_bounds(self):
            return np.array([[0.0, 1.0]])

        def from_numerical(self, x):
            calls.append(float(x[0]))
            return {"x": float(x[0])}

        def seed(self, s):
            pass

    base = opt_mod._SingleObjectiveBase.__new__(opt_mod._SingleObjectiveBase)
    base.search_space, base.max_pending_evaluations, base.pending_specifications = _Space(), None, {}
    base.losses, base.X = torch.zeros(1, 1, dtype=torch.float64), torch.zeros(1, 1, dtype=torch.float64)
    base.num_initial_random, base.af_opt_kwargs, base._next_id = 0, dict(raw_samples=64, num_restarts=4, rounds=3), 0
    base._gen = torch.Generator().manual_seed(0)
    base.model = _Model()
    base.acquisition_function_factory = lambda model: _AF()
    spec = base.generate_evaluation_specification()
    assert abs(spec.configuration["x"] - 0.5) < 0.05 and len(calls) == 1


def test_to_numerical_batch_vector_paths_equal_the_scalar_conversion():
    """ParameterSpace.to_numerical_batch (the meta-data conversion of metadata_to_numerical, reference
    scamlgp/utils.py:98-106) has a one-shot array path for all-numeric spaces and a per-column path otherwise; both
    must give exactly what the value-by-value `to_numerical` gives, including inactive (None / missing) entries."""
    import numpy as np

    from scamlgp_b200.space import CategoricalParameter, ContinuousParameter, IntegerParameter, ParameterSpace

    rng = np.random.default_rng(0)
    num = ParameterSpace()
    for k in range(4):
        num.add(ContinuousParameter(f"x{k}", (-1.0, 3.0)))
    num.add(IntegerParameter("i", (2, 11)))
    cfgs = [{**{f"x{k}": float(rng.uniform(-1, 3)) for k in range(4)}, "i": int(rng.integers(2, 12))} for _ in range(200)]
    ref = np.stack([num.to_numerical(c) for c in cfgs])
    assert np.array_equal(num.to_numerical_batch(cfgs), ref)            # one array conversion
    cfgs[7]["x2"] = None
    del cfgs[9]["i"]
    ref = np.stack([num.to_numerical(c) for c in cfgs])
    assert np.array_equal(num.to_numerical_batch(cfgs), ref, equal_nan=True)   # falls back column by column
    mixed = ParameterSpace()
    mixed.add(ContinuousParameter("lr", (1e-4, 1.0)))
    mixed.add(CategoricalParameter("opt", ["sgd", "adam", "lion"]))
    cfgs = [{"lr": float(rng.uniform(1e-4, 1)), "opt": ["sgd", "adam", "lion"][int(rng.integers(0, 3))]} for _ in range(50)]
    ref = np.stack([mixed.to_numerical(c) for c in cfgs])
    assert np.array_equal(mixed.to_numerical_batch(cfgs), ref)


def test_dataset_tensors_and_uniform_upload_fast_paths():
    """botorch's SupervisedDataset exposes X / Y as attributes with `.shape` AND as callables (reference model.py:180-181
    vs utils.py:117-118); the stand-in keeps both, and the stacked upload of uniform tasks equals the row-block copies of
    the ragged path."""
    from scamlgp_b200.engine import SourceBatch
    from scamlgp_b200.modules import SupervisedDataset

    g = torch.Generator().manual_seed(0)
    X = torch.rand(5, 7, 3, dtype=torch.float64, generator=g)
    Y = torch.rand(5, 7, 1, dtype=torch.float64, generator=g)
    ds = SupervisedDataset(X[0], Y[0])
    assert ds.X.shape == (7, 3) and ds.Y.shape == (7, 1)
    assert type(ds.X()) is torch.Tensor and torch.equal(ds.X(), X[0]) and torch.equal(ds.Y(), Y[0])
    assert type(ds.X + 1.0) is torch.Tensor  # arithmetic leaves the container type
    tasks = [(X[i], Y[i]) for i in range(5)]
    fast = SourceBatch.from_ragged(tasks, "cpu")
    slow = SourceBatch.from_ragged(tasks, "cpu", n_max=8)  # padded by one row: the general path
    assert fast.uniform and not slow.uniform
    assert torch.equal(fast.X, slow.X[:, :7]) and torch.equal(fast.Y_raw, slow.Y_raw[:, :7])
    assert torch.equal(fast.n_valid, slow.n_valid)
    assert torch.allclose(fast.y, slow.y[:, :7], rtol=0, atol=1e-15)
    assert torch.allclose(fast.ybar, slow.ybar, rtol=0, atol=1e-15) and torch.allclose(fast.ystd, slow.ystd, rtol=0, atol=1e-15)


def test_sort_numerical_fast_path_equals_the_general_path_and_ignores_the_report_order():
    """Deterministic, report-order independent arrangement of the meta-data (reference utils.py:98-106 sorts the
    evaluations): the NaN-free shortcut gives the order of the general (NaN-aware) path, ties included."""
    import numpy as np

    from scamlgp_b200 import space as S

    g = np.random.default_rng(0)
    for _ in range(40):
        n, d = int(g.integers(2, 40)), int(g.integers(1, 5))
        X = torch.tensor(np.round(g.random((n, d)), 1))  # coarse grid: many ties
        Y = torch.tensor(np.round(g.random((n, 1)), 1))
        a = S.sort_numerical(X, Y)
        Xn = torch.cat([X, torch.full((1, d), float("nan"), dtype=torch.float64)])  # a NaN row forces the general path
        Yn = torch.cat([Y, torch.zeros(1, 1, dtype=torch.float64)])
        b = S.sort_numerical(Xn, Yn)
        assert torch.equal(a[0], b[0][:-1]) and torch.equal(a[1], b[1][:-1]) and bool(torch.isnan(b[0][-1]).all())
        p = torch.as_tensor(g.permutation(n))
        c = S.sort_numerical(X[p], Y[p])
        assert torch.equal(a[0], c[0]) and torch.equal(a[1], c[1])
