"""Batch Bayesian optimisation: joint q-point posterior blocks (`ScaMLGP.posterior_blocks`, csrc/scaml_qblock.cuh),
their vector-Jacobian product, the MC batch acquisitions qUCB / qEI and `ScaMLGPBO.generate_evaluation_specifications`.

Checkers: the oracle's joint posterior (`O.scaml_posterior(..., full_cov=True)`) and autograd through it, the existing
joint path `ScaMLGP.posterior(X[b, q, d])`, the q = 1 gradient path and finite differences of the kernels' own values.
Kernel cases run on the CPU logic emulation of the kernel sources (not gpu) and on the sm_100a build (gpu)."""
import math

import numpy as np
import pytest
import torch

from oracle import scaml_oracle as O
from tests.helpers import TOL_GRAD, TOL_MEAN_VAR, rel_err

DT = torch.float64


@pytest.fixture(scope="module")
def emu_engine(emu_lib):
    from tests.emu_engine import EmuEngine

    return EmuEngine(emu_lib)


def _meta_data(M, n, d, seed, ragged):
    from scamlgp_b200.modules import SupervisedDataset

    X, Y = O.synthetic_tasks(M, n, d, seed=seed)
    out = {}
    for i in range(M):
        ni = n if not ragged else max(1, n - (n // M + 3) * i)
        out[f"task{i}"] = SupervisedDataset(X[i, :ni], Y[i, :ni].reshape(-1, 1))
    return out


_NU = {1: 0.5, 2: 1.5, 3: 2.5}


def _kernel(kernel, d, source):
    from scamlgp_b200.model import _get_default_kernel, _get_kernel_source_gp
    from scamlgp_b200.modules import MaternKernel, RBFKernel

    base = RBFKernel if kernel == 0 else (lambda **kw: MaternKernel(nu=_NU[kernel], **kw))
    return (_get_kernel_source_gp if source else _get_default_kernel)(base_kernel=base, ard_num_dims=d)


def _fitted_model(eng, M, n, d, nt, ragged, kernel, kernel_t, prune, seed=3):
    """A ScaMLGP on M fitted source tasks, nt target points, perturbed target hyper-parameters and weights (task 1
    pruned when `prune`), plus the oracle's restatement of the same state."""
    from scamlgp_b200.model import ScaMLGP, meta_fit_scamlgp
    from scamlgp_b200.modules import set_theta_raw, theta_raw_of

    md = _meta_data(M, n, d, seed, ragged)
    gps = meta_fit_scamlgp(md, covar_module=_kernel(kernel, d, True), num_restarts_log_likelihood=0, seed=0,
                           engine=eng, fit_options=dict(maxiter=3))
    g = torch.Generator().manual_seed(seed + 100)
    Xt = torch.rand(nt, d, dtype=DT, generator=g)
    Yt = torch.sin(3.0 * Xt).sum(1, keepdim=True) + 0.05 * torch.randn(nt, 1, dtype=DT, generator=g)
    model = ScaMLGP(Xt, Yt, gps, covar_module=_kernel(kernel_t, d, False), engine=eng)
    otspec = O.HyperSpec.target(kernel_t)
    tht = O.initial_theta_raw(d, otspec) + 0.3 * torch.randn(d + 2, dtype=DT, generator=g)
    set_theta_raw(model.likelihood, model.covar_module, tht)
    w = torch.linspace(1.0, 2.0, M, dtype=DT) / M
    if prune:
        w[1] = 1e-9
    model.weights = w
    model.eval()
    ospec = O.HyperSpec.source(kernel)
    states = []
    for gp in gps.values():
        X = gp.train_inputs[0]
        states.append(O.factorize(X, gp._raw_Y.reshape(-1), theta_raw_of(gp.likelihood, gp.covar_module, d), ospec))
    cache = O.build_target_cache(states, Xt, Yt) if nt > 0 else None
    return model, (states, model.weights, cache, model.theta_raw(), otspec), g


def _oracle_blocks(args, X):
    """Oracle mean [b, q] / cov [b, q, q] block by block (autograd-ready when X requires grad)."""
    ms, cs = [], []
    for i in range(X.shape[0]):
        m, c = O.scaml_posterior(*args, X[i], full_cov=True)
        ms.append(m)
        cs.append(c)
    return torch.stack(ms), torch.stack(cs)


def _blocks_case(eng, M, n, d, nb, q, nt, ragged, kernel, kernel_t, prune, coincide=False):
    model, args, g = _fitted_model(eng, M, n, d, nt, ragged, kernel, kernel_t, prune)
    X = torch.rand(nb, q, d, dtype=DT, generator=g)
    if coincide:  # a repeated point inside a block, a point on a source training input and one on a target input
        X[0, q - 1] = X[0, 0]
        X[nb - 1, 0] = O.synthetic_tasks(M, n, d, seed=3)[0][0, 0]
        if nt > 0:
            X[nb - 1, q - 1] = model.train_inputs[0][0]
    mean, cov, vjp = model.posterior_blocks(X)
    assert mean.shape == (nb, q) and cov.shape == (nb, q, q)
    assert torch.equal(cov, cov.transpose(1, 2))
    # ---- 1. values: oracle joint posterior, and the existing joint path -------------------------------------- #
    om, oc = _oracle_blocks(args, X)
    for i in range(nb):
        scale = float(oc[i].abs().max())
        assert float((mean[i] - om[i]).abs().max()) < TOL_MEAN_VAR * max(1.0, float(om[i].abs().max()))
        assert float((cov[i] - oc[i]).abs().max()) < TOL_MEAN_VAR * scale
    if q > 1:
        pj = model.posterior(X)
        jm, jc = pj.mean.reshape(nb, q), pj.mvn.covariance_matrix
        assert float((mean - jm).abs().max()) <= 1e-11 * max(1.0, float(jm.abs().max()))
        assert float((cov - jc).abs().max()) <= 1e-11 * float(jc.abs().max())
    # ---- 2. VJP against autograd through the oracle ----------------------------------------------------------- #
    gm = torch.randn(nb, q, dtype=DT, generator=g)
    gc = torch.randn(nb, q, q, dtype=DT, generator=g)
    dX = vjp(gm, gc)
    with pytest.raises(RuntimeError):
        vjp(gm, gc)
    Xg = X.clone().requires_grad_(True)
    rm, rc = _oracle_blocks(args, Xg)
    (rdX,) = torch.autograd.grad((gm * rm).sum() + (gc * rc).sum(), Xg)
    err = rel_err(dX.numpy(), rdX.numpy())
    assert err < TOL_GRAD, err
    # central finite difference of the kernels' own values (independent of the oracle), last coordinate
    h, k = 1e-5, d - 1
    vals = []
    for s in (1.0, -1.0):
        Xs = X.clone()
        Xs[:, :, k] += s * h
        m_, c_, _ = model.posterior_blocks(Xs)
        vals.append(float((gm * m_).sum() + (gc * c_).sum()))
    fd = (vals[0] - vals[1]) / (2 * h)
    assert abs(fd - float(dX[:, :, k].sum())) < 1e-5 * max(1.0, float(dX[:, :, k].abs().sum()))
    # ---- q = 1: equal to g_mean dmean + g_cov dvar of the existing gradient path ------------------------------ #
    if q == 1:
        _, _, dm, dv = model.posterior_with_grad(X)
        ref = gm.reshape(-1, 1) * dm + gc.reshape(-1, 1) * dv
        assert float((dX.reshape(-1, d) - ref).abs().max()) <= 1e-12 * float(ref.abs().max())
    return model, X


# (M, n, d, nb, q, nt, ragged, kernel, kernel_t, prune)
EMU_CASES = [
    (3, 40, 3, 3, 3, 11, True, 0, 0, False),    # ragged tasks, n_t % 8 != 0, q = 3
    (3, 33, 2, 4, 4, 5, False, 3, 2, True),     # Matern-5/2 source, Matern-3/2 target, a pruned task
    (2, 24, 9, 2, 3, 3, False, 0, 0, False),    # d > 8 (16-wide register variant)
    (2, 24, 2, 3, 16, 0, False, 1, 0, False),   # prior only (n_t = 0), Matern-1/2, q = 16
    (2, 24, 3, 43, 3, 4, False, 0, 1, False),   # 129 points: a 126-point launch and a partial one of 3
    (2, 24, 3, 7, 1, 4, False, 0, 0, False),    # q = 1 against the existing gradient path
    (2, 20, 2, 8, 16, 0, False, 0, 0, False),   # B q = 128: one full launch
    (2, 260, 2, 2, 3, 3, False, 0, 0, False),   # n_pad = 320 > 256: the staged inputs of the cov kernel
    (2, 24, 1, 3, 2, 3, False, 2, 0, False),    # d = 1
]


@pytest.mark.parametrize("M,n,d,nb,q,nt,ragged,kernel,kernel_t,prune", EMU_CASES)
def test_emu_posterior_blocks_match_oracle(emu_engine, M, n, d, nb, q, nt, ragged, kernel, kernel_t, prune):
    _blocks_case(emu_engine, M, n, d, nb, q, nt, ragged, kernel, kernel_t, prune)


@pytest.mark.gpu
@pytest.mark.parametrize("M,n,d,nb,q,nt,ragged,kernel,kernel_t,prune", EMU_CASES + [
    (5, 200, 6, 32, 4, 33, True, 0, 0, True),
    (4, 128, 10, 8, 16, 12, False, 3, 3, False),
    (3, 256, 4, 11, 3, 128, False, 2, 1, False),  # n_t = 128
    (4, 64, 6, 45, 3, 0, False, 0, 0, False),     # prior only, partial last launch
    (4, 96, 6, 40, 1, 20, False, 0, 0, False),
    (3, 320, 6, 8, 4, 12, True, 0, 0, False),   # n > 256
    (3, 512, 4, 6, 3, 20, False, 2, 1, False),  # n = 512, the model's limit
    (3, 150, 1, 10, 4, 9, False, 0, 0, False),  # d = 1
])
def test_gpu_posterior_blocks_match_oracle(engine, M, n, d, nb, q, nt, ragged, kernel, kernel_t, prune):
    _blocks_case(engine, M, n, d, nb, q, nt, ragged, kernel, kernel_t, prune)


def _blocks_beyond_model(eng, monkeypatch, d, kernel, nt):
    """d = 17, 32: the engine's q-block kernels (DMAX = 32) run beyond the model's d <= 16; the model's own block
    code is reused with its shape gate lifted, so the values and the VJP are checked against the oracle the same way."""
    from scamlgp_b200.model import ScaMLGP

    monkeypatch.setattr(ScaMLGP, "supports_candidate_gradients", property(lambda self: True))
    _blocks_case(eng, 2, 24, d, 3, 3, nt, False, kernel, kernel, False)


@pytest.mark.parametrize("d,kernel,nt", [(17, 0, 4), (32, 3, 0)])
def test_emu_qblock_beyond_model_dimension(emu_engine, monkeypatch, d, kernel, nt):
    _blocks_beyond_model(emu_engine, monkeypatch, d, kernel, nt)


@pytest.mark.gpu
@pytest.mark.parametrize("d,kernel,nt", [(17, 0, 10), (17, 1, 0), (32, 2, 10), (32, 3, 20)])
def test_gpu_qblock_beyond_model_dimension(engine, monkeypatch, d, kernel, nt):
    _blocks_beyond_model(engine, monkeypatch, d, kernel, nt)


@pytest.mark.parametrize("kernel", [0, 1, 2, 3])
def test_emu_posterior_blocks_at_coincident_points(emu_engine, kernel):
    _blocks_case(emu_engine, 2, 24, 3, 3, 3, 4, False, kernel, kernel, False, coincide=True)


@pytest.mark.gpu
@pytest.mark.parametrize("kernel", [0, 1, 2, 3])
def test_gpu_posterior_blocks_at_coincident_points(engine, kernel):
    _blocks_case(engine, 3, 128, 6, 8, 4, 12, False, kernel, kernel, False, coincide=True)


@pytest.mark.gpu
def test_gpu_posterior_blocks_deterministic_and_position_invariant(engine):
    """Fixed-order sums: repeated calls are bit-identical; a block moved to another position of the launch gives the
    same numbers up to rounding of the shared per-launch work."""
    model, _, g = _fitted_model(engine, 300, 64, 6, 20, False, 0, 0, False)
    X = torch.rand(32, 4, 6, dtype=DT, generator=g)
    gm, gc = torch.randn(32, 4, dtype=DT, generator=g), torch.randn(32, 4, 4, dtype=DT, generator=g)
    outs = []
    for _ in range(2):
        m, c, vjp = model.posterior_blocks(X)
        outs.append((m, c, vjp(gm, gc)))
    for a, b in zip(*outs):
        assert torch.equal(a, b)
    perm = torch.randperm(32, generator=g)
    m2, c2, vjp2 = model.posterior_blocks(X[perm])
    d2 = vjp2(gm[perm], gc[perm])
    m, c, dX = outs[0]
    assert float((m2 - m[perm]).abs().max()) <= 1e-13 * float(m.abs().max())
    assert float((c2 - c[perm]).abs().max()) <= 1e-13 * float(c.abs().max())
    assert float((d2 - dX[perm]).abs().max()) <= 1e-13 * float(dX.abs().max())


def test_emu_qblock_argument_checks(emu_engine):
    lib = emu_engine.lib.lib
    # B not a multiple of q, q > 16, null pointers
    assert lib.scaml_qblock_cov(None, None, None, None, None, None, None, None, None, 0, 1, 8, 2, 6, 4, 0, None) == -1
    assert lib.scaml_qblock_vjp(*([None] * 13), 1.0, None, None, None, None, 0, 1, 8, 2, 8, 4, 0, 0, 0, None) == -1
    model = _fitted_model(emu_engine, 2, 16, 2, 3, False, 0, 0, False)[0]
    with pytest.raises(NotImplementedError, match="q <= 16"):
        model.posterior_blocks(torch.rand(1, 17, 2, dtype=DT))


# ---- acquisitions ---------------------------------------------------------------------------------------------- #
def _oracle_acq(kind, args, X, z, beta=9.0, best_f=0.0):
    """Pure-torch restatement: botorch MC semantics on the oracle's joint posterior with the same base samples."""
    m, c = _oracle_blocks(args, X)
    L = torch.linalg.cholesky(c)
    xi = m.unsqueeze(1) + torch.einsum("bik,sk->bsi", L, z)
    if kind == "ucb":
        v = -m.unsqueeze(1) + math.sqrt(beta * math.pi / 2) * (xi - m.unsqueeze(1)).abs()
    else:
        v = (best_f - xi).clamp_min(0.0)
    return v.max(-1).values.mean(-1)


def _acq_case(eng, nt):
    from scamlgp_b200.utils import UpperConfidenceBound, qExpectedImprovement, qUpperConfidenceBound

    model, args, g = _fitted_model(eng, 3, 32, 3, nt, False, 0, 0, False)
    X = torch.rand(5, 3, 3, dtype=DT, generator=g)
    best_f = float(model._train_Y.min()) if nt > 0 else 0.5
    for kind, af in (("ucb", qUpperConfidenceBound(model, beta=4.0, num_samples=64, seed=3)),
                     ("ei", qExpectedImprovement(model, best_f=None if nt > 0 else best_f, num_samples=64, seed=3))):
        v, dX = af.value_and_grad(X)
        v2, dX2 = af.value_and_grad(X)
        assert torch.equal(v, v2) and torch.equal(dX, dX2)
        assert torch.equal(af(X), v)
        Xg = X.clone().requires_grad_(True)
        rv = _oracle_acq(kind, args, Xg, af.base_samples(3), beta=4.0, best_f=best_f)
        (rd,) = torch.autograd.grad(rv.sum(), Xg)
        assert rel_err(v.numpy(), rv.detach().numpy()) < 1e-7
        assert rel_err(dX.numpy(), rd.numpy()) < 1e-7
    # coincident points (a repeated point in a block, a point on a target input): singular blocks go through the
    # jitter ladder and the values and gradients stay finite
    Xs = X.clone()
    Xs[0, 1] = Xs[0, 0]
    if nt > 0:
        Xs[1, 2] = model.train_inputs[0][0]
    for af in (qUpperConfidenceBound(model, beta=4.0, num_samples=64, seed=3),
               qExpectedImprovement(model, best_f=None if nt > 0 else best_f, num_samples=64, seed=3)):
        v, dX = af.value_and_grad(Xs)
        assert bool(torch.isfinite(v).all()) and bool(torch.isfinite(dX).all())
    # q = 1: qUCB with 4096 samples is the analytic UCB up to the sampling error
    Xc = torch.rand(6, 1, 3, dtype=DT, generator=g)
    qv = qUpperConfidenceBound(model, beta=9.0, num_samples=4096)(Xc)
    av = UpperConfidenceBound(model, beta=9.0)(Xc)
    sig = model.posterior(Xc).variance.reshape(-1).sqrt()
    assert bool(((qv - av).abs() < 1e-2 * 3.0 * sig).all())


@pytest.mark.parametrize("nt", [0, 6])
def test_emu_batch_acquisitions_match_oracle(emu_engine, nt):
    _acq_case(emu_engine, nt)


@pytest.mark.gpu
@pytest.mark.parametrize("nt", [0, 6])
def test_gpu_batch_acquisitions_match_oracle(engine, nt):
    _acq_case(engine, nt)


# ---- optimizer contract -------------------------------------------------------------------------------------- #
def _E(configuration, loss):
    from scamlgp_b200.space import Evaluation

    return Evaluation(configuration=configuration, objectives={"loss": loss})


def _branin(x1, x2, a, b, c, r, s, t):
    return a * (x2 - b * x1 ** 2 + c * x1 - r) ** 2 + s * (1 - t) * np.cos(x1) + s


def _branin_problem(seed=0, M=8, n=32):
    from scamlgp_b200.space import ContinuousParameter, ParameterSpace

    rng = np.random.default_rng(seed)

    def task():
        return dict(a=rng.uniform(0.5, 1.5), b=rng.uniform(0.1, 0.15), c=rng.uniform(1.0, 2.0), r=rng.uniform(5.0, 7.0),
                    s=rng.uniform(8.0, 12.0), t=rng.uniform(0.03, 0.05))

    space = ParameterSpace()
    space.add(ContinuousParameter("x1", (-5.0, 10.0)))
    space.add(ContinuousParameter("x2", (0.0, 15.0)))
    md = {}
    for k in range(M):
        p = task()
        x1, x2 = rng.uniform(-5, 10, n), rng.uniform(0, 15, n)
        y = _branin(x1, x2, **p) + rng.normal(0, 1.0, n)
        md[k] = [_E({"x1": float(a), "x2": float(b)}, float(v)) for a, b, v in zip(x1, x2, y)]
    return space, md, task()


TINY = dict(af_optimizer_kwargs=dict(raw_samples=8, num_restarts=2, maxiter=3), fit_options=dict(maxiter=3),
            num_restarts_log_likelihood=0)


def _optimizer_scenario(eng, extra):
    from scamlgp_b200.optimizer import ScaMLGPBO
    from scamlgp_b200.space import (CategoricalParameter, ContinuousParameter, Objective, OptimizerNotReady,
                                    ParameterSpace)

    loss = Objective("loss", greater_is_better=False)
    space, md, target = _branin_problem(M=3, n=10)
    f = lambda c: float(_branin(c["x1"], c["x2"], **target))  # noqa: E731

    def make():
        return ScaMLGPBO(space, loss, md, seed=7, num_initial_random_samples=2, max_pending_evaluations=6,
                         engine=eng, **extra)

    opt = make()
    first = opt.generate_evaluation_specifications(3)  # fewer than num_initial_random_samples: random
    assert len(first) == 3 and len(opt.pending_specifications) == 3
    opt.report([s.create_evaluation(objectives={"loss": f(s.configuration)}) for s in first])
    assert opt.model.num_train == 3
    theta_before = opt.model.theta_raw().clone()
    p1 = opt.generate_evaluation_specifications(2)  # acquisition on the fitted model
    p2 = opt.generate_evaluation_specifications(3)  # conditioned on the 2 pending points
    assert len(opt.pending_specifications) == 5
    confs = [tuple(s.configuration[k] for k in ("x1", "x2")) for s in p1 + p2]
    assert len(set(confs)) == 5
    for x1, x2 in confs:
        assert -5.0 <= x1 <= 10.0 and 0.0 <= x2 <= 15.0
    with pytest.raises(OptimizerNotReady):
        opt.generate_evaluation_specifications(2)
    opt.report([s.create_evaluation(objectives={"loss": f(s.configuration)}) for s in p1 + p2])
    assert opt.model.num_train == 8 and len(opt.pending_specifications) == 0
    assert not torch.equal(opt.model.theta_raw(), theta_before)  # the report refitted the target model
    # the same seed gives the same batches
    opt2 = make()
    first2 = opt2.generate_evaluation_specifications(3)
    assert [s.configuration for s in first2] == [s.configuration for s in first]
    opt2.report([s.create_evaluation(objectives={"loss": f(s.configuration)}) for s in first2])
    assert [s.configuration for s in opt2.generate_evaluation_specifications(2)] == [s.configuration for s in p1]
    # discrete / mixed spaces are out of scope
    mixed = ParameterSpace()
    mixed.add(ContinuousParameter("x", (0.0, 1.0)))
    mixed.add(CategoricalParameter("c", ["a", "b"]))
    mopt = ScaMLGPBO(mixed, loss, {"t": [_E({"x": 0.2, "c": "a"}, 1.0), _E({"x": 0.7, "c": "b"}, 0.5)]},
                     seed=0, max_pending_evaluations=4, engine=eng, **extra)
    with pytest.raises(NotImplementedError):
        mopt.generate_evaluation_specifications(2)


def test_emu_optimizer_batch_contract(emu_engine):
    _optimizer_scenario(emu_engine, TINY)


@pytest.mark.gpu
def test_gpu_optimizer_batch_contract(engine):
    _optimizer_scenario(engine, {})


@pytest.mark.gpu
def test_gpu_branin_batches_beat_random_search(engine):
    """Branin, 8 meta-tasks x 32 points, 40 evaluations as 10 batches of q = 4 over 16 seeds: the mean simple regret is
    clearly below random search on the same seeds (and recorded next to sequential q = 1)."""
    from scamlgp_b200.optimizer import ScaMLGPBO
    from scamlgp_b200.space import Objective

    loss = Objective("loss", greater_is_better=False)
    g1, g2 = np.meshgrid(np.linspace(-5, 10, 400), np.linspace(0, 15, 400))
    regrets = {"q4": [], "q1": [], "random": []}
    for seed in range(16):
        space, md, target = _branin_problem(seed=seed)
        f = lambda c: float(_branin(c["x1"], c["x2"], **target))  # noqa: E731
        fmin = float(_branin(g1, g2, **target).min())
        opt = ScaMLGPBO(space, loss, md, seed=seed, max_pending_evaluations=4, engine=engine)
        ys = []
        for _ in range(10):
            specs = opt.generate_evaluation_specifications(4)
            evs = [s.create_evaluation(objectives={"loss": f(s.configuration)}) for s in specs]
            ys += [e.objectives["loss"] for e in evs]
            opt.report(evs)
        regrets["q4"].append(min(ys) - fmin)
        opt = ScaMLGPBO(space, loss, md, seed=seed, engine=engine)
        ys = []
        for _ in range(40):
            s = opt.generate_evaluation_specification()
            e = s.create_evaluation(objectives={"loss": f(s.configuration)})
            ys.append(e.objectives["loss"])
            opt.report(e)
        regrets["q1"].append(min(ys) - fmin)
        rng = np.random.default_rng(1000 + seed)
        regrets["random"].append(float(_branin(rng.uniform(-5, 10, 40), rng.uniform(0, 15, 40), **target).min()) - fmin)
    mean = {k: float(np.mean(v)) for k, v in regrets.items()}
    line = (f"branin, 8 meta-tasks x 32 points, 40 evaluations, 16 seeds: mean simple regret q=4 (10 batches) "
            f"{mean['q4']:.4f}, q=1 (40 steps) {mean['q1']:.4f}, random search {mean['random']:.4f}; "
            f"GPU {torch.cuda.get_device_name(0)}")
    print(line)
    assert mean["q4"] < 0.5 * mean["random"], mean
