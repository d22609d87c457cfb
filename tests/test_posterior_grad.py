"""Analytic candidate gradients of the ScaML-GP posterior (scaml_posterior_grad, csrc/scaml_grad.cuh) vs autograd
through the oracle's restatement of `ScaMLGP.forward` (eval branch, reference scamlgp/model.py:364-375) -- the
quantity botorch's optimize_acqf differentiates.  Tolerance: relative 1e-7 on gradients (north star), 1e-9 on values.

The same cases run on the CPU logic emulation of the kernel sources (not gpu) and on the sm_100a build (gpu)."""
import numpy as np
import pytest
import torch

from oracle import scaml_oracle as O
from scamlgp_b200._capi import HyperSpec
from tests.helpers import TOL_GRAD, TOL_MEAN_VAR, make_problem, rel_err

DT = torch.float64


def _case(eng, M, n, d, B, nt, nvs, kernel, kernel_t, w, seed=3, coincide=False):
    from scamlgp_b200.engine import SourceBatch

    dev = eng.device
    pb = make_problem(M, 2, n, d, seed=seed, n_valid=nvs, kernel=kernel)
    batch = SourceBatch.from_padded(pb["X"].to(dev), pb["Y"].to(dev), torch.tensor(pb["nv"]).to(dev))
    th = pb["th"][:, 1].contiguous()
    fs = eng.factorize(batch, th.to(dev), pb["cspec"])
    states = [O.factorize(pb["X"][m, : int(pb["nv"][m])], pb["Y"][m, : int(pb["nv"][m])], th[m], pb["ospec"])
              for m in range(M)]
    g = torch.Generator().manual_seed(seed + 100)
    Xc = torch.rand(B, d, dtype=DT, generator=g)
    if coincide:  # candidates on source training inputs (r^2 = 0 against one row of K_m), and a repeated candidate
        Xc[0] = pb["X"][0, 0]
        Xc[1] = pb["X"][M - 1, int(pb["nv"][M - 1]) - 1]
        Xc[B - 1] = Xc[0]
    w = torch.as_tensor(w, dtype=DT)
    otspec, ctspec = O.HyperSpec.target(kernel_t), HyperSpec.target(kernel_t)
    tht = O.initial_theta_raw(d, otspec) + 0.3 * torch.randn(d + 2, dtype=DT, generator=g)
    Xcd, wd = Xc.to(dev), w.to(dev)
    U = eng.cond_prepare(fs, Xcd, wd)  # pruned tasks (w == 0) are skipped: their slices stay zero
    for m in range(M):
        if float(w[m]) == 0.0:
            assert float(U[m].abs().max()) == 0.0
    # ---- values from U (no second pass over the factors) == the prediction kernel ---------------------------------- #
    # The two kernels round the sum over tasks and points of w_m ystd_m k*_mi alpha_mi differently.  They agree to 1e-11
    # of the mean, or to a few ulps of the sum of the magnitudes of its terms where that is larger: for a nearly
    # singular K_m (d = 1: 150 points on [0, 1], cond(K) ~ 1e7) the terms are ~1e5 times the mean they cancel to.
    terms = sum(float(w[m]) * st.ystd * (O.kernel_matrix(Xc, st.X, st.ls, st.os, st.kernel).abs() @ st.alpha.abs())
                for m, st in enumerate(states))
    mean_floor = 5e-16 * float(terms.max())

    def mean_agrees(a, ref):
        return float((a - ref).abs().max()) < max(1e-11 * float(ref.abs().max()), mean_floor)

    pm0, pv0 = eng.predict_weighted(fs, wd, Xcd)
    om0, ov0 = O.scaml_prior_predict(states, w, Xc)
    assert rel_err(pm0.cpu().numpy(), om0.numpy()) < TOL_MEAN_VAR
    prior_scale = sum(float(w[m]) ** 2 * float(st.os) * st.ystd ** 2 for m, st in enumerate(states))
    assert float((pv0.cpu() - ov0).abs().max()) < TOL_MEAN_VAR * prior_scale  # variances: relative to the prior scale
    vm, vv, _ = eng.values_from_u(fs, wd, Xcd, U)
    assert mean_agrees(vm, pm0)
    assert float((vv - pv0).abs().max()) < 1e-10 * float(pv0.abs().max())
    # ---- prior only (n_t = 0): gradient of sum_m w_m mu_m and sum_m w_m^2 var_m ------------------------------------ #
    dm, dv = eng.posterior_grad(fs, wd, Xcd, U)
    _, _, rdm, rdv = O.scaml_posterior_grad(states, w, None, tht, otspec, Xc, None)
    e0 = (rel_err(dm.cpu().numpy(), rdm.numpy()), rel_err(dv.cpu().numpy(), rdv.numpy()))
    assert max(e0) < TOL_GRAD, e0
    if nt == 0:
        return e0
    # ---- conditioned on n_t target points ------------------------------------------------------------------------- #
    Xt = torch.rand(nt, d, dtype=DT, generator=g)
    if coincide:  # a candidate on a target input
        Xt[nt - 1] = Xc[2]
    Yt = torch.sin(3.0 * Xt).sum(1, keepdim=True) + 0.05 * torch.randn(nt, 1, dtype=DT, generator=g)
    cache = O.build_target_cache(states, Xt, Yt)
    Xtd = Xt.to(dev)
    A = eng.cond_prepare(fs, Xtd)
    sm, sc = eng.cond_caches(fs, Xtd, A)
    ts = eng.target_factorize(sm, sc, Xtd, cache.yt_std.to(dev).contiguous(), wd, tht.to(dev).contiguous(),
                              cache.mu_all, cache.s_all, ctspec)
    assert ts.info == 0
    pm, pv, cross = eng.predict_conditioned(fs, wd, Xcd, Xtd, A)
    vm, vv, vc = eng.values_from_u(fs, wd, Xcd, U, Xtd, A)
    assert mean_agrees(vm, pm)
    assert float((vv - pv).abs().max()) < 1e-10 * float(pv.abs().max())
    assert float((vc - cross).abs().max()) < 1e-10 * float(cross.abs().max())
    mean0, var0 = eng.target_posterior(ts, pm, pv, cross, Xcd)
    mean, var, beta = eng.target_posterior_beta(ts, pm, pv, cross, Xcd)
    assert torch.equal(mean, mean0) and torch.equal(var, var0)  # the beta output does not disturb the values
    dm, dv = eng.posterior_grad(fs, wd, Xcd, U, ts, A, beta)
    rm, rv, rdm, rdv = O.scaml_posterior_grad(states, w, cache, tht, otspec, Xc, None)
    assert rel_err(mean.cpu().numpy(), rm.numpy()) < 1e-8
    assert float((var.cpu() - rv).abs().max()) < 1e-8 * float(rv.abs().max())
    e1 = (rel_err(dm.cpu().numpy(), rdm.numpy()), rel_err(dv.cpu().numpy(), rdv.numpy()))
    assert max(e1) < TOL_GRAD, e1
    assert float(beta[:, nt:].abs().max() if beta.shape[1] > nt else 0.0) == 0.0
    # finite differences of the kernels' own values (independent of the oracle): central, h = 1e-5
    h = 1e-5
    k = d - 1
    Xp, Xm_ = Xcd.clone(), Xcd.clone()
    Xp[:, k] += h
    Xm_[:, k] -= h
    vals = []
    for Xq in (Xp, Xm_):
        a, b_, c = eng.predict_conditioned(fs, wd, Xq.contiguous(), Xtd, A)
        vals.append(eng.target_posterior(ts, a, b_, c, Xq.contiguous()))
    fd_m = (vals[0][0] - vals[1][0]) / (2 * h)
    fd_v = (vals[0][1] - vals[1][1]) / (2 * h)
    rows = torch.ones(B, dtype=torch.bool, device=dev)
    if coincide and 1 in (kernel, kernel_t):  # Matern-1/2 has a kink at r = 0: no central difference there
        rows[[0, 1, 2, B - 1]] = False
    assert float((fd_m - dm[:, k])[rows].abs().max()) < 1e-5 * max(1.0, float(dm.abs().max()))
    assert float((fd_v - dv[:, k])[rows].abs().max()) < 1e-5 * max(1.0, float(dv.abs().max()))
    return e0 + e1


@pytest.fixture(scope="module")
def emu_engine(emu_lib):
    from tests.emu_engine import EmuEngine

    return EmuEngine(emu_lib)


@pytest.mark.parametrize("M,n,d,B,nt,nvs,kernel,kernel_t,w", [
    (3, 70, 3, 37, 11, [70, 33, 9], 0, 0, [0.5, 0.3, 0.2]),   # ragged, 2 candidate tiles with dead lanes, n_t % 8 != 0
    (3, 64, 2, 5, 4, None, 3, 2, [0.7, 0.0, 0.3]),            # Matern source / target kernels, a pruned task
    (2, 40, 9, 8, 3, None, 0, 0, [0.6, 0.4]),                 # d > 8 (16-wide register variant)
    (2, 33, 2, 3, 0, [33, 1], 1, 0, [1.0, 0.5]),              # prior only, single-point task, Matern-1/2
    (2, 30, 17, 6, 5, None, 0, 0, [0.6, 0.4]),                # d > 16 (32-wide register variant)
    (2, 24, 32, 4, 3, None, 3, 1, [0.6, 0.4]),                # d = 32, the library limit
    (2, 30, 1, 5, 4, [30, 7], 2, 0, [0.6, 0.4]),              # d = 1
])
def test_emu_posterior_grad_matches_oracle_autograd(emu_engine, M, n, d, B, nt, nvs, kernel, kernel_t, w):
    _case(emu_engine, M, n, d, B, nt, nvs, kernel, kernel_t, w)


@pytest.mark.parametrize("kernel", [0, 1, 2, 3])
def test_emu_posterior_grad_at_coincident_points(emu_engine, kernel):
    """Candidates equal to a source training input, to a target input and to each other (r^2 = 0)."""
    _case(emu_engine, 2, 30, 3, 6, 5, [30, 12], kernel, kernel, [0.6, 0.4], coincide=True)


@pytest.mark.gpu
@pytest.mark.parametrize("M,n,d,B,nt,nvs,kernel,kernel_t,w", [
    (6, 256, 6, 128, 80, None, 0, 0, None),
    (5, 200, 6, 70, 33, [200, 150, 64, 7, 1], 0, 0, [0.3, 0.0, 0.3, 0.2, 0.2]),
    (4, 128, 10, 40, 12, None, 3, 3, None),
    (3, 512, 4, 33, 20, [512, 300, 65], 2, 1, None),
    (3, 96, 16, 9, 5, None, 0, 0, None),
    (4, 64, 3, 16, 0, None, 0, 0, None),
    (3, 96, 17, 20, 12, [96, 50, 9], 0, 0, None),   # d = 17 and 32: the DMAX = 32 instantiations, all source kernels
    (3, 96, 17, 20, 12, None, 1, 0, None),
    (3, 96, 17, 20, 12, None, 2, 2, None),
    (3, 96, 17, 20, 12, None, 3, 3, None),
    (3, 128, 32, 33, 70, [128, 64, 1], 0, 1, None),
    (3, 128, 32, 33, 70, None, 1, 0, None),
    (3, 128, 32, 33, 70, None, 2, 0, None),
    (3, 128, 32, 33, 70, None, 3, 2, None),
    (4, 200, 6, 64, 20, [200, 150, 64, 7], 1, 1, None),  # Matern-1/2 source
    (3, 150, 1, 50, 30, [150, 40, 2], 0, 0, None),        # d = 1
])
def test_gpu_posterior_grad_matches_oracle_autograd(engine, M, n, d, B, nt, nvs, kernel, kernel_t, w):
    if w is None:
        w = list(np.linspace(1.0, 2.0, M) / M)
    _case(engine, M, n, d, B, nt, nvs, kernel, kernel_t, w)


@pytest.mark.gpu
@pytest.mark.parametrize("kernel", [0, 1, 2, 3])
def test_gpu_posterior_grad_at_coincident_points(engine, kernel):
    """Candidates equal to a source training input, to a target input and to each other (r^2 = 0)."""
    _case(engine, 3, 128, 6, 40, 12, [128, 60, 9], kernel, kernel, [0.5, 0.3, 0.2], coincide=True)


@pytest.mark.gpu
def test_gpu_posterior_grad_is_deterministic_and_split_invariant(engine):
    """Fixed-order reductions: repeated launches are bit-identical; many tasks (several task splits per tile)."""
    from scamlgp_b200.engine import SourceBatch

    M, n, d, B = 700, 64, 6, 48
    X, Y = O.synthetic_tasks(M, n, d, seed=1)
    th = O.sample_theta_raw(M, 2, d, O.HyperSpec.source(), seed=1)[:, 1].contiguous()
    batch = SourceBatch.from_padded(X.cuda(), Y.cuda())
    fs = engine.factorize(batch, th.cuda(), HyperSpec.source())
    Xc = torch.rand(B, d, dtype=DT, generator=torch.Generator().manual_seed(2)).cuda()
    w = torch.full((M,), 1.0 / M, dtype=DT).cuda()
    U = engine.cond_prepare(fs, Xc)
    a = engine.posterior_grad(fs, w, Xc, U)
    b = engine.posterior_grad(fs, w, Xc, U)
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])
    # linearity in the tasks: the gradient over all tasks == sum of the gradients over two halves
    w1, w2 = w.clone(), w.clone()
    w1[M // 2:] = 0.0
    w2[: M // 2] = 0.0
    g1 = engine.posterior_grad(fs, w1, Xc, U)
    g2 = engine.posterior_grad(fs, w2, Xc, U)
    for i in range(2):
        assert float((g1[i] + g2[i] - a[i]).abs().max()) < 1e-12 * float(a[i].abs().max())


def test_emu_cross_covariance_direct_term_split_over_tasks(emu_engine, monkeypatch):
    """Small candidate batches sum the direct term sum_m c_m K_m(x, x_tj) over task splits (partials + fixed-order
    finish kernel); forced here with the test knob, must equal the unsplit result to rounding."""
    from scamlgp_b200.engine import SourceBatch

    eng = emu_engine
    M, n, d, B, nt = 5, 40, 3, 7, 5
    pb = make_problem(M, 2, n, d, seed=5, n_valid=[40, 33, 20, 9, 1])
    batch = SourceBatch.from_padded(pb["X"], pb["Y"], torch.tensor(pb["nv"]))
    fs = eng.factorize(batch, pb["th"][:, 1].contiguous(), pb["cspec"])
    g = torch.Generator().manual_seed(8)
    Xc, Xt = torch.rand(B, d, dtype=DT, generator=g), torch.rand(nt, d, dtype=DT, generator=g)
    w = torch.tensor([0.3, 0.0, 0.3, 0.2, 0.2], dtype=DT)
    A = eng.cond_prepare(fs, Xt)
    ref = eng.predict_conditioned(fs, w, Xc, Xt, A)
    monkeypatch.setenv("SCAML_COMB_TSPLIT", "3")
    assert eng.lib.cond_combine_task_splits(M, B, nt) == 3
    got = eng.predict_conditioned(fs, w, Xc, Xt, A)
    U = eng.cond_prepare(fs, Xc, w)
    got_u = eng.values_from_u(fs, w, Xc, U, Xt, A)
    for r, a, b_ in zip(ref, got, got_u):
        assert float((a - r).abs().max()) <= 1e-13 * float(r.abs().max())
        assert float((b_ - r).abs().max()) <= 1e-10 * float(r.abs().max())


def test_emu_value_half_switches_kernel_with_the_number_of_target_points(emu_engine):
    """`Engine.prior_values`: values from U for n_t <= 64, the fused prediction kernel above (the 17-column-block
    variant of the values kernel is register-bound on the GPU); both must give the same numbers."""
    from scamlgp_b200.engine import SourceBatch

    eng = emu_engine
    M, n, d, B = 2, 40, 2, 5
    pb = make_problem(M, 2, n, d, seed=6)
    batch = SourceBatch.from_padded(pb["X"], pb["Y"], torch.tensor(pb["nv"]))
    fs = eng.factorize(batch, pb["th"][:, 1].contiguous(), pb["cspec"])
    g = torch.Generator().manual_seed(2)
    Xc = torch.rand(B, d, dtype=DT, generator=g)
    w = torch.tensor([0.6, 0.4], dtype=DT)
    U = eng.cond_prepare(fs, Xc, w)
    for nt in (64, 70):
        Xt = torch.rand(nt, d, dtype=DT, generator=g)
        A = eng.cond_prepare(fs, Xt)
        launches0 = eng.launches
        a = eng.prior_values(fs, w, Xc, U, Xt, A)
        used = eng.launches - launches0
        b_ = eng.values_from_u(fs, w, Xc, U, Xt, A)
        c = eng.predict_conditioned(fs, w, Xc, Xt, A)
        for x, y, z in zip(a, b_, c):
            assert float((x - y).abs().max()) <= 1e-10 * float(y.abs().max())
            assert float((x - z).abs().max()) <= 1e-10 * float(z.abs().max())
        assert used >= 2
