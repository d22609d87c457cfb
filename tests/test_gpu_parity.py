"""Parity of the sm_100a kernels (called through the C ABI via scamlgp_b200.engine) with
the CPU oracle.  Tolerances are the ones BASELINE.json's north_star states: relative 1e-9
on LML and posterior mean/variance, 1e-7 on gradients (conditioning envelope
cond(K_y) <~ 1e8, see DESIGN.md)."""
import os

import numpy as np
import pytest
import torch

from oracle import scaml_oracle as O
from scamlgp_b200._capi import HyperSpec
from tests.helpers import TOL_GRAD, TOL_LML, TOL_MEAN_VAR, grad_rel_err, lml_rel_err, make_problem, oracle_lml_grad, rel_err

pytestmark = pytest.mark.gpu
GOLDEN = os.path.join(os.path.dirname(__file__), "golden", "scaml_golden_v1.npz")


def _batch(pb):
    from scamlgp_b200.engine import SourceBatch

    return SourceBatch.from_padded(pb["X"].cuda(), pb["Y"].cuda(), torch.tensor(pb["nv"]).cuda())


@pytest.mark.parametrize("M,R,n,d,nv,kernel", [
    (64, 2, 64, 6, None, 0),            # config 2 shape (Hartmann-6, 64 x 64 x 6)
    (8, 3, 256, 6, None, 0),            # config 3 shape, sampled
    (6, 2, 192, 6, [130, 1, 64, 2, 192, 65], 0),  # ragged incl. n = 1, 2
    (4, 2, 100, 2, None, 3),
    (4, 1, 128, 4, None, 1),
    (4, 1, 128, 4, None, 2),
    (2, 1, 512, 10, None, 0),           # config 4 shape, sampled
    (3, 2, 128, 17, [128, 90, 3], 0),   # d > 8: input dimensions beyond the register-prefetched ones
    (2, 1, 320, 32, None, 3),           # d at the library limit, 5 super-tiles
    (4, 1, 577, 6, [577, 400, 513, 10], 0),  # n_pad = 640 > 512: the default dispatch picks the 8-warp kernel;
    (4, 1, 577, 6, [577, 400, 513, 10], 1),  # ragged n_valid on both sides of 512 in one batch
    (4, 1, 577, 6, [577, 400, 513, 10], 2),
    (4, 1, 577, 6, [577, 400, 513, 10], 3),
    (2, 1, 1000, 4, [1000, 300], 0),
    (3, 2, 100, 1, [100, 50, 3], 0),     # d = 1: the extreme of the input padding
])
def test_lml_grad_matches_oracle(engine, M, R, n, d, nv, kernel):
    pb = make_problem(M, R, n, d, seed=3, n_valid=nv, kernel=kernel)
    batch = _batch(pb)
    # per-task standardisation on device == botorch Standardize restatement
    assert rel_err(batch.ybar.cpu().numpy(), pb["ybar"]) < 1e-13
    assert rel_err(batch.ystd.cpu().numpy(), pb["ystd"]) < 1e-13
    lml, grad, info = engine.lml_grad(batch, pb["th"].cuda().contiguous(), pb["cspec"])
    torch.cuda.synchronize()
    v, g = oracle_lml_grad(pb)
    assert int(info.abs().max()) == 0
    assert lml_rel_err(lml.cpu().numpy(), v) < TOL_LML
    assert grad_rel_err(grad.cpu().numpy(), g) < TOL_GRAD
    fs = engine.factorize(batch, pb["th"][:, 0].contiguous().cuda(), pb["cspec"])
    assert int(fs.info.abs().max()) == 0
    for m in range(M):
        k = int(pb["nv"][m])
        st = O.factorize(pb["X"][m, :k], pb["Y"][m, :k], pb["th"][m, 0], pb["ospec"])
        assert rel_err(fs.alpha[m, :k].cpu().numpy(), st.alpha.numpy()) < 1e-8


@pytest.mark.parametrize("impl", ["4", "8"])
@pytest.mark.parametrize("M,R,n,d,nv,kernel", [
    (6, 2, 192, 6, [130, 1, 64, 2, 192, 65], 0),
    (3, 2, 256, 6, None, 3),
    (2, 1, 512, 10, None, 0),
])
def test_both_fit_kernel_variants_match_oracle_and_each_other(engine, monkeypatch, impl, M, R, n, d, nv, kernel):
    """SCAML_FIT_IMPL forces the 4-warp (3 CTAs/SM) or the 8-warp (2 CTAs/SM) fit kernel; the default picks by
    shape.  Both must meet the oracle tolerances whatever the heuristic would choose."""
    monkeypatch.setenv("SCAML_FIT_IMPL", impl)
    pb = make_problem(M, R, n, d, seed=13, n_valid=nv, kernel=kernel)
    batch = _batch(pb)
    lml, grad, info = engine.lml_grad(batch, pb["th"].cuda().contiguous(), pb["cspec"])
    v, g = oracle_lml_grad(pb)
    assert int(info.abs().max()) == 0
    assert lml_rel_err(lml.cpu().numpy(), v) < TOL_LML
    assert grad_rel_err(grad.cpu().numpy(), g) < TOL_GRAD
    fs = engine.factorize(batch, pb["th"][:, 0].contiguous().cuda(), pb["cspec"])
    for m in range(M):
        k = int(pb["nv"][m])
        st = O.factorize(pb["X"][m, :k], pb["Y"][m, :k], pb["th"][m, 0], pb["ospec"])
        assert rel_err(fs.alpha[m, :k].cpu().numpy(), st.alpha.numpy()) < 1e-8


def test_golden_fixtures(engine):
    from scamlgp_b200.engine import SourceBatch

    z = np.load(GOLDEN)
    for key in z["names"]:
        key = str(key)
        kern = int(key.split("__k")[1])
        spec = HyperSpec.source(kern)
        X = torch.tensor(z[key + "__X"]).unsqueeze(0).cuda()
        Y = torch.tensor(z[key + "__Y"]).unsqueeze(0).cuda()
        th = torch.tensor(z[key + "__theta_raw"]).unsqueeze(0).cuda().contiguous()
        batch = SourceBatch.from_padded(X, Y)
        lml, grad, info = engine.lml_grad(batch, th, spec)
        assert int(info.abs().max()) == 0, key
        assert lml_rel_err(lml.cpu().numpy()[0], z[key + "__lml"]) < TOL_LML, key
        assert grad_rel_err(grad.cpu().numpy()[0], z[key + "__grad"]) < TOL_GRAD, key
        fs = engine.factorize(batch, th[:, 1].contiguous(), spec)
        n = X.shape[1]
        assert rel_err(fs.alpha[0, :n].cpu().numpy(), z[key + "__alpha"]) < 1e-8, key
        mean, var = engine.predict_weighted(fs, torch.ones(1, device="cuda", dtype=torch.float64),
                                            torch.tensor(z[key + "__Xs"]).cuda())
        assert np.abs(mean.cpu().numpy() - z[key + "__post_mean"]).max() < TOL_MEAN_VAR * max(1.0, np.abs(z[key + "__post_mean"]).max()), key
        # variance: relative to the prior variance scale ystd^2 * s (cancellation s - ||v||^2)
        scale = float(fs.theta[0, -2]) * float(batch.ystd[0]) ** 2
        assert np.abs(var.cpu().numpy() - z[key + "__post_var"]).max() < TOL_MEAN_VAR * scale, key


def test_non_psd_pivot_reported_and_jitter_ladder(engine):
    pb = make_problem(3, 1, 64, 2, seed=1)
    pb["X"][1, 32:] = pb["X"][1, :32]
    pb["ospec"].noise_bounds = (1e-30, 1e-2)
    pb["cspec"].noise_bounds = (1e-30, 1e-2)
    spec = pb["ospec"]
    pb["th"][1, 0] = O.pack_theta(torch.full((2,), 50.0, dtype=torch.float64), 99.0, 1e-25, spec)
    batch = _batch(pb)
    th = pb["th"].cuda().contiguous()
    lml, grad, info = engine.lml_grad_raw(batch, th, pb["cspec"])
    assert int(info[1, 0]) > 0 and bool(torch.isnan(lml[1, 0])) and bool(torch.isnan(grad[1, 0]).all())
    assert int(info[0, 0]) == 0 and int(info[2, 0]) == 0  # the batch is not aborted
    lml2, grad2, info2 = engine.lml_grad(batch, th, pb["cspec"])  # psd_safe_cholesky ladder inside the kernel
    assert int(info2.abs().max()) == 0 and bool(torch.isfinite(lml2).all())
    assert torch.equal(lml2[[0, 2]], lml[[0, 2]])  # untouched rows are bit-identical
    lml3, grad3, info3 = engine.lml_grad_host_ladder(batch, th, pb["cspec"])  # the host-driven ladder: the checker
    assert torch.equal(lml3, lml2) and torch.equal(grad3, grad2) and torch.equal(info3, info2)
    fs = engine.factorize(batch, th[:, 0].contiguous(), pb["cspec"])  # same ladder on the prediction state
    assert int(fs.info.abs().max()) == 0 and bool(torch.isfinite(fs.alpha).all())


def test_factorize_and_weighted_prediction(engine):
    M, n, d, B = 12, 256, 6, 1000
    pb = make_problem(M, 2, n, d, seed=5, n_valid=[256, 77, 5, 256, 200, 64, 65, 128, 256, 31, 33, 256])
    batch = _batch(pb)
    th = pb["th"][:, 1].contiguous()
    fs = engine.factorize(batch, th.cuda(), pb["cspec"])
    assert int(fs.info.abs().max()) == 0
    states = [O.factorize(pb["X"][m, : pb["nv"][m]], pb["Y"][m, : pb["nv"][m]], th[m], pb["ospec"]) for m in range(M)]
    for m in range(M):
        nv = pb["nv"][m]
        assert rel_err(fs.alpha[m, :nv].cpu().numpy(), states[m].alpha.numpy()) < 1e-8
    g = torch.Generator().manual_seed(5)
    Xc = torch.rand(B, d, dtype=torch.float64, generator=g)
    w = torch.rand(M, dtype=torch.float64, generator=g)
    w[3] = 0.0
    for Bsub in (1, 63, 64, 65, B):  # ragged candidate tiles
        mean, var = engine.predict_weighted(fs, w.cuda(), Xc[:Bsub].cuda())
        om, ov = O.scaml_prior_predict(states, w, Xc[:Bsub])
        assert rel_err(mean.cpu().numpy(), om.numpy()) < TOL_MEAN_VAR
        assert rel_err(var.cpu().numpy(), ov.numpy()) < TOL_MEAN_VAR
    # determinism: bit-identical on repetition (fixed-order reductions, no atomics)
    m1, v1 = engine.predict_weighted(fs, w.cuda(), Xc.cuda())
    m2, v2 = engine.predict_weighted(fs, w.cuda(), Xc.cuda())
    assert torch.equal(m1, m2) and torch.equal(v1, v2)


@pytest.mark.parametrize("n,d,kernel,nvs", [
    (320, 6, 0, [320, 257, 100]),    # 32-candidate tiles (k* of 64 candidates no longer fits shared memory)
    (512, 10, 3, [512, 400, 1]),     # config-4 shape: 32-candidate tiles, task staging aliased onto the L^-1 stages
    (256, 20, 2, [256, 130, 64]),    # 64-candidate tiles, aliased staging (large d)
    (256, 6, 1, [256, 130, 64]),     # Matern-1/2: k* from direct differences (not smooth in r^2), no tensor-core distances
    (192, 7, 0, [192, 77, 3]),       # d = 7: the norm rows do not fit the contraction's padding (accumulator-init path)
    (576, 1, 0, [576, 300, 2]),      # d = 1 at the prediction kernel's largest n (scaml_predict_max_points(1))
    (256, 32, 3, [256, 200, 9]),     # d = 32: 32-candidate tiles at n_pad = 256
])
def test_weighted_prediction_other_layouts(engine, n, d, kernel, nvs):
    M, B = len(nvs), 150
    pb = make_problem(M, 2, n, d, seed=8, n_valid=nvs, kernel=kernel)
    batch = _batch(pb)
    th = pb["th"][:, 1].contiguous()
    fs = engine.factorize(batch, th.cuda(), pb["cspec"])
    assert int(fs.info.abs().max()) == 0
    states = [O.factorize(pb["X"][m, : pb["nv"][m]], pb["Y"][m, : pb["nv"][m]], th[m], pb["ospec"]) for m in range(M)]
    g = torch.Generator().manual_seed(6)
    Xc = torch.rand(B, d, dtype=torch.float64, generator=g)
    w = torch.rand(M, dtype=torch.float64, generator=g)
    mean, var = engine.predict_weighted(fs, w.cuda(), Xc.cuda())
    om, ov = O.scaml_prior_predict(states, w, Xc)
    assert rel_err(mean.cpu().numpy(), om.numpy()) < TOL_MEAN_VAR
    # variances are differences s - ||v||^2: compare relative to the prior scale (DESIGN.md section 6)
    scale = float(sum(float(wi) ** 2 * float(st.os) * st.ystd ** 2 for wi, st in zip(w, states)))
    assert float((var.cpu() - ov).abs().max()) < TOL_MEAN_VAR * scale


def test_kernel_matrix(engine):
    M, n, d = 5, 200, 6
    pb = make_problem(M, 1, n, d, seed=2, n_valid=[200, 33, 64, 199, 128])
    theta = torch.zeros(M, d + 2, dtype=torch.float64)
    for m in range(M):
        ls, os_, nz = O.split_theta(pb["th"][m, 0], pb["ospec"])
        theta[m] = torch.cat([ls, os_.reshape(1), nz.reshape(1)])
    for kernel in (0, 1, 2, 3):
        K = engine.kernel_matrix(pb["X"].cuda().contiguous(), theta.cuda(), kernel, torch.tensor(pb["nv"]).cuda())
        K = K.cpu()
        for m in range(M):
            nv = pb["nv"][m]
            ref = O.kernel_matrix(pb["X"][m, :nv], pb["X"][m, :nv], theta[m, :d], theta[m, d], kernel) + theta[m, d + 1] * torch.eye(nv, dtype=torch.float64)
            assert float((K[m, :nv, :nv] - ref).abs().max()) < 1e-13
            assert torch.equal(K[m], K[m].T)


def test_full_size_properties_config3(engine):
    """4096 x 256 x 6 (BASELINE config 3): size-independent properties + sampled oracle rows."""
    from scamlgp_b200.engine import SourceBatch

    M, R, n, d = 4096, 2, 256, 6
    X, Y = O.synthetic_tasks(M, n, d, seed=0)
    ospec, cspec = O.HyperSpec.source(), HyperSpec.source()
    th = O.sample_theta_raw(M, R, d, ospec, seed=0)
    batch = SourceBatch.from_padded(X.cuda(), Y.cuda())
    thc = th.cuda().contiguous()
    lml, grad, info = engine.lml_grad(batch, thc, cspec)
    assert int(info.abs().max()) == 0
    assert bool(torch.isfinite(lml).all()) and bool(torch.isfinite(grad).all())
    # (1) sampled rows against the oracle
    for m in (0, 1777, 4095):
        yt, _, _ = O.standardize(Y[m])
        for r in range(R):
            v, g = O.lml_and_grad_autograd(X[m], yt, th[m, r], ospec)
            assert abs(float(lml[m, r]) - float(v)) < TOL_LML * abs(float(v))
            assert float((grad[m, r].cpu() - g).abs().max()) < TOL_GRAD * float(g.abs().max())
    # (2) run-to-run determinism (bit-identical)
    lml2, grad2, _ = engine.lml_grad(batch, thc, cspec)
    assert torch.equal(lml, lml2) and torch.equal(grad, grad2)
    # (3) permutation equivariance over tasks: results do not depend on which CTA/slot ran a task
    perm = torch.randperm(M, generator=torch.Generator().manual_seed(1))
    bp = SourceBatch.from_padded(X[perm].cuda(), Y[perm].cuda())
    lml3, grad3, _ = engine.lml_grad(bp, thc[perm.cuda()].contiguous(), cspec)
    assert torch.equal(lml3, lml[perm.cuda()]) and torch.equal(grad3, grad[perm.cuda()])
    # (4) directional finite difference of the fused objective matches the fused gradient
    dirn = torch.randn(M, R, d + 2, dtype=torch.float64, generator=torch.Generator().manual_seed(2)).cuda()
    eps = 1e-6
    lp, _, _ = engine.lml_grad(batch, (thc + eps * dirn).contiguous(), cspec)
    lm, _, _ = engine.lml_grad(batch, (thc - eps * dirn).contiguous(), cspec)
    fd = (lp - lm) / (2 * eps)
    an = (grad * dirn).sum(-1)
    assert float(((fd - an).abs() / (an.abs() + 1e-2)).max()) < 1e-4


def _states(pb, col=0):
    M = pb["M"]
    return [O.factorize(pb["X"][m, : pb["nv"][m]], pb["Y"][m, : pb["nv"][m]], pb["th"][m, col], pb["ospec"])
            for m in range(M)]


@pytest.mark.parametrize("kernel,nA,nB", [(0, 100, 80), (3, 33, 31), (0, 1, 1)])
def test_predict_cross_per_task_and_reduced(engine, kernel, nA, nB):
    """source_means / source_covs caches (reference model.py:278-289) and the weighted joint blocks."""
    M, n, d = 7, 256, 6
    pb = make_problem(M, 1, n, d, seed=13, n_valid=[256, 200, 64, 65, 1, 130, 256], kernel=kernel)
    batch = _batch(pb)
    fs = engine.factorize(batch, pb["th"][:, 0].contiguous().cuda(), pb["cspec"])
    states = _states(pb)
    g = torch.Generator().manual_seed(3)
    XA = torch.rand(nA, d, dtype=torch.float64, generator=g)
    XB = torch.rand(nB, d, dtype=torch.float64, generator=g)
    mean, cov = engine.predict_cross(fs, XA.cuda(), XB.cuda())
    mean, cov = mean.cpu().numpy(), cov.cpu().numpy()
    ref = []
    for m in range(M):
        mu, c = O.posterior(states[m], torch.cat([XA, XB]), full_cov=True)
        rc = c[:nA, nA:].numpy()
        ref.append(rc)
        assert np.abs(mean[:, m] - mu[:nA].numpy()).max() < TOL_MEAN_VAR * max(1.0, float(mu.abs().max()))
        assert np.abs(cov[:, :, m] - rc).max() < TOL_MEAN_VAR * float(states[m].os) * states[m].ystd ** 2
    w = torch.rand(M, dtype=torch.float64, generator=g)
    w[2] = 0.0
    mr, cr = engine.predict_cross(fs, XA.cuda(), XB.cuda(), w=w.cuda())
    wn = w.numpy()
    scale = max(float(states[m].os) * states[m].ystd ** 2 for m in range(M))
    assert np.abs(mr.cpu().numpy() - (mean * wn[None, :]).sum(1)).max() < 1e-11 * max(1.0, np.abs(mean).max())
    assert np.abs(cr.cpu().numpy() - sum(wn[m] ** 2 * ref[m] for m in range(M))).max() < TOL_MEAN_VAR * scale
    # symmetric call: Sigma(A, A) is symmetric and its diagonal equals the q = 1 variance
    _, caa = engine.predict_cross(fs, XA.cuda(), None, w=w.cuda())
    _, var = engine.predict_weighted(fs, w.cuda(), XA.cuda())
    assert float((caa - caa.T).abs().max()) < 1e-12 * scale
    assert float((caa.diagonal() - var).abs().max()) < TOL_MEAN_VAR * scale


@pytest.mark.parametrize("kernel,nt,M", [(0, 40, 64), (3, 80, 33), (0, 116, 8), (2, 1, 5)])
def test_target_lml_grad_matches_oracle(engine, kernel, nt, M):
    """a7: ScaMLGP.forward training branch + priors (reference model.py:319-338,359-383)."""
    _target_case(engine, kernel, nt, M, 4)


@pytest.mark.parametrize("kernel,d", [(0, 2), (3, 16)])
def test_target_lml_grad_above_shared_memory_limit(engine, kernel, d):
    """The first n_t above scaml_target_max_points(d): the BIG variant of the target kernels."""
    nt = engine.lib.target_max_points(d) + 1
    _target_case(engine, kernel, nt, 5, d)


def _target_case(engine, kernel, nt, M, d):
    n, R = 64, 3
    pb = make_problem(M, 1, n, d, seed=17)
    batch = _batch(pb)
    fs = engine.factorize(batch, pb["th"][:, 0].contiguous().cuda(), pb["cspec"])
    states = _states(pb)
    g = torch.Generator().manual_seed(5)
    Xt = torch.rand(nt, d, dtype=torch.float64, generator=g)
    Yt = torch.sin(3.0 * Xt.sum(1)) + 0.1 * torch.randn(nt, dtype=torch.float64, generator=g)
    cache = O.build_target_cache(states, Xt, Yt)
    sm, sc = engine.predict_cross(fs, Xt.cuda())
    scale = max(float(s.os) * s.ystd ** 2 for s in states)
    assert float((sm.cpu() - cache.source_means).abs().max()) < TOL_MEAN_VAR * max(1.0, float(cache.source_means.abs().max()))
    assert float((sc.cpu() - cache.source_covs).abs().max()) < TOL_MEAN_VAR * scale
    ospec, cspec = O.HyperSpec.target(kernel), HyperSpec.target(kernel)
    W = torch.rand(R, M, dtype=torch.float64, generator=g) / M + 1e-3
    TH = O.sample_theta_raw(1, R, d, ospec, seed=4)[0].contiguous()
    lml, gw, gt, info = engine.target_lml_grad(sm, sc, Xt.cuda(), cache.yt_std.cuda().contiguous(), W.cuda(), TH.cuda(),
                                               cache.mu_all, cache.s_all, cspec)
    assert int(info.abs().max()) == 0
    for r in range(R):
        w = W[r].clone().requires_grad_(True)
        th = TH[r].clone().requires_grad_(True)
        v = O.target_objective(cache, w, th, ospec)
        ogw, ogt = torch.autograd.grad(v, [w, th])
        assert abs(float(lml[r]) - float(v)) < TOL_LML * abs(float(v))
        gmax = max(float(ogw.abs().max()), float(ogt.abs().max()))
        assert float((gw[r].cpu() - ogw).abs().max()) < TOL_GRAD * gmax
        assert float((gt[r].cpu() - ogt).abs().max()) < TOL_GRAD * gmax


def test_full_size_properties_config5(engine):
    """Config-5 shape (4096 fitted base GPs, n = 256, d = 6; a 16k-candidate slice of the 1 Mi batch), checked
    through size-independent properties: the weighted mean is linear in w, the weighted variance is quadratic
    in w and additive over disjoint task sets, a sub-batch of candidates reproduces the big batch bit for bit,
    sampled candidates agree with the oracle, and every variance stays in (0, prior]."""
    from scamlgp_b200.engine import SourceBatch

    M, n, d, B = 4096, 256, 6, 16384
    X, Y = O.synthetic_tasks(M, n, d, seed=21)
    ospec, cspec = O.HyperSpec.source(), HyperSpec.source()
    th = O.sample_theta_raw(M, 2, d, ospec, seed=21)[:, 1].contiguous()
    batch = SourceBatch.from_padded(X.cuda(), Y.cuda())
    fs = engine.factorize(batch, th.cuda(), cspec)
    assert int(fs.info.abs().max()) == 0
    g = torch.Generator().manual_seed(2)
    Xc = torch.rand(B, d, dtype=torch.float64, generator=g).cuda()
    w1 = torch.rand(M, dtype=torch.float64, generator=g).cuda() / M
    w2 = torch.rand(M, dtype=torch.float64, generator=g).cuda() / M
    m1, v1 = (t.clone() for t in engine.predict_weighted(fs, w1, Xc))
    m2, v2 = (t.clone() for t in engine.predict_weighted(fs, w2, Xc))
    m12, _ = (t.clone() for t in engine.predict_weighted(fs, w1 + w2, Xc))
    assert float((m12 - (m1 + m2)).abs().max()) < 1e-12 * float(m12.abs().max())          # linear in w
    m3, v3 = (t.clone() for t in engine.predict_weighted(fs, 3.0 * w1, Xc))
    assert float((v3 - 9.0 * v1).abs().max()) < 1e-12 * float(v3.abs().max())               # quadratic in w
    lo, hi = w1.clone(), w1.clone()
    lo[M // 2:] = 0.0
    hi[: M // 2] = 0.0
    ma, va = (t.clone() for t in engine.predict_weighted(fs, lo, Xc))
    mb, vb = (t.clone() for t in engine.predict_weighted(fs, hi, Xc))
    assert float((ma + mb - m1).abs().max()) < 1e-12 * float(m1.abs().max())                # additive over tasks
    assert float((va + vb - v1).abs().max()) < 1e-12 * float(v1.abs().max())
    # a sub-batch reproduces the big batch up to the re-association of the task sum (the number of task splits
    # depends on how many candidate tiles there are; within one launch shape results are bit-identical)
    ms, vs = engine.predict_weighted(fs, w1, Xc[:4096].contiguous())
    assert float((ms - m1[:4096]).abs().max()) < 1e-13 * float(m1.abs().max())
    assert float((vs - v1[:4096]).abs().max()) < 1e-13 * float(v1.abs().max())
    ms2, vs2 = engine.predict_weighted(fs, w1, torch.flip(Xc, dims=[0]).contiguous())
    assert torch.equal(torch.flip(ms2, dims=[0])[64:-64], m1[64:-64]) or \
        float((torch.flip(ms2, dims=[0]) - m1).abs().max()) < 1e-13 * float(m1.abs().max())
    prior = float((w1 ** 2 * fs.theta[:, d] * batch.ystd ** 2).sum())
    assert bool((v1 > 0).all()) and float(v1.max()) <= prior * (1 + 1e-12)
    # sampled oracle check: 3 candidates, all 4096 tasks on the CPU would take minutes -> 64 tasks with the
    # other weights zeroed (the kernel skips them, exactly as pruning does)
    sel = torch.arange(0, M, 64)
    ws = torch.zeros(M, dtype=torch.float64)
    ws[sel] = w1[sel].cpu()
    mo, vo = engine.predict_weighted(fs, ws.cuda(), Xc[:3].contiguous())
    states = [O.factorize(X[m], Y[m], th[m], ospec) for m in sel.tolist()]
    om, ov = O.scaml_prior_predict(states, ws[sel], Xc[:3].cpu())
    assert rel_err(mo.cpu().numpy(), om.numpy()) < TOL_MEAN_VAR
    assert rel_err(vo.cpu().numpy(), ov.numpy()) < TOL_MEAN_VAR
    # race-detection stand-in (compute-sanitizer is closed on this pool): the two product groups of the prediction
    # kernel run on their own named barriers and cp.async rings, the fused cross-covariance streams A_m through the
    # spare ring slots -- at full occupancy (all 148 SMs, 4096 tasks each) repeated launches must agree bit for bit
    ma2, va2 = engine.predict_weighted(fs, w1, Xc)
    assert torch.equal(ma2, m1) and torch.equal(va2, v1)
    Xt = torch.rand(32, d, dtype=torch.float64, generator=g).cuda()
    A = engine.cond_prepare(fs, Xt)
    c1 = [t.clone() for t in engine.predict_conditioned(fs, w1, Xc, Xt, A)]
    c2 = engine.predict_conditioned(fs, w1, Xc, Xt, A)
    assert all(torch.equal(a, b) for a, b in zip(c1, c2))
    assert torch.equal(c1[0], m1) and torch.equal(c1[1], v1)  # the CROSS variant leaves mean / variance untouched
    K1 = engine.kernel_matrix(batch.X, fs.theta, 0).clone()
    assert torch.equal(engine.kernel_matrix(batch.X, fs.theta, 0), K1) and torch.equal(K1, K1.transpose(1, 2))


@pytest.mark.parametrize("n,d,kernel,nvs,nt", [
    (256, 6, 0, [256, 130, 64, 7], 80),     # 64-candidate tiles, n_t = 80 (10 column blocks)
    (512, 10, 0, [512, 400, 1], 20),        # config-4 shape: 32-candidate tiles, aliased staging, 16-wide panels
    (320, 6, 3, [320, 257, 100], 116),      # Matern-5/2, n_t at the target kernels' limit
])
def test_conditioning_from_A_matches_oracle(engine, n, d, kernel, nvs, nt):
    """scaml_cond_prepare / scaml_cond_caches / scaml_predict_conditioned (cross-covariance fused into the
    prediction kernel) against the oracle at the shapes the stand-alone cross kernel cannot reach (n > 256)."""
    M, B = len(nvs), 200
    pb = make_problem(M, 2, n, d, seed=17, n_valid=nvs, kernel=kernel)
    batch = _batch(pb)
    th = pb["th"][:, 1].contiguous()
    fs = engine.factorize(batch, th.cuda(), pb["cspec"])
    assert int(fs.info.abs().max()) == 0
    g = torch.Generator().manual_seed(3)
    Xc = torch.rand(B, d, dtype=torch.float64, generator=g)
    Xt = torch.rand(nt, d, dtype=torch.float64, generator=g)
    w = torch.rand(M, dtype=torch.float64, generator=g)
    A = engine.cond_prepare(fs, Xt.cuda())
    pm, pv, cross = engine.predict_conditioned(fs, w.cuda(), Xc.cuda(), Xt.cuda(), A)
    sm, sc = engine.cond_caches(fs, Xt.cuda(), A)
    ref_cross = torch.zeros(B, nt, dtype=torch.float64)
    ref_mean = torch.zeros(B, dtype=torch.float64)
    scale = 0.0
    for m in range(M):
        k = int(pb["nv"][m])
        st = O.factorize(pb["X"][m, :k], pb["Y"][m, :k], th[m], pb["ospec"])
        mu, c = O.posterior(st, torch.cat([Xc, Xt]), full_cov=True)
        ref_cross += w[m] ** 2 * c[:B, B:]
        ref_mean += w[m] * mu[:B]
        scale += float(w[m] ** 2 * st.os * st.ystd ** 2)
        assert rel_err(sm[:, m].cpu().numpy(), mu[B:].numpy()) < TOL_MEAN_VAR
        assert float((sc[:, :, m].cpu() - c[B:, B:]).abs().max()) < TOL_MEAN_VAR * float(st.os * st.ystd ** 2)
    assert rel_err(pm.cpu().numpy(), ref_mean.numpy()) < TOL_MEAN_VAR
    assert float((cross.cpu() - ref_cross).abs().max()) < TOL_MEAN_VAR * scale


def test_repeated_launches_are_bit_identical_at_full_occupancy(engine):
    """compute-sanitizer is not available on this pool; a data race in a kernel shows up as run-to-run differences
    once every SM runs its full complement of co-resident CTAs.  Fit (both variants), prediction and the fused
    conditioned prediction are launched three times each on a batch that fills the machine."""
    from scamlgp_b200.engine import SourceBatch

    M, R, n, d = 1024, 2, 256, 6
    X, Y = O.synthetic_tasks(M, n, d, seed=31)
    th = O.sample_theta_raw(M, R, d, O.HyperSpec.source(), seed=31).cuda().contiguous()
    batch = SourceBatch.from_padded(X.cuda(), Y.cuda())
    spec = HyperSpec.source()
    for impl in ("4", "8"):
        os.environ["SCAML_FIT_IMPL"] = impl
        try:
            ref = None
            for _ in range(3):
                lml, grad, info = engine.lml_grad_raw(batch, th, spec)
                torch.cuda.synchronize()
                cur = (lml.clone(), grad.clone())
                if ref is None:
                    ref = cur
                assert torch.equal(ref[0], cur[0]) and torch.equal(ref[1], cur[1])
        finally:
            del os.environ["SCAML_FIT_IMPL"]
    fs = engine.factorize(batch, th[:, 1].contiguous(), spec)
    g = torch.Generator().manual_seed(1)
    Xc = torch.rand(148 * 64, d, dtype=torch.float64, generator=g).cuda()
    Xt = torch.rand(40, d, dtype=torch.float64, generator=g).cuda()
    w = (torch.rand(M, dtype=torch.float64, generator=g) / M).cuda()
    A = engine.cond_prepare(fs, Xt)
    assert torch.equal(A, engine.cond_prepare(fs, Xt))
    ref = None
    for _ in range(3):
        out = [t.clone() for t in engine.predict_conditioned(fs, w, Xc, Xt, A)]
        if ref is None:
            ref = out
        assert all(torch.equal(a, b) for a, b in zip(ref, out))
    pm, pv = engine.predict_weighted(fs, w, Xc)
    assert float((pm - ref[0]).abs().max()) <= 1e-13 * float(pm.abs().max())  # 16- vs 8-way assembly: same sums
