"""CPU logic-emulation of the CUDA kernel SOURCES (csrc/emu/cuda_emu.h) vs the oracle.

Not a product path and not a fallback: the emulation library is only ever loaded here.
It proves, in the GPU-less CI container, that the block algorithm (tile layouts, chunk
schedules, padding, failure codes) of the very same .cuh files is right; the `-m gpu`
tests repeat the comparisons on the real sm_100a build."""
import numpy as np
import pytest
import torch

from oracle import scaml_oracle as O
from scamlgp_b200._capi import HyperSpec, packed_tiles, pad64
from tests.helpers import TOL_GRAD, TOL_LML, TOL_MEAN_VAR, grad_rel_err, lml_rel_err, make_problem, oracle_lml_grad, rel_err


def P(a):
    return None if a is None else a.ctypes.data


def emu_lml_grad(lib, pb, jitter=None):
    M, R, n, d = pb["M"], pb["R"], pb["n"], pb["d"]
    X = np.ascontiguousarray(pb["X"].numpy())
    y = np.ascontiguousarray(pb["yt"].numpy())
    th = np.ascontiguousarray(pb["th"].numpy())
    lml = np.full((M, R), -7.0)
    grad = np.full((M, R, d + 2), -7.0)
    info = np.full((M, R), -9, dtype=np.int32)
    wsb = lib.fit_workspace_bytes(M, R, n, d)
    ws = np.zeros(wsb // 8 + 8)
    lib.lml_grad(P(X), P(y), P(pb["nv"]), P(th), P(jitter), None, P(lml), P(grad), P(info), P(ws), wsb, M, R, n, d,
                 pb["cspec"])
    return lml, grad, info


@pytest.mark.parametrize("M,R,n,d,nv,kernel", [
    (2, 2, 64, 6, None, 0),
    (1, 2, 128, 3, None, 0),
    (3, 1, 192, 6, [130, 1, 64], 0),   # ragged incl. a single-point task
    (1, 1, 100, 2, None, 3),           # n not a multiple of the 64 grid, Matern-5/2
    (1, 1, 64, 4, None, 1),
    (1, 1, 64, 4, None, 2),
])
def test_emu_lml_grad_matches_oracle(emu_lib, M, R, n, d, nv, kernel):
    pb = make_problem(M, R, n, d, seed=3, n_valid=nv, kernel=kernel)
    lml, grad, info = emu_lml_grad(emu_lib, pb)
    v, g = oracle_lml_grad(pb)
    assert (info == 0).all()
    assert lml_rel_err(lml, v) < TOL_LML
    assert grad_rel_err(grad, g) < TOL_GRAD


def test_emu_reports_non_psd_pivot_and_jitter_recovers(emu_lib):
    # duplicated inputs + minimal noise + huge outputscale -> K_y numerically singular
    pb = make_problem(1, 1, 64, 2, seed=1)
    pb["X"][0, 32:] = pb["X"][0, :32]
    pb["ospec"].noise_bounds = (1e-30, 1e-2)  # let the noise vanish against the outputscale
    pb["cspec"].noise_bounds = (1e-30, 1e-2)
    spec = pb["ospec"]
    pb["th"][0, 0] = O.pack_theta(torch.full((2,), 50.0, dtype=torch.float64), 99.0, 1e-25, spec)
    lml, grad, info = emu_lml_grad(emu_lib, pb)
    assert info[0, 0] > 0 and np.isnan(lml[0, 0]) and np.isnan(grad[0, 0]).all()
    # the oracle (torch.linalg.cholesky) fails on the same matrix
    with pytest.raises(Exception):
        O.lml_and_grad_autograd(pb["X"][0], pb["yt"][0], pb["th"][0, 0], spec)
    jit = np.full((1, 1), 1e-6)
    lml, grad, info = emu_lml_grad(emu_lib, pb, jitter=jit)
    v, g = O.lml_and_grad_autograd(pb["X"][0], pb["yt"][0], pb["th"][0, 0], spec, jitter=1e-6)
    assert info[0, 0] == 0 and np.isfinite(lml[0, 0])
    assert abs(lml[0, 0] - float(v)) < 1e-6 * abs(float(v))  # cond ~ 1e8+: loose tolerance, see DESIGN.md


@pytest.mark.parametrize("n,d,kernel,nvs", [
    (128, 3, 0, [128, 77, 5]),   # RBF, d = 3: tensor-core distances, norm rows inside the contraction's padding
    (70, 7, 0, [70, 64, 9]),     # d = 7: no room for the norm rows -> accumulators initialised with |a|^2 + |c|^2
    (70, 3, 1, [70, 33, 2]),     # Matern-1/2: k* from direct differences (thread <-> candidate path)
    (70, 4, 3, [70, 65, 1]),     # Matern-5/2 through the tensor-core distances (r^2, not the folded RBF argument)
])
def test_emu_factorize_and_weighted_prediction(emu_lib, n, d, kernel, nvs):
    lib = emu_lib
    M, B = 3, 70
    pb = make_problem(M, 2, n, d, seed=5, n_valid=nvs, kernel=kernel)
    th = pb["th"][:, 1].contiguous()
    X = np.ascontiguousarray(pb["X"].numpy())
    y = np.ascontiguousarray(pb["yt"].numpy())
    thn = np.ascontiguousarray(th.numpy())
    linv = np.full((M, packed_tiles(n), 1024), np.nan)
    alpha = np.full((M, pad64(n)), np.nan)
    theta = np.zeros((M, d + 2))
    info = np.full(M, -9, dtype=np.int32)
    wsb = lib.fit_workspace_bytes(M, 1, n, d)
    ws = np.zeros(wsb // 8 + 8)
    lib.factorize(P(X), P(y), P(pb["nv"]), P(thn), None, P(linv), P(alpha), P(theta), P(info), P(ws), wsb, M, n, d,
                  pb["cspec"])
    assert (info == 0).all()
    states = [O.factorize(pb["X"][m, : pb["nv"][m]], pb["Y"][m, : pb["nv"][m]], th[m], pb["ospec"]) for m in range(M)]
    for m in range(M):
        nv = pb["nv"][m]
        assert rel_err(alpha[m, :nv], states[m].alpha.numpy()) < 1e-9
        assert (alpha[m, nv:] == 0).all()
        ls, os_, nz = O.split_theta(th[m], pb["ospec"])
        assert rel_err(theta[m], torch.cat([ls, os_.reshape(1), nz.reshape(1)]).numpy()) < 1e-14
    g = torch.Generator().manual_seed(5)
    Xc = torch.rand(B, d, dtype=torch.float64, generator=g)
    w = torch.tensor([0.5, 0.0, 0.25], dtype=torch.float64)  # middle task pruned (w = 0)
    mean, var = np.zeros(B), np.zeros(B)
    pwb = lib.predict_workspace_bytes(M, n, d, B)
    pws = np.zeros(pwb // 8 + 8)
    Xcn, wn = np.ascontiguousarray(Xc.numpy()), w.numpy().copy()
    lib.predict_weighted(P(X), P(pb["nv"]), P(theta), P(linv), P(alpha), P(pb["ybar"]), P(pb["ystd"]), P(wn), P(Xcn),
                         P(mean), P(var), P(pws), pwb, M, n, d, B, kernel)
    om, ov = O.scaml_prior_predict(states, w, Xc)
    assert rel_err(mean, om.numpy()) < TOL_MEAN_VAR
    assert rel_err(var, ov.numpy()) < TOL_MEAN_VAR


@pytest.mark.parametrize("n", [70, 200])  # whole-task kernel / tile kernel (the emulation build switches at 16 KB)
def test_emu_kernel_matrix(emu_lib, n):
    M, d = 2, 3 if n == 70 else 6
    pb = make_problem(M, 1, n, d, seed=2, n_valid=[n, 33])
    theta = np.zeros((M, d + 2))
    for m in range(M):
        ls, os_, nz = O.split_theta(pb["th"][m, 0], pb["ospec"])
        theta[m] = torch.cat([ls, os_.reshape(1), nz.reshape(1)]).numpy()
    X = np.ascontiguousarray(pb["X"].numpy())
    for kernel in (0, 3):
        K = np.full((M, n, n), np.nan)
        emu_lib.kernel_matrix(P(X), P(pb["nv"]), P(theta), P(K), M, n, d, kernel)
        for m in range(M):
            nv = pb["nv"][m]
            t = torch.tensor(theta[m])
            ref = O.kernel_matrix(pb["X"][m, :nv], pb["X"][m, :nv], t[:d], t[d], kernel) + t[d + 1] * torch.eye(nv, dtype=torch.float64)
            assert np.abs(K[m, :nv, :nv] - ref.numpy()).max() < 1e-14
            assert np.array_equal(K[m], K[m].T)
            if nv < n:
                assert np.array_equal(K[m, nv:, nv:], np.eye(n - nv))
                assert (K[m, :nv, nv:] == 0).all() and (K[m, nv:, :nv] == 0).all()


def test_emu_predict_cross_per_task_and_reduced(emu_lib):
    """source_means / source_covs caches (per task) and the weighted joint prior blocks (reduced)."""
    lib = emu_lib
    M, n, d = 3, 128, 3
    pb = make_problem(M, 2, n, d, seed=7, n_valid=[128, 70, 9])
    th = pb["th"][:, 1].contiguous()
    X = np.ascontiguousarray(pb["X"].numpy())
    y = np.ascontiguousarray(pb["yt"].numpy())
    thn = np.ascontiguousarray(th.numpy())
    linv = np.zeros((M, packed_tiles(n), 1024))
    alpha = np.zeros((M, pad64(n)))
    theta = np.zeros((M, d + 2))
    info = np.zeros(M, dtype=np.int32)
    wsb = lib.fit_workspace_bytes(M, 1, n, d)
    ws = np.zeros(wsb // 8 + 8)
    lib.factorize(P(X), P(y), P(pb["nv"]), P(thn), None, P(linv), P(alpha), P(theta), P(info), P(ws), wsb, M, n, d,
                  pb["cspec"])
    states = [O.factorize(pb["X"][m, : pb["nv"][m]], pb["Y"][m, : pb["nv"][m]], th[m], pb["ospec"]) for m in range(M)]
    g = torch.Generator().manual_seed(11)
    XA = torch.rand(37, d, dtype=torch.float64, generator=g)
    XB = torch.rand(33, d, dtype=torch.float64, generator=g)
    XAn, XBn = np.ascontiguousarray(XA.numpy()), np.ascontiguousarray(XB.numpy())
    nA, nB = XA.shape[0], XB.shape[0]
    # per task
    mean = np.full((nA, M), np.nan)
    cov = np.full((nA, nB, M), np.nan)
    lib.predict_cross(P(X), P(pb["nv"]), P(theta), P(linv), P(alpha), P(pb["ybar"]), P(pb["ystd"]), None, P(XAn),
                      P(XBn), P(mean), P(cov), None, 0, M, n, d, nA, nB, 0, 0)
    ref_cov = []
    for m in range(M):
        mu, c = O.posterior(states[m], torch.cat([XA, XB]), full_cov=True)
        assert rel_err(mean[:, m], mu[:nA].numpy()) < TOL_MEAN_VAR
        rc = c[:nA, nA:].numpy()
        ref_cov.append(rc)
        assert np.abs(cov[:, :, m] - rc).max() < TOL_MEAN_VAR * float(states[m].os) * states[m].ystd ** 2
    # reduced with weights (one task pruned)
    w = np.array([0.7, 0.0, 0.2])
    wb = lib.predict_cross_workspace_bytes(M, nA, nB, 1)
    wsr = np.zeros(wb // 8 + 8)
    mean_r = np.full(nA, np.nan)
    cov_r = np.full((nA, nB), np.nan)
    lib.predict_cross(P(X), P(pb["nv"]), P(theta), P(linv), P(alpha), P(pb["ybar"]), P(pb["ystd"]), P(w), P(XAn),
                      P(XBn), P(mean_r), P(cov_r), P(wsr), wb, M, n, d, nA, nB, 0, 1)
    assert rel_err(mean_r, (mean * w[None, :]).sum(1)) < 1e-12
    assert np.abs(cov_r - sum(w[m] ** 2 * ref_cov[m] for m in range(M))).max() < 1e-9


def _oracle_target_value_and_grads(cache, w, th, ospec):
    w = w.clone().requires_grad_(True)
    th = th.clone().requires_grad_(True)
    v = O.target_objective(cache, w, th, ospec)
    gw, gt = torch.autograd.grad(v, [w, th])
    return float(v.detach()), gw.numpy(), gt.numpy()


@pytest.mark.parametrize("kernel,nt", [(0, 9), (3, 17), (1, 1), (0, 121)])  # 121 > the shared-memory limit: BIG variant
def test_emu_target_lml_grad_matches_oracle(emu_lib, kernel, nt):
    """a7: target objective on the ScaMLGP training branch + gradient wrt weights and raw kernel params."""
    lib = emu_lib
    M, n, d, R = 5, 64, 3, 2
    pb = make_problem(M, 1, n, d, seed=9, n_valid=[64, 40, 64, 7, 33])
    states = [O.factorize(pb["X"][m, : pb["nv"][m]], pb["Y"][m, : pb["nv"][m]], pb["th"][m, 0], pb["ospec"])
              for m in range(M)]
    g = torch.Generator().manual_seed(21)
    Xt = torch.rand(nt, d, dtype=torch.float64, generator=g)
    Yt = torch.randn(nt, dtype=torch.float64, generator=g)
    cache = O.build_target_cache(states, Xt, Yt)
    ospec, cspec = O.HyperSpec.target(kernel), HyperSpec.target(kernel)
    W = torch.rand(R, M, dtype=torch.float64, generator=g) + 0.05
    TH = O.sample_theta_raw(1, R, d, ospec, seed=4)[0]
    sm = np.ascontiguousarray(cache.source_means.numpy())
    sc = np.ascontiguousarray(cache.source_covs.numpy())
    Xtn, ytn = np.ascontiguousarray(Xt.numpy()), np.ascontiguousarray(cache.yt_std.numpy())
    Wn, THn = np.ascontiguousarray(W.numpy()), np.ascontiguousarray(TH.numpy())
    lml = np.full(R, np.nan)
    gw = np.full((R, M), np.nan)
    gt = np.full((R, d + 2), np.nan)
    info = np.full(R, -9, dtype=np.int32)
    wsb = lib.target_workspace_bytes(nt, R)
    ws = np.zeros(wsb // 8 + 8)
    lib.target_lml_grad(P(sm), P(sc), P(Xtn), P(ytn), P(Wn), P(THn), None, cache.mu_all, cache.s_all, P(lml), P(gw),
                        P(gt), P(info), P(ws), wsb, M, nt, d, R, cspec)
    assert (info == 0).all()
    for r in range(R):
        v, ogw, ogt = _oracle_target_value_and_grads(cache, W[r], TH[r], ospec)
        assert abs(lml[r] - v) < TOL_LML * abs(v)
        assert np.abs(gw[r] - ogw).max() < TOL_GRAD * np.abs(ogw).max()
        assert np.abs(gt[r] - ogt).max() < TOL_GRAD * max(np.abs(ogt).max(), np.abs(ogw).max())


def test_device_exp_is_accurate_to_two_ulp(emu_lib):
    """exp_nonpos (csrc/scaml_device.cuh) replaces libdevice exp in every kernel: < 2 ulp on [-707, 0] against
    50-digit mpmath at sampled points and numpy elsewhere; clamped to exp(-708) = 3.3e-308 below, NaN propagates."""
    import ctypes as C

    import mpmath

    rng = np.random.default_rng(0)
    x = np.concatenate([-rng.uniform(0, 707, 200000), -np.exp(rng.uniform(-40, 6.5, 200000)),
                        -np.arange(0, 1024) * np.log(2) / 2, [0.0, -0.0, -1e-300, -706.999]])
    x = np.ascontiguousarray(np.minimum(x, 0.0))
    out = np.empty_like(x)
    f = emu_lib.lib.scaml_debug_exp_nonpos
    f.argtypes = [C.c_void_p, C.c_void_p, C.c_int]
    f(x.ctypes.data, out.ctypes.data, x.size)
    ref = np.exp(x)
    ulp = np.spacing(ref)
    sel = x > -707.0
    assert np.max(np.abs(out[sel] - ref[sel]) / ulp[sel]) < 2.0
    mpmath.mp.dps = 50
    for i in rng.integers(0, x.size, 300):
        if x[i] > -707.0:
            exact = mpmath.exp(mpmath.mpf(float(x[i])))
            assert abs(mpmath.mpf(float(out[i])) - exact) < 1.5 * mpmath.mpf(float(ulp[i]))
    special = np.array([-707.5, -750.0, -1e6, -np.inf, np.nan])
    so = np.empty_like(special)
    f(special.ctypes.data, so.ctypes.data, special.size)
    assert (so[:4] >= 0.0).all() and (so[:4] < 1e-307).all() and np.isnan(so[4])


def test_emu_fused_conditioning_matches_cross_kernel_and_oracle(emu_lib):
    """scaml_cond_prepare + scaml_predict_conditioned (cross-covariance fused into the prediction kernel) against
    the stand-alone cross kernel (reduce = 1) and the oracle; ragged tasks, a pruned task, n_t not a multiple of 8."""
    from tests.emu_engine import EmuEngine
    from scamlgp_b200.engine import SourceBatch

    eng = EmuEngine(emu_lib)
    M, n, d, B, nt = 3, 128, 3, 70, 11
    pb = make_problem(M, 2, n, d, seed=9, n_valid=[128, 70, 9], kernel=0)
    batch = SourceBatch.from_padded(pb["X"], pb["Y"], torch.tensor(pb["nv"]))
    th = pb["th"][:, 1].contiguous()
    fs = eng.factorize(batch, th, pb["cspec"])
    g = torch.Generator().manual_seed(4)
    Xc = torch.rand(B, d, dtype=torch.float64, generator=g)
    Xt = torch.rand(nt, d, dtype=torch.float64, generator=g)
    for w in (torch.tensor([0.5, 0.3, 0.2], dtype=torch.float64), torch.tensor([0.7, 0.0, 0.3], dtype=torch.float64)):
        A = eng.cond_prepare(fs, Xt)
        pm, pv, cross = eng.predict_conditioned(fs, w, Xc, Xt, A)
        pm0, pv0 = eng.predict_weighted(fs, w, Xc)
        _, cross0 = eng.predict_cross(fs, Xc, Xt, w=w)
        assert rel_err(pm.numpy(), pm0.numpy()) < 1e-12 and rel_err(pv.numpy(), pv0.numpy()) < 1e-12
        scale = float(cross0.abs().max())
        assert float((cross - cross0).abs().max()) < 1e-10 * scale
        # oracle: sum_m w_m^2 Sigma_m(x, X_t)
        ref = torch.zeros(B, nt, dtype=torch.float64)
        for m in range(M):
            k = int(pb["nv"][m])
            st = O.factorize(pb["X"][m, :k], pb["Y"][m, :k], th[m], pb["ospec"])
            _, c = O.posterior(st, torch.cat([Xc, Xt]), full_cov=True)
            ref += w[m] ** 2 * c[:B, B:]
        assert float((cross - ref).abs().max()) < 1e-9 * float(ref.abs().max())
    # per-task caches from A_m == the stand-alone cross kernel (reduce = 0)
    sm0, sc0 = eng.predict_cross(fs, Xt)
    sm1, sc1 = eng.cond_caches(fs, Xt, A)
    assert rel_err(sm1.numpy(), sm0.numpy()) < 1e-11
    assert float((sc1 - sc0).abs().max()) < 1e-10 * float(sc0.abs().max())
    # A_m itself: K_m^-1 K_m(X_m, X_t)
    k = int(pb["nv"][1])
    st = O.factorize(pb["X"][1, :k], pb["Y"][1, :k], th[1], pb["ospec"])
    Kmt = O.kernel_matrix(pb["X"][1, :k], Xt, st.ls, st.os, 0)
    Aref = torch.cholesky_solve(Kmt, st.L)
    assert float((A[1, :k, :nt] - Aref).abs().max()) < 1e-9 * float(Aref.abs().max())
    assert float(A[1, k:].abs().max()) == 0.0 and float(A[1, :, nt:].abs().max()) == 0.0


def test_emu_target_jitter_ladder_inside_the_kernel_matches_the_host_ladder(emu_lib):
    from tests.emu_engine import EmuEngine

    _target_ladder_case(EmuEngine(emu_lib))


@pytest.mark.gpu
def test_gpu_target_jitter_ladder_inside_the_kernel_matches_the_host_ladder(engine):
    _target_ladder_case(engine)


def _target_ladder_case(eng):
    """A weighted prior covariance that is slightly negative definite: the factorisation fails at jitter 0 and 1e-8
    and succeeds at 1e-7 (psd_safe_cholesky semantics).  The in-kernel ladder must give exactly what re-running the
    failed row from the host gives; a healthy row is untouched; a hopeless row reports info > 0 and NaN."""
    dev = eng.device
    M, nt, d, R = 3, 3, 2, 3
    spec = HyperSpec.target()
    ospec = O.HyperSpec.target()
    th = O.initial_theta_raw(d, ospec).reshape(1, -1).repeat(R, 1).contiguous()
    ls, os_, noise = O.split_theta(th[0], ospec)
    Xt = torch.tensor([[0.0, 0.0], [40.0, 0.0], [0.0, 40.0]], dtype=torch.float64)  # kappa ~ 0 off the diagonal
    yt = torch.tensor([0.1, -0.2, 0.05], dtype=torch.float64)
    sm = torch.zeros(nt, M, dtype=torch.float64)
    sc = torch.zeros(nt, nt, M, dtype=torch.float64)
    w = torch.full((R, M), 1e-6, dtype=torch.float64)  # (weights of exactly 0 have no Gamma(1, 1) log density)
    w[0, 0] = w[1, 1] = w[2, 2] = 1.0
    for a in range(nt):
        sc[a, a, 0] = -(float(os_) + float(noise)) - 3e-8   # row 0: K_y = -3e-8 I  -> recovers at +1e-7
        sc[a, a, 1] = 0.5                                   # row 1: healthy
        sc[a, a, 2] = -(float(os_) + float(noise)) - 1.0    # row 2: hopeless
    sm, sc, Xt, yt, w, th = (t.to(dev) for t in (sm, sc, Xt, yt, w, th))
    a_ = eng.target_lml_grad_safe(sm, sc, Xt, yt, w, th, 0.0, 1.0, spec)
    b_ = eng.target_lml_grad_host_ladder(sm, sc, Xt, yt, w, th, 0.0, 1.0, spec)
    assert a_[3].tolist() == b_[3].tolist() and a_[3][0] == 0 and a_[3][1] == 0 and a_[3][2] > 0
    for x, y in zip(a_[:3], b_[:3]):
        assert torch.equal(torch.nan_to_num(x, nan=-7.0), torch.nan_to_num(y, nan=-7.0))
    assert torch.isfinite(a_[0][:2]).all() and torch.isnan(a_[0][2])
    plain = eng.target_lml_grad(sm, sc, Xt, yt, w, th, 0.0, 1.0, spec)
    assert plain[3][0] > 0 and torch.equal(plain[0][1], a_[0][1])


def _source_ladder_case(eng, n=64):
    """Source fit: psd_safe_cholesky ladder inside the kernel == the host-driven ladder (bit for bit), on a ragged
    batch with a skip mask -- which also exercises the schedule pre-pass (active rows, largest tasks first)."""
    from scamlgp_b200.engine import SourceBatch

    dev = eng.device
    pb = make_problem(4, 2, n, 2, seed=1, n_valid=[n, n, n // 2 + 1, 3])
    pb["X"][1, n // 2:] = pb["X"][1, : n // 2]  # task 1: duplicated inputs -> singular without noise
    for sp in (pb["ospec"], pb["cspec"]):
        sp.noise_bounds = (1e-30, 1e-2)
    pb["th"][1, 0] = O.pack_theta(torch.full((2,), 50.0, dtype=torch.float64), 99.0, 1e-25, pb["ospec"])
    batch = SourceBatch.from_padded(pb["X"].to(dev), pb["Y"].to(dev), torch.tensor(pb["nv"]).to(dev))
    th = pb["th"].to(dev).contiguous()
    skip = torch.zeros(4, 2, dtype=torch.int32, device=dev)
    skip[0, 1] = skip[3, 0] = 1
    raw = eng.lml_grad_raw(batch, th, pb["cspec"])
    assert int(raw[2][1, 0]) > 0 and bool(torch.isnan(raw[0][1, 0]))  # fails without jitter
    a_ = eng.lml_grad(batch, th, pb["cspec"], skip=skip)
    b_ = eng.lml_grad_host_ladder(batch, th, pb["cspec"], skip=skip)
    for x, y in zip(a_, b_):
        assert torch.equal(torch.nan_to_num(x.to(torch.float64), nan=-7.0), torch.nan_to_num(y.to(torch.float64), nan=-7.0))
    assert int(a_[2].abs().max()) == 0 and bool(torch.isfinite(a_[0][skip == 0]).all())
    assert bool(torch.isnan(a_[0][skip != 0]).all())  # skipped rows are neither evaluated nor written
    assert torch.equal(a_[0][2], raw[0][2]) and torch.equal(a_[1][0, 0], raw[1][0, 0])  # healthy rows untouched
    fs = eng.factorize(batch, th[:, 0].contiguous(), pb["cspec"])
    assert int(fs.info.abs().max()) == 0 and bool(torch.isfinite(fs.alpha).all())


def test_emu_source_jitter_ladder_inside_the_kernel_matches_the_host_ladder(emu_lib):
    from tests.emu_engine import EmuEngine

    _source_ladder_case(EmuEngine(emu_lib))


@pytest.mark.gpu
def test_gpu_source_jitter_ladder_inside_the_kernel_matches_the_host_ladder(engine):
    _source_ladder_case(engine)
    _source_ladder_case(engine, n=192)


def _large_nt_case(eng, n_t, M=3, n=48, d=2, B=9):
    """n_t beyond the shared-memory limit of the target-GP kernels (116 at small d; the reference is exact to 800,
    model.py:359-384 + gpytorch's max_cholesky_size): objective, gradients, prediction state and conditioning run on
    the global-memory variants and must match the oracle like the small case."""
    from scamlgp_b200.engine import SourceBatch

    dev = eng.device
    pb = make_problem(M, 1, n, d, seed=19)
    states = [O.factorize(pb["X"][m], pb["Y"][m], pb["th"][m, 0], pb["ospec"]) for m in range(M)]
    g = torch.Generator().manual_seed(8)
    Xt = torch.rand(n_t, d, dtype=torch.float64, generator=g)
    Yt = torch.sin(4.0 * Xt).sum(1) + 0.1 * torch.randn(n_t, dtype=torch.float64, generator=g)
    cache = O.build_target_cache(states, Xt, Yt)
    ospec, cspec = O.HyperSpec.target(), HyperSpec.target()
    w = torch.rand(M, dtype=torch.float64, generator=g) + 0.1
    th = O.initial_theta_raw(d, ospec)
    batch = SourceBatch.from_padded(pb["X"].to(dev), pb["Y"].to(dev))
    fs = eng.factorize(batch, pb["th"][:, 0].contiguous().to(dev), pb["cspec"])
    assert not eng.cond_supported(fs, n_t) or n_t <= 128
    sm, sc = eng.predict_cross(fs, Xt.to(dev))
    assert float((sm.cpu() - cache.source_means).abs().max()) < TOL_MEAN_VAR * float(cache.source_means.abs().max())
    yt = cache.yt_std.to(dev).contiguous()
    g2 = torch.Generator().manual_seed(9)  # a second row with its own w and theta: per-row offsets of the global block
    W = torch.stack([w, torch.rand(M, dtype=torch.float64, generator=g2) + 0.1])
    TH = torch.stack([th, th + 0.3 * torch.randn(th.shape, dtype=torch.float64, generator=g2)])
    lml, gw, gt, info = eng.target_lml_grad_safe(sm, sc, Xt.to(dev), yt, W.to(dev), TH.to(dev), cache.mu_all,
                                                 cache.s_all, cspec)
    for r in range(2):
        v, ogw, ogt = _oracle_target_value_and_grads(cache, W[r], TH[r], ospec)
        assert int(info[r]) == 0 and abs(float(lml[r]) - v) < TOL_LML * abs(v)
        assert np.abs(gw[r].cpu().numpy() - ogw).max() < TOL_GRAD * np.abs(ogw).max()
        assert np.abs(gt[r].cpu().numpy() - ogt).max() < TOL_GRAD * max(np.abs(ogt).max(), np.abs(ogw).max())
    ts = eng.target_factorize(sm, sc, Xt.to(dev), yt, w.to(dev), th.to(dev), cache.mu_all, cache.s_all, cspec)
    Xc = torch.rand(B, d, dtype=torch.float64, generator=g)
    pm, pv = eng.predict_weighted(fs, w.to(dev), Xc.to(dev))
    _, cross = eng.predict_cross(fs, Xc.to(dev), Xt.to(dev), w=w.to(dev))
    mean, var = eng.target_posterior(ts, pm, pv, cross, Xc.to(dev).contiguous())
    om, ov = O.scaml_posterior(states, w, cache, th, ospec, Xc, prune_threshold=None)
    assert float((mean.cpu() - om).abs().max()) < 1e-8 * float(om.abs().max())
    assert float((var.cpu() - ov).abs().max()) < 1e-8 * float(ov.abs().max())


def test_emu_target_kernels_beyond_the_shared_memory_limit(emu_lib):
    from tests.emu_engine import EmuEngine

    _large_nt_case(EmuEngine(emu_lib), 124)


@pytest.mark.gpu
@pytest.mark.parametrize("n_t", [130, 400])
def test_gpu_target_kernels_beyond_the_shared_memory_limit(engine, n_t):
    _large_nt_case(engine, n_t, M=6, n=96, d=3, B=200)
