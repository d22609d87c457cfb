"""Every kernel instantiation the C ABI can dispatch to is launched by some test case.

The entry points pick a template instantiation (or a plain helper kernel) from the shape of the call: the 4- or
8-warp fit kernel, the prediction tile width and the CROSS flag, the `cond_prepare` panel width (NJT), the
values-from-U register variant (NCB), DMAX of the gradient and q-block kernels, the small or BIG target kernels,
the split-reduction kernels.  Template selection depends on the shape only, never on the SM count, so which
instantiation a shape reaches on the CPU logic emulation is which it reaches on the sm_100a build.

The emulation build records the demangled name of every kernel it launches (`scaml_debug_launch_log`).  The table
below runs small shapes through the engine and checks
  (a) that each case launched the instantiations it names, and
  (b) that every `scaml::*_kernel` symbol the emulation library exports is launched by some case, or is listed in
      UNREACHABLE with the reason.
A new variant without a case fails (b); a shape rule that moves a case to another variant fails (a).  The
numerical checks of the same variants against the oracle live in the other test modules."""
import ctypes as C
import re
import subprocess

import pytest
import torch

from oracle import scaml_oracle as O
from scamlgp_b200._capi import HyperSpec
from tests.helpers import make_problem

DT = torch.float64

# exported kernels no emulated shape reaches, with the reason
UNREACHABLE = {
    # task-split reduction with >= 32 splits; the number of splits is at most 2 x (SM count), and the emulation has
    # 2 SMs.  Its reduction order is checked on the GPU (test_gpu_parity: many tasks, few candidates).
    "scaml::scaml_predict_reduce_wide_kernel",
}


def _log(lib):
    f = lib.lib.scaml_debug_launch_log
    f.restype, f.argtypes = C.c_size_t, [C.c_char_p, C.c_size_t]
    n = f(None, 0)
    buf = C.create_string_buffer(n + 1)
    f(buf, n + 1)
    return set(x for x in buf.value.decode().split("\n") if x)


def _short(name):
    """'void scaml::scaml_fit_kernel<0>(scaml::FitParams)' -> 'scaml::scaml_fit_kernel<0>'."""
    name = re.sub(r"^void ", "", name)
    depth, out = 0, []
    for ch in name:  # cut the parameter list: the first '(' outside template brackets
        if ch == "(" and depth == 0:
            break
        depth += ch == "<"
        depth -= ch == ">"
        out.append(ch)
    return "".join(out).strip()


def _sources(eng, K, n, d, nvs=None, M=3, seed=0):
    from scamlgp_b200.engine import SourceBatch

    pb = make_problem(M, 2, n, d, seed=seed, n_valid=nvs, kernel=K)
    batch = SourceBatch.from_padded(pb["X"], pb["Y"], torch.tensor(pb["nv"]))
    return pb, batch


def _fit(K, n, nvs=None, impl=None, d=3, M=2):
    def run(eng, monkeypatch):
        if impl is not None:
            monkeypatch.setenv("SCAML_FIT_IMPL", impl)
        pb, batch = _sources(eng, K, n, d, nvs, M=M)
        _, _, info = eng.lml_grad(batch, pb["th"][:, :1].contiguous(), pb["cspec"])
        assert int(info.abs().max()) == 0
    return run


def _kmat(d, n):
    def run(eng, monkeypatch):
        g = torch.Generator().manual_seed(1)
        X = torch.rand(2, n, d, dtype=DT, generator=g)
        th = torch.cat([torch.full((2, d), 0.4, dtype=DT), torch.ones(2, 1, dtype=DT), torch.full((2, 1), 1e-3, dtype=DT)], 1)
        for K in range(4):
            eng.kernel_matrix(X, th, K)
    return run


def _chain(K, d, n, B, nt, q, nvs=None, Kt=0, cross=True):
    """One pass of the q = 1, q-block and gradient paths through the engine (values are checked elsewhere)."""
    def run(eng, monkeypatch):
        pb, batch = _sources(eng, K, n, d, nvs)
        fs = eng.factorize(batch, pb["th"][:, 1].contiguous(), pb["cspec"])
        g = torch.Generator().manual_seed(2)
        w = torch.tensor([0.5, 0.3, 0.2], dtype=DT)
        Xc, Xt = torch.rand(B, d, dtype=DT, generator=g), torch.rand(nt, d, dtype=DT, generator=g)
        yt = torch.randn(nt, dtype=DT, generator=g)
        otspec, ctspec = O.HyperSpec.target(Kt), HyperSpec.target(Kt)
        tht = O.initial_theta_raw(d, otspec)
        eng.predict_weighted(fs, w, Xc)
        if cross:
            eng.predict_cross(fs, Xc, None, w=w)
            eng.predict_cross(fs, Xt)
        A = eng.cond_prepare(fs, Xt)
        sm, sc = eng.cond_caches(fs, Xt, A)
        ts = eng.target_factorize(sm, sc, Xt, yt, w, tht, 0.0, 1.0, ctspec)
        pm, pv, cr = eng.predict_conditioned(fs, w, Xc, Xt, A)
        U = eng.cond_prepare(fs, Xc, w)
        eng.values_from_u(fs, w, Xc, U)
        eng.values_from_u(fs, w, Xc, U, Xt, A)
        mean, var, beta = eng.target_posterior_beta(ts, pm, pv, cr, Xc)
        eng.target_posterior(ts, pm, pv, cr, Xc)
        eng.posterior_grad(fs, w, Xc, U.clone())
        eng.qblock_cov(fs, w, Xc, U, q)
        theta_t = ts.theta.clone()
        theta_t[d + 1] = 0.0
        gm, gc = torch.randn(B, dtype=DT, generator=g), torch.randn(B // q, q, q, dtype=DT, generator=g)
        eng.qblock_vjp(fs, w, Xc, U.clone(), q, gm, gc, theta_t, Kt, ts, A, beta)
        eng.posterior_grad(fs, w, Xc, U, ts, A, beta)
    return run


def _target(K, d, nt, R=2):
    """Target-GP training objective, factorisation and posterior at n_t (BIG above scaml_target_max_points(d))."""
    def run(eng, monkeypatch):
        M = 3
        g = torch.Generator().manual_seed(4)
        Xt = torch.rand(nt, d, dtype=DT, generator=g)
        S = torch.randn(nt, M, dtype=DT, generator=g)
        Z = torch.randn(M, nt, nt + 2, dtype=DT, generator=g)
        Cs = (Z @ Z.transpose(1, 2) / (nt + 2)).permute(1, 2, 0).contiguous()
        yt = torch.randn(nt, dtype=DT, generator=g)
        w = torch.tensor([0.5, 0.3, 0.2], dtype=DT)
        otspec, ctspec = O.HyperSpec.target(K), HyperSpec.target(K)
        th = O.initial_theta_raw(d, otspec).reshape(1, -1).repeat(R, 1).contiguous()
        wr = w.reshape(1, -1).repeat(R, 1).contiguous()
        eng.target_lml_grad(S, Cs, Xt, yt, wr, th, 0.0, 1.0, ctspec)
        ts = eng.target_factorize(S, Cs, Xt, yt, w, th[0].contiguous(), 0.0, 1.0, ctspec)
        Xc = torch.rand(5, d, dtype=DT, generator=g)
        eng.target_posterior(ts, torch.zeros(5, dtype=DT), torch.ones(5, dtype=DT), torch.zeros(5, nt, dtype=DT), Xc)
    return run


def _lbfgs(D):
    def run(eng, monkeypatch):
        from scamlgp_b200.lbfgs import lbfgs_minimize_device

        x0 = torch.full((2, D), 0.3, dtype=DT)
        lbfgs_minimize_device(eng, lambda x, a: ((x * x).sum(1), 2 * x), x0, maxiter=3)
    return run


def _split_combine(eng, monkeypatch):
    monkeypatch.setenv("SCAML_COMB_TSPLIT", "3")  # the task-split direct term at a tiny shape
    _chain(0, 2, 24, 4, 3, 2)(eng, monkeypatch)


# (id, run, instantiations it must launch: short names as in `_short`)
CASES = []
for _K in range(4):
    CASES += [
        (f"fit4-k{_K}", _fit(_K, 70, [70, 33]), [f"scaml::scaml_fit_kernel<{_K}>", "scaml::scaml_fit_schedule_kernel<0>"]),
        (f"fit8-forced-k{_K}", _fit(_K, 40, impl="8"), [f"scaml::f8::scaml_fit8_kernel<{_K}>"]),
        # d <= 8: DMAX 8, NJT 1 (B = 6) and 2 (n_t = 12), NCB 5, CT 64
        (f"chain-d3-k{_K}", _chain(_K, 3, 40, 6, 12, 3, [40, 21, 1], Kt=_K),
         [f"scaml::scaml_grad_contract_kernel<{_K}, 8>", f"scaml::scaml_qblock_cov_kernel<{_K}, 8>",
          f"scaml::scaml_qblock_direct_kernel<{_K}, 8>", f"scaml::scaml_cond_prepare_kernel<{_K}, 1>",
          f"scaml::scaml_cond_prepare_kernel<{_K}, 2>", f"scaml::scaml_grad_values_kernel<{_K}, 5>",
          f"scaml::scaml_predict_kernel<{_K}, 64, false>", f"scaml::scaml_predict_kernel<{_K}, 64, true>",
          f"scaml::scaml_cross_kernel<{_K}>", f"scaml::scaml_cond_caches_kernel<{_K}>",
          f"scaml::scaml_cond_combine_kernel<{_K}>", f"scaml::scaml_target_factor_kernel<{_K}, false>",
          "scaml::scaml_grad_mix_kernel", "scaml::scaml_qblock_fold_kernel", "scaml::scaml_qblock_fold_beta_kernel",
          "scaml::scaml_target_posterior_kernel<false>"]),
        # 8 < d <= 16: DMAX 16, NJT 4 (B = 20) and 8 (n_t = 40), NCB 9
        (f"chain-d12-k{_K}", _chain(_K, 12, 30, 20, 40, 4),
         [f"scaml::scaml_grad_contract_kernel<{_K}, 16>", f"scaml::scaml_qblock_cov_kernel<{_K}, 16>",
          f"scaml::scaml_qblock_direct_kernel<{_K}, 16>", f"scaml::scaml_cond_prepare_kernel<{_K}, 4>",
          f"scaml::scaml_cond_prepare_kernel<{_K}, 8>", f"scaml::scaml_grad_values_kernel<{_K}, 9>"]),
        # d = 32 at n_pad = 256: DMAX 32, 32-wide prediction tiles, NCB 17 (n_t = 70); n > 192 is beyond the
        # cross-covariance kernel at d = 32
        (f"chain-d32-k{_K}", _chain(_K, 32, 200, 4, 70, 2, [200, 70, 9], cross=False),
         [f"scaml::scaml_grad_contract_kernel<{_K}, 32>", f"scaml::scaml_qblock_cov_kernel<{_K}, 32>",
          f"scaml::scaml_qblock_direct_kernel<{_K}, 32>", f"scaml::scaml_grad_values_kernel<{_K}, 17>",
          f"scaml::scaml_predict_kernel<{_K}, 32, false>", f"scaml::scaml_predict_kernel<{_K}, 32, true>"]),
        # first n_t above scaml_target_max_points(2) = 117: the BIG factor kernel; n_t = 170 also puts L_t^-1 of the
        # posterior kernel out of shared memory
        (f"target-big-k{_K}", _target(_K, 2, 170 if _K == 0 else 118),
         [f"scaml::scaml_target_factor_kernel<{_K}, true>", "scaml::scaml_target_reduce_kernel",
          "scaml::scaml_target_wgrad_kernel"] + (["scaml::scaml_target_posterior_kernel<true>"] if _K == 0 else [])),
    ]
CASES += [
    # n_pad = 576 > 512: the 8-warp kernel is the default (one task, the emulation runs it one thread at a time)
    ("fit8-default", _fit(0, 513, d=2, M=1), ["scaml::f8::scaml_fit8_kernel<0>"]),
    ("kmat-task", _kmat(2, 20), [f"scaml::scaml_kmat_task_kernel<{k}>" for k in range(4)]),
    ("kmat-tile", _kmat(6, 200), [f"scaml::scaml_kmat_tile_kernel<{k}>" for k in range(4)]),
    ("lbfgs-narrow", _lbfgs(5), ["scaml::scaml_lbfgs_step_kernel<1>"]),
    ("lbfgs-wide", _lbfgs(600), ["scaml::scaml_lbfgs_step_kernel<8>"]),
    ("split-reductions", _split_combine,
     ["scaml::scaml_cond_combine_finish_kernel", "scaml::scaml_predict_reduce_kernel",
      "scaml::scaml_cross_reduce_kernel", "scaml::scaml_grad_finish_kernel", "scaml::scaml_grad_values_finish_kernel",
      "scaml::scaml_qblock_cov_finish_kernel"]),
]


@pytest.fixture(scope="module")
def launched(emu_lib):
    """Short names of the kernels each case launched (all cases run once per module)."""
    from tests.emu_engine import EmuEngine

    eng = EmuEngine(emu_lib)
    out = {}
    mp = pytest.MonkeyPatch()
    try:
        for cid, run, _ in CASES:
            emu_lib.lib.scaml_debug_launch_log_clear()
            with mp.context() as m:
                run(eng, m)
            out[cid] = {_short(x) for x in _log(emu_lib)}
    finally:
        mp.undo()
    return out


@pytest.mark.parametrize("cid,expected", [(c[0], c[2]) for c in CASES], ids=[c[0] for c in CASES])
def test_case_launches_its_variant(launched, cid, expected):
    missing = [e for e in expected if e not in launched[cid]]
    assert not missing, (missing, sorted(launched[cid]))


def test_every_exported_kernel_is_launched(emu_lib, launched):
    nm = subprocess.run(["nm", "-DC", "--defined-only", emu_lib.path], capture_output=True, text=True, check=True)
    kernels = set()
    for line in nm.stdout.splitlines():
        parts = line.split(" ", 2)
        if len(parts) == 3 and parts[1] in ("T", "W", "t", "w"):
            name = _short(parts[2])
            if re.match(r"^scaml::(f8::)?scaml_\w+_kernel(<[^()]*>)?$", name):
                kernels.add(name)
    assert len(kernels) > 100, sorted(kernels)  # the symbol scan itself works
    hit = set().union(*launched.values())
    assert UNREACHABLE <= kernels, UNREACHABLE - kernels  # the list names real kernels
    missing = sorted(kernels - hit - UNREACHABLE)
    assert not missing, missing
    assert not (UNREACHABLE & hit), UNREACHABLE & hit  # an "unreachable" kernel that is reached leaves the list
