"""ctypes binding of the C ABI declared in include/scaml_b200.h.

The binding is address based (plain integers for pointers) so the same code drives
  * the product library  csrc/libscaml_b200.so  (sm_100a, device pointers), and
  * in CPU-only CI, the logic-emulation build of the same kernel sources
    (tests/ only; host pointers) -- see csrc/emu/cuda_emu.h.
Nothing here falls back to a CPU implementation: `load_cuda_library()` raises if the
sm_100a library has not been built.
"""
from __future__ import annotations

import ctypes as C
import os
from dataclasses import dataclass
from typing import Optional, Tuple

KERNEL_RBF, KERNEL_MATERN12, KERNEL_MATERN32, KERNEL_MATERN52 = 0, 1, 2, 3
PRIOR_NONE, PRIOR_GAMMA, PRIOR_LOGNORMAL = 0, 1, 2

_HERE = os.path.dirname(os.path.abspath(__file__))
CUDA_LIB_PATH = os.path.join(_HERE, "csrc", "libscaml_b200.so")


class CHyperSpec(C.Structure):
    _fields_ = [
        ("kernel", C.c_int32),
        ("ls_prior", C.c_int32),
        ("os_prior", C.c_int32),
        ("noise_prior", C.c_int32),
        ("ls_lo", C.c_double),
        ("ls_hi", C.c_double),
        ("os_lo", C.c_double),
        ("os_hi", C.c_double),
        ("noise_lo", C.c_double),
        ("noise_hi", C.c_double),
        ("ls_p1", C.c_double),
        ("ls_p2", C.c_double),
        ("os_p1", C.c_double),
        ("os_p2", C.c_double),
        ("noise_p1", C.c_double),
        ("noise_p2", C.c_double),
    ]


@dataclass
class HyperSpec:
    """Kernel family, Interval constraints, priors and initial values of one GP.

    Defaults are the source-GP settings of the reference (scamlgp/model.py:25-70);
    `HyperSpec.target()` gives the target-GP defaults (model.py:73-105).
    """

    kernel: int = KERNEL_RBF
    ls_bounds: Tuple[float, float] = (1e-4, 1e2)
    os_bounds: Tuple[float, float] = (1e-4, 1e2)
    noise_bounds: Tuple[float, float] = (1e-8, 1e-2)
    ls_prior: Tuple[int, float, float] = (PRIOR_GAMMA, 3.0, 6.0)
    os_prior: Tuple[int, float, float] = (PRIOR_GAMMA, 2.0, 0.15)
    noise_prior: Tuple[int, float, float] = (PRIOR_LOGNORMAL, -8.0, 2.0)
    ls_init: float = 0.5
    os_init: float = 1.0
    noise_init: float = 1e-3

    @staticmethod
    def source(kernel: int = KERNEL_RBF) -> "HyperSpec":
        return HyperSpec(kernel=kernel)

    @staticmethod
    def target(kernel: int = KERNEL_RBF) -> "HyperSpec":
        return HyperSpec(
            kernel=kernel,
            ls_prior=(PRIOR_LOGNORMAL, 0.5, 1.5),
            os_prior=(PRIOR_LOGNORMAL, -2.0, 3.0),
            ls_init=1.0,
            os_init=0.1,
        )

    def to_c(self) -> CHyperSpec:
        return CHyperSpec(
            int(self.kernel), int(self.ls_prior[0]), int(self.os_prior[0]), int(self.noise_prior[0]),
            self.ls_bounds[0], self.ls_bounds[1], self.os_bounds[0], self.os_bounds[1],
            self.noise_bounds[0], self.noise_bounds[1],
            float(self.ls_prior[1]), float(self.ls_prior[2]),
            float(self.os_prior[1]), float(self.os_prior[2]),
            float(self.noise_prior[1]), float(self.noise_prior[2]),
        )


class CLbfgsState(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in ("x", "f", "g", "d", "t", "S", "Y", "rho", "count", "head", "iters",
                                          "ls_count", "flags")]


EXPORTED_SYMBOLS = (
    "scaml_version",
    "scaml_fit_limits",
    "scaml_fit_workspace_bytes",
    "scaml_kernel_matrix",
    "scaml_lml_grad",
    "scaml_lml_grad_ladder",
    "scaml_factorize",
    "scaml_factorize_ladder",
    "scaml_predict_max_points",
    "scaml_predict_workspace_bytes",
    "scaml_predict_weighted",
    "scaml_predict_cross_max_points",
    "scaml_predict_cross_workspace_bytes",
    "scaml_predict_cross",
    "scaml_target_workspace_bytes",
    "scaml_target_max_points",
    "scaml_target_lml_grad",
    "scaml_target_lml_grad_ladder",
    "scaml_target_posterior_beta",
    "scaml_posterior_grad_workspace_bytes",
    "scaml_posterior_grad",
    "scaml_qblock_cov_workspace_bytes",
    "scaml_qblock_cov",
    "scaml_qblock_vjp_workspace_bytes",
    "scaml_qblock_vjp",
    "scaml_cond_prepare_pruned",
    "scaml_cond_combine_task_splits",
    "scaml_posterior_values_from_u_workspace_bytes",
    "scaml_posterior_values_from_u",
    "scaml_target_factorize",
    "scaml_target_posterior",
    "scaml_lbfgs_step",
    "scaml_cond_prepare",
    "scaml_cond_caches",
    "scaml_predict_conditioned_workspace_bytes",
    "scaml_predict_conditioned",
)


class ScamlError(RuntimeError):
    pass


class NotPSDError(ScamlError):
    """linear_operator.utils.errors.NotPSDError stand-in: a covariance is not positive definite even after the
    psd_safe_cholesky jitter ladder (1e-8, 1e-7, 1e-6)."""


_ERRORS = {-1: "bad argument", -2: "workspace too small", -3: "unsupported size (d or n_max)",
           -4: "configuration does not fit shared memory"}


def _check(rc: int, what: str) -> None:
    if rc != 0:
        msg = _ERRORS.get(rc, f"CUDA error {rc}" if rc > 0 else f"error {rc}")
        raise ScamlError(f"{what}: {msg}")


class ScamlLib:
    """Typed view of one loaded libscaml shared object."""

    def __init__(self, path: str):
        if not os.path.exists(path):
            raise ScamlError(
                f"{path} not found: build the sm_100a library first "
                "(python -c 'import __graft_entry__ as g; g.build()'). There is no CPU fallback."
            )
        self.path = path
        self.lib = C.CDLL(path)
        L = self.lib
        vp, i32, sz = C.c_void_p, C.c_int, C.c_size_t
        L.scaml_version.restype = C.c_char_p
        L.scaml_fit_limits.argtypes = [C.POINTER(C.c_int), C.POINTER(C.c_int)]
        L.scaml_fit_workspace_bytes.restype = sz
        L.scaml_fit_workspace_bytes.argtypes = [i32, i32, i32, i32]
        L.scaml_kernel_matrix.argtypes = [vp, vp, vp, vp, i32, i32, i32, i32, vp]
        L.scaml_lml_grad.argtypes = [vp] * 10 + [sz, i32, i32, i32, i32, C.POINTER(CHyperSpec), vp]
        L.scaml_factorize.argtypes = [vp] * 10 + [sz, i32, i32, i32, C.POINTER(CHyperSpec), vp]
        L.scaml_lml_grad_ladder.argtypes = [vp] * 9 + [sz, i32, i32, i32, i32, C.POINTER(CHyperSpec), vp]
        L.scaml_factorize_ladder.argtypes = [vp] * 9 + [sz, i32, i32, i32, C.POINTER(CHyperSpec), vp]
        L.scaml_predict_workspace_bytes.restype = sz
        L.scaml_predict_workspace_bytes.argtypes = [i32, i32, i32, i32]
        L.scaml_predict_weighted.argtypes = [vp] * 12 + [sz, i32, i32, i32, i32, i32, vp]
        L.scaml_predict_cross_workspace_bytes.restype = sz
        L.scaml_predict_cross_workspace_bytes.argtypes = [i32, i32, i32, i32]
        L.scaml_predict_cross.argtypes = [vp] * 13 + [sz, i32, i32, i32, i32, i32, i32, i32, vp]
        dbl = C.c_double
        L.scaml_target_factorize.argtypes = ([vp] * 6 + [dbl, dbl, dbl] + [vp] * 6 +
                                             [sz, i32, i32, i32, C.POINTER(CHyperSpec), vp])
        L.scaml_target_posterior.argtypes = [vp] * 8 + [dbl, dbl, vp, vp, i32, i32, i32, i32, vp]
        L.scaml_target_posterior_beta.argtypes = [vp] * 8 + [dbl, dbl, vp, vp, vp, i32, i32, i32, i32, vp]
        L.scaml_posterior_grad_workspace_bytes.restype = sz
        L.scaml_posterior_grad_workspace_bytes.argtypes = [i32, i32, i32, i32]
        L.scaml_posterior_grad.argtypes = [vp] * 13 + [dbl, vp, vp, vp, sz] + [i32] * 7 + [vp]
        L.scaml_qblock_cov_workspace_bytes.restype = sz
        L.scaml_qblock_cov_workspace_bytes.argtypes = [i32, i32, i32]
        L.scaml_qblock_cov.argtypes = [vp] * 9 + [sz] + [i32] * 6 + [vp]
        L.scaml_qblock_vjp_workspace_bytes.restype = sz
        L.scaml_qblock_vjp_workspace_bytes.argtypes = [i32] * 5
        L.scaml_qblock_vjp.argtypes = [vp] * 13 + [dbl] + [vp] * 4 + [sz] + [i32] * 8 + [vp]
        L.scaml_posterior_values_from_u_workspace_bytes.restype = sz
        L.scaml_posterior_values_from_u_workspace_bytes.argtypes = [i32, i32, i32]
        L.scaml_posterior_values_from_u.argtypes = [vp] * 15 + [sz] + [i32] * 6 + [vp]
        L.scaml_lbfgs_step.argtypes = [C.POINTER(CLbfgsState), vp, vp, vp, vp, i32, i32, i32, i32, dbl, dbl, i32, i32, vp]
        L.scaml_cond_prepare.argtypes = [vp] * 6 + [i32] * 5 + [vp]
        L.scaml_cond_prepare_pruned.argtypes = [vp] * 7 + [i32] * 5 + [vp]
        L.scaml_cond_caches.argtypes = [vp] * 10 + [i32] * 5 + [vp]
        L.scaml_cond_combine_task_splits.argtypes = [i32, i32, i32]
        L.scaml_predict_conditioned_workspace_bytes.restype = sz
        L.scaml_predict_conditioned_workspace_bytes.argtypes = [i32] * 5
        L.scaml_predict_conditioned.argtypes = [vp] * 15 + [sz] + [i32] * 6 + [vp]
        L.scaml_target_workspace_bytes.restype = sz
        L.scaml_target_workspace_bytes.argtypes = [i32, i32]
        L.scaml_target_max_points.argtypes = [i32]
        L.scaml_target_max_points.restype = i32
        L.scaml_predict_max_points.argtypes = [i32]
        L.scaml_predict_max_points.restype = i32
        L.scaml_predict_cross_max_points.argtypes = [i32]
        L.scaml_predict_cross_max_points.restype = i32
        L.scaml_target_lml_grad_ladder.argtypes = ([vp] * 6 + [C.c_double, C.c_double] + [vp] * 5 +
                                                   [sz, i32, i32, i32, i32, C.POINTER(CHyperSpec), i32, C.c_double,
                                                    C.c_double, vp])
        L.scaml_target_lml_grad.argtypes = ([vp] * 7 + [C.c_double, C.c_double] + [vp] * 5 +
                                            [sz, i32, i32, i32, i32, C.POINTER(CHyperSpec), i32, C.c_double,
                                             C.c_double, vp])

    # ---- thin, address-based wrappers ------------------------------------------------ #
    def version(self) -> str:
        return self.lib.scaml_version().decode()

    def fit_limits(self) -> Tuple[int, int]:
        n, d = C.c_int(0), C.c_int(0)
        self.lib.scaml_fit_limits(C.byref(n), C.byref(d))
        return n.value, d.value

    def fit_workspace_bytes(self, M: int, R: int, n_max: int, d: int) -> int:
        return int(self.lib.scaml_fit_workspace_bytes(M, R, n_max, d))

    def predict_workspace_bytes(self, M: int, n_max: int, d: int, B: int) -> int:
        return int(self.lib.scaml_predict_workspace_bytes(M, n_max, d, B))

    def kernel_matrix(self, X, n_valid, theta, K, M, n_max, d, kernel, stream=0):
        _check(self.lib.scaml_kernel_matrix(X, n_valid, theta, K, M, n_max, d, kernel, stream), "scaml_kernel_matrix")

    def lml_grad(self, X, y, n_valid, theta_raw, jitter, skip, lml, grad, info, ws, ws_bytes, M, R, n_max, d,
                 spec: HyperSpec, stream=0):
        cs = spec.to_c()
        _check(self.lib.scaml_lml_grad(X, y, n_valid, theta_raw, jitter, skip, lml, grad, info, ws, ws_bytes,
                                       M, R, n_max, d, C.byref(cs), stream), "scaml_lml_grad")

    def lml_grad_ladder(self, X, y, n_valid, theta_raw, skip, lml, grad, info, ws, ws_bytes, M, R, n_max, d,
                        spec: HyperSpec, stream=0):
        cs = spec.to_c()
        _check(self.lib.scaml_lml_grad_ladder(X, y, n_valid, theta_raw, skip, lml, grad, info, ws, ws_bytes,
                                              M, R, n_max, d, C.byref(cs), stream), "scaml_lml_grad_ladder")

    def factorize_ladder(self, X, y, n_valid, theta_raw, linv, alpha, theta, info, ws, ws_bytes, M, n_max, d,
                         spec: HyperSpec, stream=0):
        cs = spec.to_c()
        _check(self.lib.scaml_factorize_ladder(X, y, n_valid, theta_raw, linv, alpha, theta, info, ws, ws_bytes,
                                               M, n_max, d, C.byref(cs), stream), "scaml_factorize_ladder")

    def factorize(self, X, y, n_valid, theta_raw, jitter, linv, alpha, theta, info, ws, ws_bytes, M, n_max, d,
                  spec: HyperSpec, stream=0):
        cs = spec.to_c()
        _check(self.lib.scaml_factorize(X, y, n_valid, theta_raw, jitter, linv, alpha, theta, info, ws, ws_bytes,
                                        M, n_max, d, C.byref(cs), stream), "scaml_factorize")

    def predict_weighted(self, X, n_valid, theta, linv, alpha, ybar, ystd, w, Xc, mean, var, ws, ws_bytes,
                         M, n_max, d, B, kernel, stream=0):
        _check(self.lib.scaml_predict_weighted(X, n_valid, theta, linv, alpha, ybar, ystd, w, Xc, mean, var,
                                               ws, ws_bytes, M, n_max, d, B, kernel, stream),
               "scaml_predict_weighted")

    def predict_cross_workspace_bytes(self, M: int, nA: int, nB: int, reduce: int) -> int:
        return int(self.lib.scaml_predict_cross_workspace_bytes(M, nA, nB, reduce))

    def predict_cross(self, X, n_valid, theta, linv, alpha, ybar, ystd, w, XA, XB, mean, cov, ws, ws_bytes,
                      M, n_max, d, nA, nB, kernel, reduce, stream=0):
        _check(self.lib.scaml_predict_cross(X, n_valid, theta, linv, alpha, ybar, ystd, w, XA, XB, mean, cov,
                                            ws, ws_bytes, M, n_max, d, nA, nB, kernel, reduce, stream),
               "scaml_predict_cross")


    def target_factorize(self, smeans, scovs, Xt, yt, w, theta_raw, jitter_value, mu_all, s_all, linv_t, alpha_t, theta,
                         lml, info, ws, ws_bytes, M, n_t, d, spec: HyperSpec, stream=0):
        cs = spec.to_c()
        _check(self.lib.scaml_target_factorize(smeans, scovs, Xt, yt, w, theta_raw, float(jitter_value), float(mu_all),
                                               float(s_all), linv_t, alpha_t, theta, lml, info, ws, ws_bytes, M, n_t, d,
                                               C.byref(cs), stream), "scaml_target_factorize")

    def target_posterior(self, pm, pv, cross, Xc, Xt, theta, linv_t, alpha_t, mu_all, s_all, mean, var, B, n_t, d,
                         kernel, stream=0):
        _check(self.lib.scaml_target_posterior(pm, pv, cross, Xc, Xt, theta, linv_t, alpha_t, float(mu_all),
                                               float(s_all), mean, var, B, n_t, d, kernel, stream),
               "scaml_target_posterior")

    def target_posterior_beta(self, pm, pv, cross, Xc, Xt, theta, linv_t, alpha_t, mu_all, s_all, mean, var, beta, B,
                              n_t, d, kernel, stream=0):
        _check(self.lib.scaml_target_posterior_beta(pm, pv, cross, Xc, Xt, theta, linv_t, alpha_t, float(mu_all),
                                                    float(s_all), mean, var, beta, B, n_t, d, kernel, stream),
               "scaml_target_posterior_beta")

    def posterior_grad_workspace_bytes(self, M: int, n_max: int, d: int, B: int) -> int:
        return int(self.lib.scaml_posterior_grad_workspace_bytes(M, n_max, d, B))

    def posterior_grad(self, X, n_valid, theta, alpha, ystd, w, Xc, U, Xt, A, alpha_t, beta, theta_t, s_all, dmean,
                       dvar, ws, ws_bytes, M, n_max, d, B, n_t, kernel, kernel_t, stream=0):
        _check(self.lib.scaml_posterior_grad(X, n_valid, theta, alpha, ystd, w, Xc, U, Xt, A, alpha_t, beta, theta_t,
                                             float(s_all), dmean, dvar, ws, ws_bytes, M, n_max, d, B, n_t, kernel,
                                             kernel_t, stream), "scaml_posterior_grad")

    def qblock_cov_workspace_bytes(self, M: int, B: int, q: int) -> int:
        return int(self.lib.scaml_qblock_cov_workspace_bytes(M, B, q))

    def qblock_cov(self, X, n_valid, theta, ystd, w, Xc, U, cov, ws, ws_bytes, M, n_max, d, B, q, kernel, stream=0):
        _check(self.lib.scaml_qblock_cov(X, n_valid, theta, ystd, w, Xc, U, cov, ws, ws_bytes, M, n_max, d, B, q, kernel,
                                         stream), "scaml_qblock_cov")

    def qblock_vjp_workspace_bytes(self, M: int, n_max: int, d: int, B: int, n_t: int) -> int:
        return int(self.lib.scaml_qblock_vjp_workspace_bytes(M, n_max, d, B, n_t))

    def qblock_vjp(self, X, n_valid, theta, alpha, ystd, w, Xc, U, Xt, A, alpha_t, beta, theta_t, s_all, g_mean, g_cov,
                   dX, ws, ws_bytes, M, n_max, d, B, q, n_t, kernel, kernel_t, stream=0):
        _check(self.lib.scaml_qblock_vjp(X, n_valid, theta, alpha, ystd, w, Xc, U, Xt, A, alpha_t, beta, theta_t,
                                         float(s_all), g_mean, g_cov, dX, ws, ws_bytes, M, n_max, d, B, q, n_t, kernel,
                                         kernel_t, stream), "scaml_qblock_vjp")

    def posterior_values_from_u_workspace_bytes(self, M: int, B: int, n_t: int) -> int:
        return int(self.lib.scaml_posterior_values_from_u_workspace_bytes(M, B, n_t))

    def posterior_values_from_u(self, X, n_valid, theta, alpha, ybar, ystd, w, Xc, U, Xt, A, mean, var, cross, ws,
                                ws_bytes, M, n_max, d, B, n_t, kernel, stream=0):
        _check(self.lib.scaml_posterior_values_from_u(X, n_valid, theta, alpha, ybar, ystd, w, Xc, U, Xt, A, mean, var,
                                                      cross, ws, ws_bytes, M, n_max, d, B, n_t, kernel, stream),
               "scaml_posterior_values_from_u")

    def lbfgs_step(self, state: "CLbfgsState", xt, ft, gt, lower, E, D, m, init, gtol, ftol, maxiter, max_ls, stream=0):
        _check(self.lib.scaml_lbfgs_step(C.byref(state), xt, ft, gt, lower, E, D, m, int(init), float(gtol),
                                         float(ftol), int(maxiter), int(max_ls), stream), "scaml_lbfgs_step")

    def cond_prepare(self, X, n_valid, theta, linv, Xt, A, M, n_max, d, n_t, kernel, stream=0):
        _check(self.lib.scaml_cond_prepare(X, n_valid, theta, linv, Xt, A, M, n_max, d, n_t, kernel, stream),
               "scaml_cond_prepare")

    def cond_prepare_pruned(self, X, n_valid, theta, linv, Xt, w, A, M, n_max, d, n_t, kernel, stream=0):
        _check(self.lib.scaml_cond_prepare_pruned(X, n_valid, theta, linv, Xt, w, A, M, n_max, d, n_t, kernel, stream),
               "scaml_cond_prepare_pruned")

    def cond_caches(self, X, n_valid, theta, alpha, ybar, ystd, Xt, A, mean, cov, M, n_max, d, n_t, kernel, stream=0):
        _check(self.lib.scaml_cond_caches(X, n_valid, theta, alpha, ybar, ystd, Xt, A, mean, cov, M, n_max, d, n_t, kernel,
                                          stream), "scaml_cond_caches")

    def cond_combine_task_splits(self, M: int, B: int, n_t: int) -> int:
        return int(self.lib.scaml_cond_combine_task_splits(M, B, n_t))

    def predict_conditioned_workspace_bytes(self, M, n_max, d, B, n_t) -> int:
        return int(self.lib.scaml_predict_conditioned_workspace_bytes(M, n_max, d, B, n_t))

    def predict_conditioned(self, X, n_valid, theta, linv, alpha, ybar, ystd, w, Xc, Xt, A, mean, var, cross, ws,
                            ws_bytes, M, n_max, d, B, n_t, kernel, stream=0):
        _check(self.lib.scaml_predict_conditioned(X, n_valid, theta, linv, alpha, ybar, ystd, w, Xc, Xt, A, mean, var,
                                                  cross, ws, ws_bytes, M, n_max, d, B, n_t, kernel, stream),
               "scaml_predict_conditioned")

    def target_workspace_bytes(self, n_t: int, R: int) -> int:
        return int(self.lib.scaml_target_workspace_bytes(n_t, R))

    def target_max_points(self, d: int) -> int:
        return int(self.lib.scaml_target_max_points(int(d)))

    def predict_max_points(self, d: int) -> int:
        return int(self.lib.scaml_predict_max_points(int(d)))

    def predict_cross_max_points(self, d: int) -> int:
        return int(self.lib.scaml_predict_cross_max_points(int(d)))

    def target_lml_grad(self, smeans, scovs, Xt, yt, w, theta_raw, jitter, mu_all, s_all, lml, grad_w, grad_theta,
                        info, ws, ws_bytes, M, n_t, d, R, spec: HyperSpec, w_prior=(PRIOR_GAMMA, 1.0, 1.0), stream=0):
        cs = spec.to_c()
        _check(self.lib.scaml_target_lml_grad(smeans, scovs, Xt, yt, w, theta_raw, jitter, float(mu_all), float(s_all),
                                              lml, grad_w, grad_theta, info, ws, ws_bytes, M, n_t, d, R, C.byref(cs),
                                              int(w_prior[0]), float(w_prior[1]), float(w_prior[2]), stream),
               "scaml_target_lml_grad")


    def target_lml_grad_ladder(self, smeans, scovs, Xt, yt, w, theta_raw, mu_all, s_all, lml, grad_w, grad_theta, info,
                               ws, ws_bytes, M, n_t, d, R, spec: HyperSpec, w_prior=(PRIOR_GAMMA, 1.0, 1.0), stream=0):
        cs = spec.to_c()
        _check(self.lib.scaml_target_lml_grad_ladder(smeans, scovs, Xt, yt, w, theta_raw, float(mu_all), float(s_all),
                                                     lml, grad_w, grad_theta, info, ws, ws_bytes, M, n_t, d, R,
                                                     C.byref(cs), int(w_prior[0]), float(w_prior[1]),
                                                     float(w_prior[2]), stream), "scaml_target_lml_grad_ladder")


_cuda_lib: Optional[ScamlLib] = None


def load_cuda_library() -> ScamlLib:
    """The product library. Raises ScamlError when it has not been built."""
    global _cuda_lib
    if _cuda_lib is None:
        _cuda_lib = ScamlLib(CUDA_LIB_PATH)
    return _cuda_lib


def packed_tiles(n_max: int) -> int:
    """Number of 32x32 tiles in the packed lower-triangular factor of one task."""
    nb = ((n_max + 63) // 64) * 2
    return nb * (nb + 1) // 2


def pad64(n: int) -> int:
    return ((n + 63) // 64) * 64
