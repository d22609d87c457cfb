"""Batched GP engine: torch CUDA tensors in, hand-written sm_100a kernels underneath.

This is the host side of the hot path: it owns the device-resident padded task batch,
the scratch workspaces and the jitter ladder, and calls the C ABI
(include/scaml_b200.h) with `tensor.data_ptr()` on the caller's current CUDA stream.
torch is plumbing only (memory, streams, torch.distributed); every n^2 / n^3 operation
runs in libscaml_b200.so.  There is no CPU or eager fallback: constructing an Engine
without a GPU or without the built library raises.

Reference call sites replaced:
  * the per-task loop of meta_fit_scamlgp            scamlgp/model.py:176-188
  * one LML(+grad) closure evaluation                scamlgp/utils.py:171-177,190-192
  * per-task posterior loops                         scamlgp/model.py:128-134, 280-289
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import List, Optional, Sequence, Tuple

import torch

from ._capi import (PRIOR_GAMMA, HyperSpec, NotPSDError, ScamlError, ScamlLib, load_cuda_library, pad64,
                    packed_tiles)

JITTER_LADDER = (1e-8, 1e-7, 1e-6)  # linear_operator psd_safe_cholesky (fp64), SURVEY A.5


def _ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


def standardize_rows(Y: torch.Tensor, n_valid: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
    """botorch Standardize(m=1) per task on a padded [M, n_max] batch (SURVEY A.2).

    Unbiased std; std < 1e-8 or NaN (n = 1) -> 1.  Returns (y_std [M,n_max] with zeros in
    the padding, ybar [M], ystd [M]).
    """
    M, n_max = Y.shape
    idx = torch.arange(n_max, device=Y.device).unsqueeze(0)
    mask = idx < n_valid.unsqueeze(1)
    cnt = n_valid.to(Y.dtype)
    Ym = torch.where(mask, Y, torch.zeros_like(Y))
    ybar = Ym.sum(1) / cnt
    dev = torch.where(mask, Y - ybar.unsqueeze(1), torch.zeros_like(Y))
    var = (dev * dev).sum(1) / (cnt - 1.0)
    std = torch.sqrt(var)
    std = torch.where(std >= 1e-8, std, torch.ones_like(std))  # NaN (n=1) fails the test -> 1
    return dev / std.unsqueeze(1), ybar, std


@dataclass
class SourceBatch:
    """Device-resident, padded meta-data: the input layout of the kernels.

    X [M, n_max, d], y [M, n_max] (standardised, zero padded), n_valid [M] int32,
    ybar/ystd [M] (the per-task Standardize state), Y_raw [M, n_max] (raw targets).
    """

    X: torch.Tensor
    y: torch.Tensor
    n_valid: torch.Tensor
    ybar: torch.Tensor
    ystd: torch.Tensor
    Y_raw: torch.Tensor
    uniform: bool = False  # every task has n_max points (known on the host: lets the fit skip its schedule pre-pass)

    @property
    def M(self) -> int:
        return self.X.shape[0]

    @property
    def n_max(self) -> int:
        return self.X.shape[1]

    @property
    def d(self) -> int:
        return self.X.shape[2]

    @staticmethod
    def from_padded(X: torch.Tensor, Y: torch.Tensor, n_valid: Optional[torch.Tensor] = None) -> "SourceBatch":
        X = X.to(torch.float64).contiguous()
        Y = Y.to(torch.float64).reshape(X.shape[0], X.shape[1]).contiguous()
        uniform = n_valid is None
        if n_valid is None:
            n_valid = torch.full((X.shape[0],), X.shape[1], dtype=torch.int32, device=X.device)
        n_valid = n_valid.to(device=X.device, dtype=torch.int32).contiguous()
        y, ybar, ystd = standardize_rows(Y, n_valid)
        return SourceBatch(X, y.contiguous(), n_valid, ybar.contiguous(), ystd.contiguous(), Y, uniform)

    @staticmethod
    def from_ragged(tasks: Sequence[Tuple[torch.Tensor, torch.Tensor]], device,
                    n_max: Optional[int] = None) -> "SourceBatch":
        """tasks: sequence of (X_i [n_i, d], Y_i [n_i] or [n_i, 1]) host or device tensors."""
        M = len(tasks)
        d = tasks[0][0].shape[-1]
        n_max = max([int(t[0].shape[-2]) for t in tasks] + [int(n_max or 0)])
        if all(int(t[0].shape[-2]) == n_max and t[0].dim() == 2 for t in tasks):
            # every task has n_max points (the usual meta-data layout): two stacks instead of 2 M row-block copies
            X = torch.stack([t[0].detach() for t in tasks]).to("cpu", torch.float64)
            Y = torch.stack([t[1].detach().reshape(-1) for t in tasks]).to("cpu", torch.float64)
            b = SourceBatch.from_padded(X.to(device), Y.to(device))
            return b
        X = torch.zeros(M, n_max, d, dtype=torch.float64)
        Y = torch.zeros(M, n_max, dtype=torch.float64)
        nv = torch.zeros(M, dtype=torch.int32)
        for i, (xi, yi) in enumerate(tasks):
            n = int(xi.shape[-2])
            X[i, :n] = xi.detach().to("cpu", torch.float64)
            Y[i, :n] = yi.detach().to("cpu", torch.float64).reshape(-1)
            nv[i] = n
        b = SourceBatch.from_padded(X.to(device), Y.to(device), nv.to(device))
        b.uniform = bool((nv == n_max).all())
        return b

    def slice(self, lo: int, hi: int) -> "SourceBatch":
        return SourceBatch(self.X[lo:hi].contiguous(), self.y[lo:hi].contiguous(), self.n_valid[lo:hi].contiguous(),
                           self.ybar[lo:hi].contiguous(), self.ystd[lo:hi].contiguous(), self.Y_raw[lo:hi].contiguous(),
                           self.uniform)


@dataclass
class FittedSources:
    """Prediction state of M fitted source GPs (output of Engine.factorize)."""

    batch: SourceBatch
    theta_raw: torch.Tensor  # [M, P]
    theta: torch.Tensor  # [M, P] constrained (lengthscales, outputscale, noise)
    linv: torch.Tensor  # [M, tiles, 1024] packed L^-1, column-major 32x32 tiles
    alpha: torch.Tensor  # [M, n_pad]
    info: torch.Tensor  # [M] int32
    spec: HyperSpec

    def select(self, idx: torch.Tensor) -> "FittedSources":
        """Sub-batch of the tasks `idx` (copies; used when a caller re-orders or subsets the source GPs)."""
        b = self.batch
        nb = SourceBatch(b.X[idx].contiguous(), b.y[idx].contiguous(), b.n_valid[idx].contiguous(),
                         b.ybar[idx].contiguous(), b.ystd[idx].contiguous(), b.Y_raw[idx].contiguous())
        return FittedSources(nb, self.theta_raw[idx].contiguous(), self.theta[idx].contiguous(),
                             self.linv[idx].contiguous(), self.alpha[idx].contiguous(), self.info[idx].contiguous(),
                             self.spec)

    def task_slice(self, i: int) -> "FittedSources":
        """Zero-copy view of the single task i."""
        b = self.batch
        nb = SourceBatch(b.X[i:i + 1], b.y[i:i + 1], b.n_valid[i:i + 1], b.ybar[i:i + 1], b.ystd[i:i + 1],
                         b.Y_raw[i:i + 1])
        return FittedSources(nb, self.theta_raw[i:i + 1], self.theta[i:i + 1], self.linv[i:i + 1],
                             self.alpha[i:i + 1], self.info[i:i + 1], self.spec)


class _DeviceGuardedLib:
    """View of the library that makes `device` current around every call that is made while another device is
    current: the C ABI launches on the CURRENT device (attributes, SM count, kernel launches), while the engine's
    buffers and stream live on `Engine.device`."""

    def __init__(self, lib: ScamlLib, device: torch.device):
        self._lib, self._index = lib, device.index if device.index is not None else torch.cuda.current_device()

    def __getattr__(self, name):
        fn = getattr(self._lib, name)
        if not callable(fn):
            return fn
        index = self._index

        def guarded(*args, **kwargs):
            if torch.cuda.current_device() == index:
                return fn(*args, **kwargs)
            with torch.cuda.device(index):
                return fn(*args, **kwargs)

        self.__dict__[name] = guarded  # resolved once per entry point
        return guarded


class Engine:
    """One engine per process / GPU.  All methods run on torch's current CUDA stream of `device`."""

    def __init__(self, device: Optional[torch.device] = None, lib: Optional[ScamlLib] = None):
        if not torch.cuda.is_available():
            raise ScamlError("scamlgp_b200 needs a CUDA device (B200, sm_100a); there is no CPU fallback")
        self.device = torch.device(device if device is not None else f"cuda:{torch.cuda.current_device()}")
        self.lib = _DeviceGuardedLib(lib if lib is not None else load_cuda_library(), self.device)
        self._ws: Optional[torch.Tensor] = None
        self._pws: Optional[torch.Tensor] = None
        self._cws: Optional[torch.Tensor] = None
        self._tws: Optional[torch.Tensor] = None
        self._gws: Optional[torch.Tensor] = None
        self._vws: Optional[torch.Tensor] = None
        self.launches = 0  # kernels launched through this engine (bench.py reports it)

    # ---- workspaces ------------------------------------------------------------------ #
    def _fit_ws(self, M: int, R: int, n_max: int, d: int) -> torch.Tensor:
        need = self.lib.fit_workspace_bytes(M, R, n_max, d)
        if self._ws is None or self._ws.numel() * 8 < need:
            self._ws = torch.empty((need + 7) // 8, dtype=torch.float64, device=self.device)
        return self._ws

    def _pred_ws(self, M: int, n_max: int, d: int, B: int) -> Tuple[Optional[torch.Tensor], int]:
        need = self.lib.predict_workspace_bytes(M, n_max, d, B)
        if need == 0:
            return None, 0
        if self._pws is None or self._pws.numel() * 8 < need:
            self._pws = torch.empty((need + 7) // 8, dtype=torch.float64, device=self.device)
        return self._pws, need

    def _stream(self) -> int:
        return torch.cuda.current_stream(self.device).cuda_stream

    # ---- K1 standalone ----------------------------------------------------------------- #
    def kernel_matrix(self, X: torch.Tensor, theta: torch.Tensor, kernel: int = 0,
                      n_valid: Optional[torch.Tensor] = None, out: Optional[torch.Tensor] = None) -> torch.Tensor:
        M, n_max, d = X.shape
        if out is None:
            out = torch.empty(M, n_max, n_max, dtype=torch.float64, device=self.device)
        self.lib.kernel_matrix(_ptr(X), _ptr(n_valid), _ptr(theta), _ptr(out), M, n_max, d, kernel, self._stream())
        self.launches += 1
        return out

    # ---- K1-K5 fused ------------------------------------------------------------------- #
    def lml_grad_raw(self, batch: SourceBatch, theta_raw: torch.Tensor, spec: HyperSpec,
                     jitter: Optional[torch.Tensor] = None, skip: Optional[torch.Tensor] = None,
                     out: Optional[Tuple[torch.Tensor, torch.Tensor, torch.Tensor]] = None):
        """One launch, no jitter ladder.  theta_raw [M, R, P] -> lml [M,R], grad [M,R,P], info [M,R]."""
        M, R, P = theta_raw.shape
        assert M == batch.M and P == batch.d + 2 and theta_raw.is_contiguous()
        if out is None:
            lml = torch.empty(M, R, dtype=torch.float64, device=self.device)
            grad = torch.empty(M, R, P, dtype=torch.float64, device=self.device)
            info = torch.empty(M, R, dtype=torch.int32, device=self.device)
        else:
            lml, grad, info = out
        ws = self._fit_ws(M, R, batch.n_max, batch.d)
        uniform = batch.uniform and skip is None  # full batch of equal-size tasks: no schedule pre-pass needed
        self.lib.lml_grad(_ptr(batch.X), _ptr(batch.y), None if uniform else _ptr(batch.n_valid), _ptr(theta_raw),
                          _ptr(jitter), _ptr(skip), _ptr(lml), _ptr(grad), _ptr(info), _ptr(ws), ws.numel() * 8, M, R,
                          batch.n_max, batch.d, spec, self._stream())
        self.launches += 1 if uniform else 2
        return lml, grad, info

    def lml_grad(self, batch: SourceBatch, theta_raw: torch.Tensor, spec: HyperSpec,
                 skip: Optional[torch.Tensor] = None,
                 out: Optional[Tuple[torch.Tensor, torch.Tensor, torch.Tensor]] = None):
        """LML+grad with the psd_safe_cholesky jitter ladder applied inside the kernel (`scaml_lml_grad_ladder`): no
        device -> host read of `info`, so an optimiser driving this call never synchronises with the device.

        skip [M, R] int32 (optional): non-zero rows are neither evaluated nor written (their outputs
        are NaN / info 0).  Rows that still fail at jitter 1e-6 keep info > 0 and NaN outputs -- the reference hands
        NaN to scipy in that case (SURVEY 3.2)."""
        M, R, P = theta_raw.shape
        assert M == batch.M and P == batch.d + 2 and theta_raw.is_contiguous()
        if out is not None:
            lml, grad, info = out
        elif skip is not None:
            lml = torch.full((M, R), float("nan"), dtype=torch.float64, device=self.device)
            grad = torch.full((M, R, P), float("nan"), dtype=torch.float64, device=self.device)
            info = torch.zeros(M, R, dtype=torch.int32, device=self.device)
        else:
            lml = torch.empty(M, R, dtype=torch.float64, device=self.device)
            grad = torch.empty(M, R, P, dtype=torch.float64, device=self.device)
            info = torch.empty(M, R, dtype=torch.int32, device=self.device)
        ws = self._fit_ws(M, R, batch.n_max, batch.d)
        uniform = batch.uniform and skip is None
        self.lib.lml_grad_ladder(_ptr(batch.X), _ptr(batch.y), None if uniform else _ptr(batch.n_valid),
                                 _ptr(theta_raw), _ptr(skip), _ptr(lml), _ptr(grad), _ptr(info), _ptr(ws),
                                 ws.numel() * 8, M, R, batch.n_max, batch.d, spec, self._stream())
        self.launches += 1 if uniform else 2
        return lml, grad, info

    def lml_grad_host_ladder(self, batch: SourceBatch, theta_raw: torch.Tensor, spec: HyperSpec,
                             skip: Optional[torch.Tensor] = None):
        """The same ladder driven from the host (failed rows re-run with explicit jitters, one `info` read-back per
        step); kept as the checker of the in-kernel ladder (tests)."""
        out = None
        if skip is not None:
            M, R, P = theta_raw.shape
            out = (torch.full((M, R), float("nan"), dtype=torch.float64, device=self.device),
                   torch.full((M, R, P), float("nan"), dtype=torch.float64, device=self.device),
                   torch.zeros(M, R, dtype=torch.int32, device=self.device))
        lml, grad, info = self.lml_grad_raw(batch, theta_raw, spec, skip=skip, out=out)
        if bool((info > 0).any()):
            for jit in JITTER_LADDER:
                bad = info > 0
                if not bool(bad.any()):
                    break
                skip_j = (~bad).to(torch.int32).contiguous()
                jitter = torch.where(bad, torch.full_like(lml, jit), torch.zeros_like(lml)).contiguous()
                self.lml_grad_raw(batch, theta_raw, spec, jitter=jitter, skip=skip_j, out=(lml, grad, info))
        return lml, grad, info

    # ---- K1-K3 for prediction ------------------------------------------------------------ #
    def factorize(self, batch: SourceBatch, theta_raw: torch.Tensor, spec: HyperSpec,
                  check: bool = True) -> FittedSources:
        """L^-1 (packed), alpha and the constrained parameters of every task; psd_safe_cholesky jitter ladder on the
        failed tasks.  check=True raises NotPSDError when a task is still not positive definite afterwards (the
        reference surfaces linear_operator's NotPSDError out of `posterior`); check=False returns the state with
        `info > 0` / NaN rows for the caller to inspect."""
        M, P = theta_raw.shape
        assert M == batch.M and P == batch.d + 2
        theta_raw = theta_raw.contiguous()
        n_pad = pad64(batch.n_max)
        linv = torch.zeros(M, packed_tiles(batch.n_max), 1024, dtype=torch.float64, device=self.device)
        alpha = torch.zeros(M, n_pad, dtype=torch.float64, device=self.device)
        theta = torch.empty(M, P, dtype=torch.float64, device=self.device)
        info = torch.empty(M, dtype=torch.int32, device=self.device)
        ws = self._fit_ws(M, 1, batch.n_max, batch.d)
        # psd_safe_cholesky jitter ladder inside the kernel: one launch, `info` is read once (the check below)
        self.lib.factorize_ladder(_ptr(batch.X), _ptr(batch.y), None if batch.uniform else _ptr(batch.n_valid),
                                  _ptr(theta_raw), _ptr(linv), _ptr(alpha), _ptr(theta), _ptr(info), _ptr(ws),
                                  ws.numel() * 8, M, batch.n_max, batch.d, spec, self._stream())
        self.launches += 1 if batch.uniform else 2
        if check and bool((info != 0).any()):
            # linear_operator's psd_safe_cholesky raises NotPSDError once the jitter ladder is exhausted; handing the
            # NaN factors on would poison every weighted prediction (and topk / argmax rank NaN first)
            bad = torch.nonzero(info != 0).flatten().tolist()
            raise NotPSDError(f"Matrix not positive definite after repeatedly adding jitter up to "
                              f"{JITTER_LADDER[-1]:.1e} (source tasks {bad[:16]}{'...' if len(bad) > 16 else ''})")
        return FittedSources(batch, theta_raw, theta, linv, alpha, info, spec)

    # ---- K6-K9 fused --------------------------------------------------------------------- #
    def predict_weighted(self, fs: FittedSources, w: torch.Tensor, Xc: torch.Tensor,
                         out: Optional[Tuple[torch.Tensor, torch.Tensor]] = None):
        """mean[b] = sum_m w_m mu_m(x_b), var[b] = sum_m w_m^2 var_m(x_b) (raw-Y units)."""
        b = fs.batch
        Xc = Xc.to(torch.float64).contiguous()
        B = Xc.shape[0]
        w = w.to(torch.float64).contiguous()
        if out is None:
            mean = torch.empty(B, dtype=torch.float64, device=self.device)
            var = torch.empty(B, dtype=torch.float64, device=self.device)
        else:
            mean, var = out
        pws, need = self._pred_ws(b.M, b.n_max, b.d, B)
        self.lib.predict_weighted(_ptr(b.X), _ptr(b.n_valid), _ptr(fs.theta), _ptr(fs.linv), _ptr(fs.alpha),
                                  _ptr(b.ybar), _ptr(b.ystd), _ptr(w), _ptr(Xc), _ptr(mean), _ptr(var), _ptr(pws), need,
                                  b.M, b.n_max, b.d, B, fs.spec.kernel, self._stream())
        self.launches += 2 if need else 1
        return mean, var

    def predict_cross(self, fs: FittedSources, XA: torch.Tensor, XB: Optional[torch.Tensor] = None,
                      w: Optional[torch.Tensor] = None):
        """Source posteriors at point sets A, B (B defaults to A), raw-Y units.

        w is None : per task -> mean [nA, M], cov [nA, nB, M]  (`source_means` / `source_covs`,
                    reference model.py:278-289)
        w given   : reduced  -> mean [nA] = sum_m w_m mean_m, cov [nA, nB] = sum_m w_m^2 Sigma_m
        """
        b = fs.batch
        XA = XA.to(torch.float64).contiguous()
        XB = XA if XB is None else XB.to(torch.float64).contiguous()
        nA, nB = XA.shape[0], XB.shape[0]
        reduce = 0 if w is None else 1
        if reduce:
            w = w.to(torch.float64).contiguous()
            mean = torch.empty(nA, dtype=torch.float64, device=self.device)
            cov = torch.empty(nA, nB, dtype=torch.float64, device=self.device)
        else:
            mean = torch.empty(nA, b.M, dtype=torch.float64, device=self.device)
            cov = torch.empty(nA, nB, b.M, dtype=torch.float64, device=self.device)
        need = self.lib.predict_cross_workspace_bytes(b.M, nA, nB, reduce)
        ws = None
        if need:
            if self._cws is None or self._cws.numel() * 8 < need:
                self._cws = torch.empty((need + 7) // 8, dtype=torch.float64, device=self.device)
            ws = self._cws
        self.lib.predict_cross(_ptr(b.X), _ptr(b.n_valid), _ptr(fs.theta), _ptr(fs.linv), _ptr(fs.alpha),
                               _ptr(b.ybar), _ptr(b.ystd), _ptr(w), _ptr(XA), _ptr(XB), _ptr(mean), _ptr(cov),
                               _ptr(ws), need, b.M, b.n_max, b.d, nA, nB, fs.spec.kernel, reduce, self._stream())
        self.launches += 2 if need else 1
        return mean, cov

    # ---- conditioning at scale (cross-covariance fused into the prediction kernel) ------- #
    def predict_supported(self, fs: FittedSources) -> bool:
        """The prediction kernel (`predict_weighted`, `predict_conditioned`) accepts the tasks' (n_max, d)."""
        return fs.batch.n_max <= self.lib.predict_max_points(fs.batch.d)

    def cross_supported(self, fs: FittedSources) -> bool:
        """The stand-alone cross-covariance kernel (`predict_cross`) accepts the tasks' (n_max, d)."""
        return fs.batch.n_max <= self.lib.predict_cross_max_points(fs.batch.d)

    def cond_supported(self, fs: FittedSources, n_t: int) -> bool:
        """The A_m-based conditioning kernels cover what the prediction kernel covers (n_max <= 512, and less for
        d > 10: `predict_supported`), d <= 16 and n_t <= 128."""
        b = fs.batch
        return 0 < n_t <= 128 and b.n_max <= 512 and b.d <= 16 and self.predict_supported(fs)

    def cond_prepare(self, fs: FittedSources, Xt: torch.Tensor, w: Optional[torch.Tensor] = None) -> torch.Tensor:
        """A [M, n_pad, n_tp] with A_m = K_m^-1 K_m(X_m, X_t): once per set of target inputs.  With w given, tasks
        with w == 0 (pruned) are skipped and their slices stay zero."""
        b = fs.batch
        Xt = Xt.to(torch.float64).contiguous()
        n_t = Xt.shape[0]
        n_tp = ((n_t + 7) // 8) * 8
        A = torch.zeros(b.M, pad64(b.n_max), n_tp, dtype=torch.float64, device=self.device)
        if w is not None:
            w = w.to(torch.float64).contiguous()
            self.lib.cond_prepare_pruned(_ptr(b.X), _ptr(b.n_valid), _ptr(fs.theta), _ptr(fs.linv), _ptr(Xt), _ptr(w),
                                         _ptr(A), b.M, b.n_max, b.d, n_t, fs.spec.kernel, self._stream())
        else:
            self.lib.cond_prepare(_ptr(b.X), _ptr(b.n_valid), _ptr(fs.theta), _ptr(fs.linv), _ptr(Xt), _ptr(A), b.M,
                                  b.n_max, b.d, n_t, fs.spec.kernel, self._stream())
        self.launches += 1
        return A

    def cond_caches(self, fs: FittedSources, Xt: torch.Tensor, A: torch.Tensor):
        """`source_means` [n_t, M] / `source_covs` [n_t, n_t, M] (reference model.py:278-289) from A."""
        b = fs.batch
        Xt = Xt.to(torch.float64).contiguous()
        n_t = Xt.shape[0]
        mean = torch.empty(n_t, b.M, dtype=torch.float64, device=self.device)
        cov = torch.empty(n_t, n_t, b.M, dtype=torch.float64, device=self.device)
        self.lib.cond_caches(_ptr(b.X), _ptr(b.n_valid), _ptr(fs.theta), _ptr(fs.alpha), _ptr(b.ybar), _ptr(b.ystd),
                             _ptr(Xt), _ptr(A), _ptr(mean), _ptr(cov), b.M, b.n_max, b.d, n_t, fs.spec.kernel,
                             self._stream())
        self.launches += 1
        return mean, cov

    def predict_conditioned(self, fs: FittedSources, w: torch.Tensor, Xc: torch.Tensor, Xt: torch.Tensor,
                            A: torch.Tensor):
        """Weighted prior mean [B], variance [B] and cross-covariance with the target inputs [B, n_t] (raw-Y units)."""
        b = fs.batch
        Xc = Xc.to(torch.float64).contiguous()
        Xt = Xt.to(torch.float64).contiguous()
        w = w.to(torch.float64).contiguous()
        B, n_t = Xc.shape[0], Xt.shape[0]
        mean = torch.empty(B, dtype=torch.float64, device=self.device)
        var = torch.empty(B, dtype=torch.float64, device=self.device)
        cross = torch.empty(B, n_t, dtype=torch.float64, device=self.device)
        need = self.lib.predict_conditioned_workspace_bytes(b.M, b.n_max, b.d, B, n_t)
        if self._pws is None or self._pws.numel() * 8 < need:
            self._pws = torch.empty((need + 7) // 8, dtype=torch.float64, device=self.device)
        self.lib.predict_conditioned(_ptr(b.X), _ptr(b.n_valid), _ptr(fs.theta), _ptr(fs.linv), _ptr(fs.alpha),
                                     _ptr(b.ybar), _ptr(b.ystd), _ptr(w), _ptr(Xc), _ptr(Xt), _ptr(A), _ptr(mean),
                                     _ptr(var), _ptr(cross), _ptr(self._pws), need, b.M, b.n_max, b.d, B, n_t,
                                     fs.spec.kernel, self._stream())
        self.launches += 3 + (self.lib.cond_combine_task_splits(b.M, B, n_t) > 1)
        return mean, var, cross

    # ---- a7: target objective ------------------------------------------------------------ #
    def target_lml_grad(self, source_means: torch.Tensor, source_covs: torch.Tensor, Xt: torch.Tensor,
                        yt: torch.Tensor, w: torch.Tensor, theta_raw: torch.Tensor, mu_all: float, s_all: float,
                        spec: HyperSpec, w_prior=(PRIOR_GAMMA, 1.0, 1.0), jitter: Optional[torch.Tensor] = None):
        """ScaML-GP target objective (training branch) for R rows: w [R, M], theta_raw [R, P].

        source_means [n_t, M], source_covs [n_t, n_t, M] are the per-task caches of `predict_cross`
        (reference model.py:278-289), yt the targets standardised with the frozen all-data transform.
        Returns lml [R], grad_w [R, M], grad_theta [R, P], info [R] (no jitter ladder: see
        `target_lml_grad_safe`)."""
        R, M = w.shape
        nt, d = Xt.shape
        P = d + 2
        assert source_means.shape == (nt, M) and source_covs.shape == (nt, nt, M) and theta_raw.shape == (R, P)
        for t in (source_means, source_covs, Xt, yt, w, theta_raw):
            assert t.is_contiguous() and t.dtype == torch.float64
        lml = torch.empty(R, dtype=torch.float64, device=self.device)
        gw = torch.empty(R, M, dtype=torch.float64, device=self.device)
        gt = torch.empty(R, P, dtype=torch.float64, device=self.device)
        info = torch.empty(R, dtype=torch.int32, device=self.device)
        need = self.lib.target_workspace_bytes(nt, R)
        if self._tws is None or self._tws.numel() * 8 < need:
            self._tws = torch.empty((need + 7) // 8, dtype=torch.float64, device=self.device)
        self.lib.target_lml_grad(_ptr(source_means), _ptr(source_covs), _ptr(Xt), _ptr(yt), _ptr(w), _ptr(theta_raw),
                                 _ptr(jitter), mu_all, s_all, _ptr(lml), _ptr(gw), _ptr(gt), _ptr(info),
                                 _ptr(self._tws), need, M, nt, d, R, spec, w_prior, self._stream())
        self.launches += 3
        return lml, gw, gt, info

    def target_lml_grad_safe(self, source_means, source_covs, Xt, yt, w, theta_raw, mu_all, s_all, spec,
                             w_prior=(PRIOR_GAMMA, 1.0, 1.0)):
        """target_lml_grad with the psd_safe_cholesky jitter ladder applied inside the kernel on failed rows: no
        device -> host read between the rounds of the L-BFGS driver (the host-driven ladder cost one
        synchronisation per round: 0.5 ms of a 0.9 ms round at 4096 tasks)."""
        R, M = w.shape
        nt, d = Xt.shape
        P = d + 2
        assert source_means.shape == (nt, M) and source_covs.shape == (nt, nt, M) and theta_raw.shape == (R, P)
        for t in (source_means, source_covs, Xt, yt, w, theta_raw):
            assert t.is_contiguous() and t.dtype == torch.float64
        lml = torch.empty(R, dtype=torch.float64, device=self.device)
        gw = torch.empty(R, M, dtype=torch.float64, device=self.device)
        gt = torch.empty(R, P, dtype=torch.float64, device=self.device)
        info = torch.empty(R, dtype=torch.int32, device=self.device)
        need = self.lib.target_workspace_bytes(nt, R)
        if self._tws is None or self._tws.numel() * 8 < need:
            self._tws = torch.empty((need + 7) // 8, dtype=torch.float64, device=self.device)
        self.lib.target_lml_grad_ladder(_ptr(source_means), _ptr(source_covs), _ptr(Xt), _ptr(yt), _ptr(w),
                                        _ptr(theta_raw), mu_all, s_all, _ptr(lml), _ptr(gw), _ptr(gt), _ptr(info),
                                        _ptr(self._tws), need, M, nt, d, R, spec, w_prior, self._stream())
        self.launches += 3
        return lml, gw, gt, info

    def target_lml_grad_host_ladder(self, source_means, source_covs, Xt, yt, w, theta_raw, mu_all, s_all, spec,
                                    w_prior=(PRIOR_GAMMA, 1.0, 1.0)):
        """The same ladder driven from the host (re-runs the failed rows with explicit jitters); kept as the checker
        of the in-kernel ladder (tests)."""
        out = self.target_lml_grad(source_means, source_covs, Xt, yt, w, theta_raw, mu_all, s_all, spec, w_prior)
        lml, gw, gt, info = out
        for jit in JITTER_LADDER:
            bad = info > 0
            if not bool(bad.any()):
                break
            idx = bad.nonzero().flatten()
            jitter = torch.full((idx.numel(),), jit, dtype=torch.float64, device=self.device)
            l2, gw2, gt2, i2 = self.target_lml_grad(source_means, source_covs, Xt, yt, w[idx].contiguous(),
                                                    theta_raw[idx].contiguous(), mu_all, s_all, spec, w_prior, jitter)
            lml[idx], gw[idx], gt[idx], info[idx] = l2, gw2, gt2, i2
        return lml, gw, gt, info

    # ---- target prediction state + conditioning ---------------------------------------- #
    def target_factorize(self, source_means, source_covs, Xt, yt, w, theta_raw, mu_all, s_all, spec,
                         check: bool = True) -> "TargetState":
        """L_t^-1, alpha_t and constrained kernel parameters of the target GP at (w [M], theta_raw [P]);
        psd_safe_cholesky jitter ladder on failure, NotPSDError when it is exhausted (check=True)."""
        nt, d = Xt.shape
        M, P = w.numel(), d + 2
        linv = torch.empty(nt, nt, dtype=torch.float64, device=self.device)
        alpha = torch.empty(nt, dtype=torch.float64, device=self.device)
        theta = torch.empty(P, dtype=torch.float64, device=self.device)
        lml = torch.empty(1, dtype=torch.float64, device=self.device)
        info = torch.empty(1, dtype=torch.int32, device=self.device)
        need = self.lib.target_workspace_bytes(nt, 1) + 8 * (d + 3)
        if self._tws is None or self._tws.numel() * 8 < need:
            self._tws = torch.empty((need + 7) // 8, dtype=torch.float64, device=self.device)
        for jit in (0.0,) + JITTER_LADDER:
            self.lib.target_factorize(_ptr(source_means), _ptr(source_covs), _ptr(Xt), _ptr(yt), _ptr(w),
                                      _ptr(theta_raw), jit, mu_all, s_all, _ptr(linv), _ptr(alpha), _ptr(theta),
                                      _ptr(lml), _ptr(info), _ptr(self._tws), need, M, nt, d, spec, self._stream())
            self.launches += 2
            if int(info.item()) == 0:
                break
        if check and int(info.item()) != 0:
            raise NotPSDError(f"Target covariance not positive definite after repeatedly adding jitter up to "
                              f"{JITTER_LADDER[-1]:.1e} (first failing pivot {int(info.item())})")
        return TargetState(Xt, linv, alpha, theta, float(mu_all), float(s_all), int(info.item()), float(lml.item()),
                           spec.kernel)

    def target_posterior(self, ts: "TargetState", prior_mean, prior_var, cross, Xc):
        """Condition the weighted source prior at candidates Xc [B, d] on the target data (q = 1)."""
        B, d = Xc.shape
        nt = ts.Xt.shape[0]
        mean = torch.empty(B, dtype=torch.float64, device=self.device)
        var = torch.empty(B, dtype=torch.float64, device=self.device)
        self.lib.target_posterior(_ptr(prior_mean), _ptr(prior_var), _ptr(cross), _ptr(Xc), _ptr(ts.Xt), _ptr(ts.theta),
                                  _ptr(ts.linv), _ptr(ts.alpha), ts.mu_all, ts.s_all, _ptr(mean), _ptr(var), B, nt, d,
                                  ts.kernel, self._stream())
        self.launches += 1
        return mean, var


    # ---- f3: analytic candidate gradients (reference: autograd through ScaMLGP.forward, model.py:364-375) ---- #
    def target_posterior_beta(self, ts: "TargetState", prior_mean, prior_var, cross, Xc):
        """`target_posterior` plus beta [B, n_tp] = K_t^-1 k_s(x_b), the vector the variance gradient contracts with."""
        B, d = Xc.shape
        nt = ts.Xt.shape[0]
        n_tp = ((nt + 7) // 8) * 8
        mean = torch.empty(B, dtype=torch.float64, device=self.device)
        var = torch.empty(B, dtype=torch.float64, device=self.device)
        beta = torch.empty(B, n_tp, dtype=torch.float64, device=self.device)
        self.lib.target_posterior_beta(_ptr(prior_mean), _ptr(prior_var), _ptr(cross), _ptr(Xc), _ptr(ts.Xt),
                                       _ptr(ts.theta), _ptr(ts.linv), _ptr(ts.alpha), ts.mu_all, ts.s_all, _ptr(mean),
                                       _ptr(var), _ptr(beta), B, nt, d, ts.kernel, self._stream())
        self.launches += 1
        return mean, var, beta

    def values_from_u(self, fs: FittedSources, w: torch.Tensor, Xc: torch.Tensor, U: torch.Tensor,
                      Xt: Optional[torch.Tensor] = None, A: Optional[torch.Tensor] = None):
        """Weighted prior mean [B], variance [B] (and cross-covariance [B, n_t] when Xt / A are given) from
        U = cond_prepare(fs, Xc): the quantities of `predict_conditioned` without a second pass over the factors."""
        b = fs.batch
        B, d = Xc.shape
        n_t = 0 if Xt is None else Xt.shape[0]
        w = w.to(torch.float64).contiguous()
        mean = torch.empty(B, dtype=torch.float64, device=self.device)
        var = torch.empty(B, dtype=torch.float64, device=self.device)
        cross = torch.empty(B, n_t, dtype=torch.float64, device=self.device) if n_t > 0 else None
        need = self.lib.posterior_values_from_u_workspace_bytes(b.M, B, n_t)
        if self._vws is None or self._vws.numel() * 8 < need:
            self._vws = torch.empty((need + 7) // 8, dtype=torch.float64, device=self.device)
        self.lib.posterior_values_from_u(_ptr(b.X), _ptr(b.n_valid), _ptr(fs.theta), _ptr(fs.alpha), _ptr(b.ybar),
                                         _ptr(b.ystd), _ptr(w), _ptr(Xc), _ptr(U), _ptr(Xt), _ptr(A), _ptr(mean), _ptr(var),
                                         _ptr(cross), _ptr(self._vws), need, b.M, b.n_max, d, B, n_t, fs.spec.kernel,
                                         self._stream())
        self.launches += (3 + (self.lib.cond_combine_task_splits(b.M, B, n_t) > 1)) if n_t > 0 else 2
        return mean, var, cross

    def prior_values(self, fs: FittedSources, w: torch.Tensor, Xc: torch.Tensor, U: torch.Tensor,
                     Xt: Optional[torch.Tensor] = None, A: Optional[torch.Tensor] = None):
        """Value half of a value-and-gradient evaluation: from U when its register-light variants apply (n_t <= 64,
        0.9 ms vs 1.4 ms at 4096 tasks x 64 candidates), else the fused prediction kernel (measured faster at
        n_t = 80: 3.9 ms vs 5.0 ms at 128 candidates; profiles/r1_grad_path_v5_*.txt)."""
        n_t = 0 if Xt is None else Xt.shape[0]
        if n_t <= 64:
            return self.values_from_u(fs, w, Xc, U, Xt, A)
        return self.predict_conditioned(fs, w, Xc, Xt, A)

    def posterior_grad(self, fs: FittedSources, w: torch.Tensor, Xc: torch.Tensor, U: torch.Tensor,
                       ts: Optional["TargetState"] = None, A: Optional[torch.Tensor] = None,
                       beta: Optional[torch.Tensor] = None, target_terms: bool = True):
        """d mean / d x and d var / d x [B, d] of the (un-standardised) ScaML-GP posterior at B <= 128 candidates.

        U = cond_prepare(fs, Xc) (K_m^-1 k*_m of every task); with target data: ts / A / beta from
        `target_factorize`, `cond_prepare(fs, X_t)` and `target_posterior_beta`; without: the weighted prior.
        With target data U is consumed (overwritten by U - A beta).  target_terms=False leaves out the target-kernel
        terms (task-sharded partial sums: only one rank may add them)."""
        b = fs.batch
        B, d = Xc.shape
        n_t = 0 if ts is None else ts.Xt.shape[0]
        w = w.to(torch.float64).contiguous()
        dmean = torch.empty(B, d, dtype=torch.float64, device=self.device)
        dvar = torch.empty(B, d, dtype=torch.float64, device=self.device)
        need = self.lib.posterior_grad_workspace_bytes(b.M, b.n_max, d, B)
        if self._gws is None or self._gws.numel() * 8 < need:
            self._gws = torch.empty((need + 7) // 8, dtype=torch.float64, device=self.device)
        if n_t > 0:
            self.lib.posterior_grad(_ptr(b.X), _ptr(b.n_valid), _ptr(fs.theta), _ptr(fs.alpha), _ptr(b.ystd), _ptr(w),
                                    _ptr(Xc), _ptr(U), _ptr(ts.Xt), _ptr(A), _ptr(ts.alpha), _ptr(beta), _ptr(ts.theta),
                                    ts.s_all, _ptr(dmean), _ptr(dvar), _ptr(self._gws), need, b.M, b.n_max, d, B, n_t,
                                    fs.spec.kernel, ts.kernel if target_terms else -1, self._stream())
        else:
            self.lib.posterior_grad(_ptr(b.X), _ptr(b.n_valid), _ptr(fs.theta), _ptr(fs.alpha), _ptr(b.ystd), _ptr(w),
                                    _ptr(Xc), _ptr(U), None, None, None, None, None, 1.0, _ptr(dmean), _ptr(dvar),
                                    _ptr(self._gws), need, b.M, b.n_max, d, B, 0, fs.spec.kernel, 0, self._stream())
        self.launches += 2
        return dmean, dvar

    # ---- joint q-point blocks (batch acquisition: autograd through ScaMLGP.forward with q > 1) ---------------- #
    def _grad_ws(self, need: int) -> torch.Tensor:
        if self._gws is None or self._gws.numel() * 8 < need:
            self._gws = torch.empty((need + 7) // 8, dtype=torch.float64, device=self.device)
        return self._gws

    def qblock_cov(self, fs: FittedSources, w: torch.Tensor, Xc: torch.Tensor, U: torch.Tensor, q: int) -> torch.Tensor:
        """Weighted prior block [B / q, q, q] of every block of q consecutive points of Xc [B, d] (raw-Y units), from
        U = cond_prepare(fs, Xc, w); U is left unchanged.  B <= 128, q <= 16."""
        b = fs.batch
        B, d = Xc.shape
        w = w.to(torch.float64).contiguous()
        cov = torch.empty(B // q, q, q, dtype=torch.float64, device=self.device)
        need = self.lib.qblock_cov_workspace_bytes(b.M, B, q)
        ws = self._grad_ws(need)
        self.lib.qblock_cov(_ptr(b.X), _ptr(b.n_valid), _ptr(fs.theta), _ptr(b.ystd), _ptr(w), _ptr(Xc), _ptr(U), _ptr(cov),
                            _ptr(ws), need, b.M, b.n_max, d, B, q, fs.spec.kernel, self._stream())
        self.launches += 2
        return cov

    def qblock_vjp(self, fs: FittedSources, w: torch.Tensor, Xc: torch.Tensor, U: torch.Tensor, q: int,
                   g_mean: torch.Tensor, g_cov: torch.Tensor, theta_t: torch.Tensor, kernel_t: int,
                   ts: Optional["TargetState"] = None, A: Optional[torch.Tensor] = None,
                   beta: Optional[torch.Tensor] = None) -> torch.Tensor:
        """dX [B, d] = d a / d Xc for the upstream gradients g_mean [B] = d a / d mean and g_cov [B / q, q, q] =
        d a / d Sigma of the joint block posterior (un-standardised).  Inputs as for `posterior_grad`, plus the
        constrained target-kernel parameters theta_t [P] (its kernel enters every block).  U is consumed."""
        b = fs.batch
        B, d = Xc.shape
        n_t = 0 if ts is None else ts.Xt.shape[0]
        w = w.to(torch.float64).contiguous()
        g_mean = g_mean.to(self.device, torch.float64).contiguous()
        g_cov = g_cov.to(self.device, torch.float64).contiguous()
        dX = torch.empty(B, d, dtype=torch.float64, device=self.device)
        need = self.lib.qblock_vjp_workspace_bytes(b.M, b.n_max, d, B, n_t)
        ws = self._grad_ws(need)
        self.lib.qblock_vjp(_ptr(b.X), _ptr(b.n_valid), _ptr(fs.theta), _ptr(fs.alpha), _ptr(b.ystd), _ptr(w), _ptr(Xc),
                            _ptr(U), _ptr(ts.Xt) if n_t else None, _ptr(A), _ptr(ts.alpha) if n_t else None, _ptr(beta),
                            _ptr(theta_t), ts.s_all if n_t else 1.0, _ptr(g_mean), _ptr(g_cov), _ptr(dX), _ptr(ws), need,
                            b.M, b.n_max, d, B, q, n_t, fs.spec.kernel, kernel_t, self._stream())
        self.launches += 6 if n_t else 4  # fold (+ beta fold, mix), contract, finish, direct terms
        return dX


@dataclass
class TargetState:
    """Prediction state of the fitted target GP (output of Engine.target_factorize)."""

    Xt: torch.Tensor  # [n_t, d]
    linv: torch.Tensor  # [n_t, n_t] row-major L_t^-1
    alpha: torch.Tensor  # [n_t]
    theta: torch.Tensor  # [P] constrained
    mu_all: float
    s_all: float
    info: int
    lml: float
    kernel: int


_default_engine: Optional[Engine] = None


def default_engine() -> Engine:
    global _default_engine
    if _default_engine is None:
        _default_engine = Engine()
    return _default_engine
