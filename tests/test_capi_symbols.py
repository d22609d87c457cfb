"""The sm_100a library builds without a GPU, loads, and exports every symbol that
include/scaml_b200.h declares (no compute calls here)."""
import os
import re

from scamlgp_b200 import build
from scamlgp_b200._capi import EXPORTED_SYMBOLS, ScamlLib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_header_symbols_are_exported():
    lib = ScamlLib(build.build_cuda())
    header = open(os.path.join(ROOT, "include", "scaml_b200.h")).read()
    declared = set(re.findall(r"\b(scaml_[a-z0-9_]+)\s*\(", header))
    assert declared == set(EXPORTED_SYMBOLS), declared ^ set(EXPORTED_SYMBOLS)
    for s in declared:
        assert getattr(lib.lib, s) is not None
    assert "sm_100a" in lib.version()


def test_argument_validation_without_gpu():
    lib = ScamlLib(build.build_cuda())
    n_lim, d_lim = lib.fit_limits()
    # above n_pad = 512 the default dispatch runs the 8-warp fit kernel (3 n_pad doubles of shared memory)
    assert n_lim == 6720 and d_lim == 32
    # null pointers / bad sizes are rejected before any CUDA call
    assert lib.lib.scaml_lml_grad(None, None, None, None, None, None, None, None, None, None, 0, 1, 1, 64, 2, None, None) == -1
    assert lib.lib.scaml_kernel_matrix(None, None, None, None, 1, 64, 2, 0, None) == -1


def test_product_path_has_no_cpu_fallback():
    import pytest
    import torch

    from scamlgp_b200._capi import ScamlError
    from scamlgp_b200.engine import Engine

    if torch.cuda.is_available():
        pytest.skip("GPU present")
    with pytest.raises(ScamlError):
        Engine()
    # the product package never imports the oracle or the emulation library
    pkg = os.path.join(ROOT, "scalable-meta-learning-with-gaussian-processes_b200")
    for fn in os.listdir(pkg):
        if fn.endswith(".py"):
            src = open(os.path.join(pkg, fn)).read()
            assert "oracle" not in src.replace("# oracle", ""), fn
            assert "libscaml_emu" not in src and "build_emu" not in src, fn


def test_fit_limit_is_what_the_default_dispatch_accepts(emu_lib):
    """At the reported n_max limit scaml_lml_grad gets as far as the workspace check; one 64-row block more does not
    fit shared memory.  (Argument checks only: both calls return before any kernel runs.)"""
    import ctypes as C

    from scamlgp_b200._capi import HyperSpec

    n_lim, _ = emu_lib.fit_limits()
    assert n_lim == ScamlLib(build.build_cuda()).fit_limits()[0]
    buf = C.create_string_buffer(64)
    spec = HyperSpec.source().to_c()
    f = emu_lib.lib.scaml_lml_grad
    for n_max, rc in ((n_lim, -2), (n_lim + 64, -4), (512, -2)):
        assert f(buf, buf, None, buf, None, None, buf, buf, buf, buf, 0, 1, 1, n_max, 6, C.byref(spec), None) == rc, n_max
