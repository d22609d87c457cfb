"""In-tree builds of the native code (explicit nvcc / g++ command lines, no JIT cache).

build_cuda(): csrc/*.cu -> csrc/libscaml_b200.so for sm_100a (the product library).
The CPU logic-emulation build of the same kernel sources (-DSCAML_EMU, g++) is test infrastructure and lives
in tests/emu_build.py; nothing in this package builds or loads it.
"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
CUDA_LIB = os.path.join(CSRC, "libscaml_b200.so")

CUDA_SOURCES = ["scaml_capi.cu", "scaml_microbench.cu"]
HEADERS = ["scaml_device.cuh", "scaml_fit.cuh", "scaml_fit8.cuh", "scaml_kmat.cuh", "scaml_predict.cuh", "scaml_cond.cuh", "scaml_cross.cuh", "scaml_target.cuh", "scaml_lbfgs.cuh", "scaml_grad.cuh", "scaml_gradval.cuh", "scaml_qblock.cuh",
           os.path.join("emu", "cuda_emu.h"), os.path.join("..", "..", "include", "scaml_b200.h")]

NVCC_COMPILE_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-lineinfo", "-O3", "-std=c++17",
    "-Xcompiler", "-fPIC",
]
NVCC_LINK_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-shared",
    # link the CUDA runtime dynamically (libcudart.so.12: the one torch has already loaded into the process, else the
    # toolkit's via rpath) instead of embedding a static copy in the artefact
    "-cudart", "shared", "-Xlinker", "-rpath=/usr/local/cuda/lib64",
]


def _newer(target: str, deps) -> bool:
    if not os.path.exists(target):
        return False
    t = os.path.getmtime(target)
    return all(os.path.getmtime(d) <= t for d in deps if os.path.exists(d))


def _nvcc() -> str:
    for cand in (shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found")


PARTS = (0, 1, 2, 3)  # scaml_capi.cu is compiled once per part (see its header), in parallel


def _compile_parts(extra, out: str, verbose: bool = False, parts=PARTS) -> None:
    """nvcc -c per part (parallel processes) + scaml_microbench.cu, then one link.  parts=(None,): one translation unit
    (SCAML_PART undefined)."""
    from concurrent.futures import ThreadPoolExecutor

    nvcc = _nvcc()
    tag = os.path.splitext(os.path.basename(out))[0]
    objdir = os.path.join(CSRC, "build")
    os.makedirs(objdir, exist_ok=True)
    jobs = []
    for part in parts:
        obj = os.path.join(objdir, f"{tag}_part{part}.o")
        jobs.append((obj, [nvcc] + NVCC_COMPILE_FLAGS + extra + (["-Xptxas", "-v"] if verbose else []) +
                     ([f"-DSCAML_PART={part}"] if part is not None else []) + ["-c", "-o", obj, "scaml_capi.cu"]))
    obj = os.path.join(objdir, f"{tag}_microbench.o")
    jobs.append((obj, [nvcc] + NVCC_COMPILE_FLAGS + extra + ["-c", "-o", obj, "scaml_microbench.cu"]))

    def run(job):
        res = subprocess.run(job[1], cwd=CSRC, capture_output=True, text=True)
        return job, res

    with ThreadPoolExecutor(max_workers=len(jobs)) as ex:
        results = list(ex.map(run, jobs))
    for (obj, cmd), res in results:
        if verbose:
            sys.stderr.write(res.stderr)
        if res.returncode != 0:
            raise RuntimeError("nvcc failed:\n" + " ".join(cmd) + "\n" + res.stdout + res.stderr)
    cmd = [nvcc] + NVCC_LINK_FLAGS + ["-o", out] + [j[0] for j in jobs]
    res = subprocess.run(cmd, cwd=CSRC, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("nvcc link failed:\n" + " ".join(cmd) + "\n" + res.stdout + res.stderr)


def build_cuda(force: bool = False, verbose: bool = False) -> str:
    deps = [os.path.join(CSRC, s) for s in CUDA_SOURCES + HEADERS]
    if not force and _newer(CUDA_LIB, deps):
        return CUDA_LIB
    _compile_parts([], CUDA_LIB, verbose)
    return CUDA_LIB


def build_prof(force: bool = False) -> str:
    """Diagnostics variant with per-phase clock64 counters (-DSCAML_PROF); not used by the product path."""
    out = os.path.join(CSRC, "libscaml_b200_prof.so")
    deps = [os.path.join(CSRC, s) for s in CUDA_SOURCES + HEADERS]
    if not force and _newer(out, deps):
        return out
    _compile_parts(["-DSCAML_PROF"], out)
    return out


def build_ablate(force: bool = False) -> str:
    """Timing-only ablation variant (-DSCAML_ABLATE, wrong results by design); experiments only."""
    out = os.path.join(CSRC, "libscaml_b200_abl.so")
    deps = [os.path.join(CSRC, s) for s in CUDA_SOURCES + HEADERS]
    if not force and _newer(out, deps):
        return out
    # one translation unit: the ablation switch is a __device__ variable, and with it nvcc gives the file-scope helpers
    # of scaml_capi.cu external linkage under a name derived from the FILE name -- the four parts would collide
    _compile_parts(["-DSCAML_ABLATE"], out, parts=(None,))
    return out


def build_variant(tag: str, defines, force: bool = False) -> str:
    """A/B experiment builds (e.g. build_variant("nosplit", ["-DSCAML_FIT_NOSPLIT"])) -> csrc/libscaml_b200_<tag>.so;
    experiments only, never loaded by the package."""
    out = os.path.join(CSRC, f"libscaml_b200_{tag}.so")
    deps = [os.path.join(CSRC, s) for s in CUDA_SOURCES + HEADERS]
    if not force and _newer(out, deps):
        return out
    _compile_parts(list(defines), out)
    return out


if __name__ == "__main__":
    print(build_cuda(force="--force" in sys.argv, verbose="-v" in sys.argv))
