"""In-tree build of the native code (no JIT cache: the built .so files travel with the tree).

  lib/libodecol.so   pure C ABI (include/odecol.h), hand-written CUDA for sm_100a, built with nvcc
  _odecol_ext*.so    PyTorch C++ extension: tensor checks + current stream, then straight into the C ABI

Run ``python ode-column_b200/build.py`` or call ``build()``; both are no-ops when outputs are newer than sources.
"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys
import sysconfig
from pathlib import Path

PKG = Path(__file__).resolve().parent
ROOT = PKG.parent
CSRC = PKG / "csrc"
LIBDIR = PKG / "lib"
LIB = LIBDIR / "libodecol.so"
# variant builds (A/B experiments): ODECOL_LIB_OUT=path/to/variant.so with ODECOL_NVCC_EXTRA=... compiles into its own object
# directory and leaves the shipped library, its objects and the extension alone
VARIANT_OUT = os.environ.get("ODECOL_LIB_OUT")
EXT = PKG / ("_odecol_ext" + (sysconfig.get_config_var("EXT_SUFFIX") or ".so"))

CUDA_SOURCES = ["abi.cu", "small_kernels.cu", "stage_em.cu", "stage_tc.cu", "stage_tc_bwd.cu", "stage_tc_persist.cu", "tiny_tc.cu", "ww_kernel.cu", "readout_kernels.cu"]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
    "--expt-relaxed-constexpr", "-Xcompiler", "-fPIC",
]


# experiments: extra nvcc flags (e.g. ODECOL_NVCC_EXTRA="-DODECOL_TC_STAGES=4") for an A/B rebuild on the GPU box
NVCC_FLAGS += os.environ.get("ODECOL_NVCC_EXTRA", "").split()


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found")


def _stale(out: Path, deps) -> bool:
    if not out.exists():
        return True
    t = out.stat().st_mtime
    return any(Path(d).stat().st_mtime > t for d in deps)


def _run(cmd, verbose):
    if verbose:
        print("+", " ".join(map(str, cmd)), flush=True)
    res = subprocess.run(list(map(str, cmd)), capture_output=True, text=True)
    if res.returncode != 0:
        sys.stderr.write(res.stdout + res.stderr)
        raise RuntimeError(f"build step failed: {cmd[0]}")
    return res.stdout + res.stderr


def build_lib(force: bool = False, verbose: bool = False) -> Path:
    srcs = [CSRC / s for s in CUDA_SOURCES if (CSRC / s).exists()]
    deps = srcs + list(CSRC.glob("*.cuh")) + list(CSRC.glob("*.h")) + [ROOT / "include" / "odecol.h"]
    target = Path(VARIANT_OUT).resolve() if VARIANT_OUT else LIB
    force = force or bool(VARIANT_OUT)
    LIBDIR.mkdir(exist_ok=True)
    objs = []
    procs = []
    objdir = PKG / ("build_variant" if VARIANT_OUT else "build")
    objdir.mkdir(exist_ok=True)
    for s in srcs:                                       # compile translation units in parallel
        o = objdir / (s.stem + ".o")
        objs.append(o)
        if force or _stale(o, deps):
            cmd = [_nvcc(), *NVCC_FLAGS, "-c", s, "-o", o]
            if verbose:
                print("+", " ".join(map(str, cmd)), flush=True)
            procs.append((cmd, subprocess.Popen(list(map(str, cmd)), stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    for cmd, pr in procs:
        log, _ = pr.communicate()
        if pr.returncode != 0:
            sys.stderr.write(log)
            raise RuntimeError(f"nvcc failed on {cmd[-3]}")
    if procs or _stale(target, objs):
        _run([_nvcc(), "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", target, *objs, "-lcuda"], verbose)
    return target


def build_ext(force: bool = False, verbose: bool = False) -> Path:
    src = CSRC / "torch_ext.cpp"
    deps = [src, ROOT / "include" / "odecol.h", LIB]
    if force or _stale(EXT, deps):
        import torch
        from torch.utils import cpp_extension as ce
        inc = []
        for d in ce.include_paths(device_type="cuda") if "device_type" in ce.include_paths.__code__.co_varnames else ce.include_paths(cuda=True):
            inc += ["-isystem", d]
        inc += ["-isystem", sysconfig.get_paths()["include"], "-isystem", "/usr/local/cuda/include"]
        torch_lib = Path(torch.__file__).parent / "lib"
        abi = int(torch._C._GLIBCXX_USE_CXX11_ABI)
        cmd = [
            os.environ.get("CXX", "g++"), "-O2", "-std=c++17", "-fPIC", "-shared", "-fvisibility=hidden",
            f"-D_GLIBCXX_USE_CXX11_ABI={abi}", "-DTORCH_EXTENSION_NAME=_odecol_ext", "-DTORCH_API_INCLUDE_EXTENSION_H",
            *inc, src, "-o", EXT,
            f"-L{LIBDIR}", "-lodecol", "-Wl,-rpath,$ORIGIN/lib",
            f"-L{torch_lib}", "-ltorch", "-ltorch_cpu", "-ltorch_cuda", "-ltorch_python", "-lc10", "-lc10_cuda",
            f"-Wl,-rpath,{torch_lib}",
        ]
        _run(cmd, verbose)
    return EXT


def build(force: bool = False, verbose: bool = False):
    if VARIANT_OUT:
        return build_lib(force, verbose), EXT
    build_lib(force, verbose)
    build_ext(force, verbose)
    return LIB, EXT


if __name__ == "__main__":
    build(force="--force" in sys.argv, verbose=True)
    print("built", LIB, EXT)
