#!/usr/bin/env python
"""Recipe: compile the REFERENCE's own CUDA backends for sm_100a into ``oracle/_ref/``
(SURVEY.md 8c "B3": the comparator `north_star` calls "the reference's own torchsparse build").

MEASUREMENT / TEST INFRASTRUCTURE ONLY (the "reference arm") - the product (openpcseg_b200/) never imports it.

What it does (build container only; nvcc cross-compiles without a GPU)
  * unpacks ``/root/reference/package/{torchsparse,sparsehash,range_lib}.zip`` into a
    throw-away directory under ``$TMPDIR`` (never into this repo);
  * applies the two-pattern source patch torch >= 2 needs, to the TEMP copy only:
      ``X.type()`` -> ``X.scalar_type()`` inside ``AT_DISPATCH_FLOATING_TYPES_AND_HALF``
      (convolution_cuda.cu:138,153,238,248,266; devoxelize_cuda.cu:70,90; voxelize_cuda.cu:54,73)
      ``<THC/THCAtomics.cuh>`` -> ``<ATen/cuda/Atomic.cuh>`` (voxelize_cuda.cu:5, devoxelize_cuda.cu:6)
    nothing else of the reference is touched: kernels, launch shapes, host loops, cuBLAS calls
    are the reference's own;
  * compiles every ``*_cuda.cu`` with ``nvcc -O3 -gencode arch=compute_100a,code=sm_100a``
    (the reference's flags, zip torchsparse/setup.py:25-28, + the arch) and every ``*_cpu.cpp``
    + ``pybind_cuda.cpp`` with g++, one command per file (no setup.py);
  * links ``oracle/_ref/ts_ref_backend_cuda*.so`` (the 20-function pybind module of
    TS/backend/pybind_cuda.cpp:18-39) and ``oracle/_ref/rangelib_cuda*.so``
    (range_lib/range_utils/src/rangelib_bindings_gpu.cpp:7-12).

``oracle/_ref/`` is git-ignored: no reference source or binary enters the history.  Without the reference
package this script is a no-op that reports whether prebuilt modules are present.
"""
from __future__ import annotations

import glob
import os
import re
import subprocess
import sys
import sysconfig
import tempfile
import zipfile
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
OUT_DIR = os.path.join(HERE, "_ref")
REF_PKG = "/root/reference/package"
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
TS_MOD, RL_MOD = "ts_ref_backend_cuda", "rangelib_cuda"

sys.path.insert(0, os.path.dirname(HERE))
from oracle.build_ref import _SPARSECONFIG              # noqa: E402  same generated header as the CPU recipe


def module_path(name: str) -> str | None:
    hits = glob.glob(os.path.join(OUT_DIR, name + ".*so"))
    return hits[0] if hits else None


def _patch(path: str) -> None:
    src = open(path).read()
    new = re.sub(r"AT_DISPATCH_FLOATING_TYPES_AND_HALF\(\s*([A-Za-z_]+)\.type\(\)",
                 r"AT_DISPATCH_FLOATING_TYPES_AND_HALF(\1.scalar_type()", src)
    new = new.replace("<THC/THCAtomics.cuh>", "<ATen/cuda/Atomic.cuh>")
    if new != src:
        open(path, "w").write(new)


def _compile(srcs, mod_name, inc, tmp, out):
    import torch
    abi = "-D_GLIBCXX_USE_CXX11_ABI=" + str(int(torch._C._GLIBCXX_USE_CXX11_ABI))
    common = ["-DTORCH_API_INCLUDE_EXTENSION_H", f"-DTORCH_EXTENSION_NAME={mod_name}", abi]
    common += ["-I" + p for p in inc]
    cxx = ["g++", "-O3", "-fopenmp", "-fPIC", "-std=c++17", "-w", *common]
    nvcc = [NVCC, "-O3", "-gencode", "arch=compute_100a,code=sm_100a", "-std=c++17", "-w",
            "-Xcompiler", "-fPIC", "--expt-relaxed-constexpr", *common]

    def cc(src: str) -> str:
        obj = os.path.join(tmp, mod_name + "_" + os.path.basename(src) + ".o")
        subprocess.check_call([*(nvcc if src.endswith(".cu") else cxx), "-c", src, "-o", obj])
        return obj

    with ThreadPoolExecutor(max_workers=min(8, os.cpu_count() or 1)) as ex:
        objs = list(ex.map(cc, srcs))
    libdir = os.path.join(os.path.dirname(torch.__file__), "lib")
    subprocess.check_call(["g++", "-shared", *objs, "-o", out, "-fopenmp", "-L" + libdir,
                           "-L/usr/local/cuda/lib64", "-lc10", "-lc10_cuda", "-ltorch", "-ltorch_cpu",
                           "-ltorch_cuda", "-ltorch_python", "-lcudart", "-Wl,-rpath," + libdir])
    return out


def build(force: bool = False, verbose: bool = True):
    have = (module_path(TS_MOD), module_path(RL_MOD))
    if all(have) and not force:
        return have
    if not os.path.isdir(REF_PKG):
        if verbose:
            print("[oracle/_ref] reference package absent; prebuilt CUDA modules:", have)
        return have
    from torch.utils import cpp_extension

    os.makedirs(OUT_DIR, exist_ok=True)
    ext = sysconfig.get_config_var("EXT_SUFFIX") or ".so"
    with tempfile.TemporaryDirectory(prefix="b2s_refcuda_") as tmp:
        for z in ("torchsparse", "sparsehash", "range_lib"):
            zipfile.ZipFile(os.path.join(REF_PKG, z + ".zip")).extractall(tmp)
        backend = os.path.join(tmp, "torchsparse", "torchsparse", "backend")
        sh_src = os.path.join(tmp, "sparsehash-master", "src")
        with open(os.path.join(sh_src, "sparsehash", "internal", "sparseconfig.h"), "w") as f:
            f.write(_SPARSECONFIG)
        inc = cpp_extension.include_paths(device_type="cuda") + [sysconfig.get_paths()["include"], sh_src]
        srcs = sorted(set(glob.glob(os.path.join(backend, "**", "*_cpu.cpp"), recursive=True))
                      | set(glob.glob(os.path.join(backend, "**", "*_cuda.cu"), recursive=True)))
        srcs = [s for s in srcs if not os.path.basename(s).startswith("pybind_")]
        srcs.append(os.path.join(backend, "pybind_cuda.cpp"))
        for s in srcs:
            _patch(s)
        ts_out = _compile(srcs, TS_MOD, inc + [backend], tmp, os.path.join(OUT_DIR, TS_MOD + ext))
        rl = os.path.join(tmp, "range_lib", "range_utils", "src")
        rl_srcs = sorted(glob.glob(os.path.join(rl, "*.cpp")) + glob.glob(os.path.join(rl, "*.cu")))
        rl_out = _compile(rl_srcs, RL_MOD, inc + [rl], tmp, os.path.join(OUT_DIR, RL_MOD + ext))
    if verbose:
        print("[oracle/_ref] built", ts_out, rl_out)
    return ts_out, rl_out


def load(name: str = TS_MOD):
    """Import a compiled reference CUDA module, or return None when it is not built."""
    path = module_path(name)
    if path is None:
        return None
    import importlib.util

    import torch  # noqa: F401
    spec = importlib.util.spec_from_file_location(name, path)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


if __name__ == "__main__":
    build(force="--force" in sys.argv)
