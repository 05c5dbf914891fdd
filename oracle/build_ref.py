#!/usr/bin/env python
"""Recipe: compile the REFERENCE's own CPU backend into ``oracle/_ref/``.

TEST INFRASTRUCTURE ONLY (see oracle/ref_ops.py header).

What it does
  * reads the reference sources where they lie: the two zips
    ``/root/reference/package/{torchsparse,sparsehash}.zip`` are unpacked into a
    throw-away directory under ``$TMPDIR`` (never into this repo);
  * compiles ``torchsparse/backend/**/*_cpu.cpp`` + ``pybind_cpu.cpp`` with plain
    ``g++`` (one command per file, no setup.py / configure / cmake) against the
    torch headers of this interpreter;
  * the only non-reference file is a 12-line ``sparseconfig.h`` (the header
    sparsehash's ``configure`` would generate; the zip ships only the Windows
    copy) written into the temp dir;
  * links ``oracle/_ref/ts_ref_backend*.so`` - a pybind11 module exporting the
    reference's ``*_cpu`` functions (TS/backend/pybind_cpu.cpp:12-23).

``oracle/_ref/`` is git-ignored (no reference sources or binaries enter the
history) but NOT gpurun-ignored, so the built module travels to the GPU box,
where ``/root/reference`` does not exist.  Without ``/root/reference`` this
script is a no-op that reports whether a prebuilt module is present.
"""
from __future__ import annotations

import glob
import os
import subprocess
import sys
import sysconfig
import tempfile
import zipfile
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
OUT_DIR = os.path.join(HERE, "_ref")
MOD_NAME = "ts_ref_backend"
REF_PKG = "/root/reference/package"

_SPARSECONFIG = """\
#define GOOGLE_NAMESPACE ::google
#define HASH_FUN_H <functional>
#define HASH_NAMESPACE std
#define HAVE_INTTYPES_H 1
#define HAVE_LONG_LONG 1
#define HAVE_MEMCPY 1
#define HAVE_STDINT_H 1
#define HAVE_SYS_TYPES_H 1
#define HAVE_UINT16_T 1
#define HAVE_U_INT16_T 1
#define SPARSEHASH_HASH HASH_NAMESPACE::hash
#define _END_GOOGLE_NAMESPACE_ }
#define _START_GOOGLE_NAMESPACE_ namespace google {
"""


def module_path() -> str | None:
    hits = glob.glob(os.path.join(OUT_DIR, MOD_NAME + ".*so"))     # not ts_ref_backend_cuda
    return hits[0] if hits else None


def build(force: bool = False, verbose: bool = True) -> str | None:
    have = module_path()
    if have and not force:
        return have
    if not os.path.isdir(REF_PKG):
        if verbose:
            print("[oracle/_ref] /root/reference absent; prebuilt module:", have)
        return have
    import torch
    from torch.utils import cpp_extension

    os.makedirs(OUT_DIR, exist_ok=True)
    with tempfile.TemporaryDirectory(prefix="b2s_refbuild_") as tmp:
        zipfile.ZipFile(os.path.join(REF_PKG, "torchsparse.zip")).extractall(tmp)
        zipfile.ZipFile(os.path.join(REF_PKG, "sparsehash.zip")).extractall(tmp)
        backend = os.path.join(tmp, "torchsparse", "torchsparse", "backend")
        sh_src = os.path.join(tmp, "sparsehash-master", "src")
        cfg_dir = os.path.join(sh_src, "sparsehash", "internal")
        with open(os.path.join(cfg_dir, "sparseconfig.h"), "w") as f:
            f.write(_SPARSECONFIG)
        srcs = sorted(set(glob.glob(os.path.join(backend, "**", "*_cpu.cpp"), recursive=True)))
        inc = cpp_extension.include_paths() + [sysconfig.get_paths()["include"], sh_src]
        cflags = ["-O3", "-fopenmp", "-fPIC", "-std=c++17", "-w",
                  "-DTORCH_API_INCLUDE_EXTENSION_H", f"-DTORCH_EXTENSION_NAME={MOD_NAME}",
                  "-D_GLIBCXX_USE_CXX11_ABI=" + str(int(torch._C._GLIBCXX_USE_CXX11_ABI))]
        cflags += ["-I" + p for p in inc]

        def cc(src: str) -> str:
            obj = os.path.join(tmp, os.path.basename(src) + ".o")
            subprocess.check_call(["g++", *cflags, "-c", src, "-o", obj])
            return obj

        with ThreadPoolExecutor(max_workers=min(8, os.cpu_count() or 1)) as ex:
            objs = list(ex.map(cc, srcs))
        ext = sysconfig.get_config_var("EXT_SUFFIX") or ".so"
        out = os.path.join(OUT_DIR, MOD_NAME + ext)
        libdir = os.path.join(os.path.dirname(torch.__file__), "lib")
        subprocess.check_call(["g++", "-shared", *objs, "-o", out, "-fopenmp", "-L" + libdir,
                               "-lc10", "-ltorch", "-ltorch_cpu", "-ltorch_python",
                               "-Wl,-rpath," + libdir])
    if verbose:
        print("[oracle/_ref] built", out)
    return out


def load():
    """Import the compiled reference backend, or return None when it is not built."""
    path = module_path()
    if path is None:
        return None
    import importlib.util

    import torch  # noqa: F401  (libtorch must be loaded first)
    spec = importlib.util.spec_from_file_location(MOD_NAME, path)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


if __name__ == "__main__":
    build(force="--force" in sys.argv)
