#!/usr/bin/env python
"""Stage the UNMODIFIED reference's callers of the hot path (no reference file enters git).

Where the reference tree is available, this script copies, byte for byte, into the git-ignored
``oracle/_ref/py/`` (next to the reference backends that oracle/build_ref.py and oracle/build_ref_cuda.py
compile), so that the reference arm runs from ``oracle/_ref/`` alone:

  pcseg/model/segmentor/base_segmentors.py, voxel/{minkunet,cylinder3d}/*.py,
  fusion/{spvcnn,rpvnet}/*.py          the four sparse segmentors = the CALLERS of the hot path
  pcseg/loss/*.py                       their criterion
  tools/utils/common/{__init__,seg_utils,lovasz_losses}.py
  tools/cfgs/{voxel,fusion}/semantic_kitti/*.yaml
  torchsparse/**.py                     python half of package/torchsparse.zip (v1.4.0), for the
                                        reference-on-its-own-backend arms (not used by our backend)
  range_utils/**.py                     python half of package/range_lib.zip

``pcseg/model/__init__.py`` and ``pcseg/model/segmentor/__init__.py`` are deliberately NOT staged: they
import every segmentor of the repo (range-view CNNs and their extra dependencies); without them the
directories are namespace packages and ``pcseg.model.segmentor.voxel.minkunet.minkunet`` etc. import
exactly as in the reference tree.

With ``--cuda`` it also runs ``oracle/build_ref_cuda.py`` (the reference's CUDA backends for sm_100a).
"""
from __future__ import annotations

import glob
import os
import shutil
import sys
import zipfile

HERE = os.path.dirname(os.path.abspath(__file__))
OUT = os.path.join(HERE, "_ref", "py")
REF = "/root/reference"

_FILES = [
    "pcseg/model/segmentor/base_segmentors.py",
    "pcseg/model/segmentor/voxel/minkunet/*.py",
    "pcseg/model/segmentor/voxel/cylinder3d/*.py",
    "pcseg/model/segmentor/fusion/spvcnn/*.py",
    "pcseg/model/segmentor/fusion/rpvnet/*.py",
    "pcseg/loss/*.py",
    "tools/utils/common/__init__.py",
    "tools/utils/common/seg_utils.py",
    "tools/utils/common/lovasz_losses.py",
    "tools/cfgs/voxel/semantic_kitti/*.yaml",
    "tools/cfgs/fusion/semantic_kitti/*.yaml",
]


def staged() -> bool:
    return os.path.isfile(os.path.join(OUT, "pcseg/model/segmentor/voxel/minkunet/minkunet.py"))


def stage(force: bool = False, verbose: bool = True) -> str | None:
    if staged() and not force:
        return OUT
    if not os.path.isdir(REF):
        if verbose:
            print("[oracle/_ref] reference tree absent; staged tree present:", staged())
        return OUT if staged() else None
    shutil.rmtree(OUT, ignore_errors=True)
    n = 0
    for pat in _FILES:
        for src in glob.glob(os.path.join(REF, pat)):
            dst = os.path.join(OUT, os.path.relpath(src, REF))
            os.makedirs(os.path.dirname(dst), exist_ok=True)
            shutil.copyfile(src, dst)
            n += 1
    for zname, prefix, top in (("torchsparse.zip", "torchsparse/torchsparse/", "torchsparse"),
                               ("range_lib.zip", "range_lib/range_utils/", "range_utils")):
        with zipfile.ZipFile(os.path.join(REF, "package", zname)) as z:
            for name in z.namelist():
                if name.startswith(prefix) and name.endswith(".py"):
                    dst = os.path.join(OUT, top, name[len(prefix):])
                    os.makedirs(os.path.dirname(dst), exist_ok=True)
                    with open(dst, "wb") as f:
                        f.write(z.read(name))
                    n += 1
    if verbose:
        print(f"[oracle/_ref] staged {n} reference files under {OUT}")
    return OUT


if __name__ == "__main__":
    stage(force="--force" in sys.argv)
    if "--cuda" in sys.argv:
        sys.path.insert(0, os.path.dirname(HERE))
        from oracle import build_ref_cuda
        build_ref_cuda.build(force="--force" in sys.argv)
