"""Load the reference's OWN segmentor classes (staged byte-for-byte under ``oracle/_ref/py`` by
``oracle/stage_ref.py``) on a chosen sparse backend.  Not product code: the product is the backend
under them; this is how tests and bench.py run the unmodified callers.

    ns = activate("b2s")        # torchsparse / range_utils / torch_scatter resolve to openpcseg_b200
    ns = activate("ref_cuda")   # ... resolve to the reference's python package + its CUDA build (B3)
    ns = activate("ref_cpu")    # ... its CPU build (oracle/_ref), range_utils / torch_scatter = torch stand-ins
    net = ns.build_model("minkunet34")            # MODEL block of the reference yaml, IF_DIST False
    batch = ns.batch_dict(arrays, device)         # tensors -> the reference's batch_dict (SparseTensor of `ns`)

Only ONE backend is active per process at a time: activating another one purges ``torchsparse*``,
``range_utils*``, ``rangelib_cuda``, ``torch_scatter``, ``pcseg*``, ``tools*`` from ``sys.modules`` so that
the model modules are re-imported and re-bound.  Objects created under a previous activation keep
working (their modules stay alive through their globals) except for imports done lazily at call time.
"""
from __future__ import annotations

import glob
import importlib
import importlib.util
import os
import sys
import types

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
REF_DIR = os.path.join(ROOT, "oracle", "_ref")
PY = os.path.join(REF_DIR, "py")

MODELS = {
    "minkunet34": ("voxel/semantic_kitti/minkunet_mk34_cr10.yaml",
                   "pcseg.model.segmentor.voxel.minkunet.minkunet", "MinkUNet"),
    "minkunet18": ("voxel/semantic_kitti/minkunet_mk18_cr10.yaml",
                   "pcseg.model.segmentor.voxel.minkunet.minkunet", "MinkUNet"),
    "spvcnn18": ("fusion/semantic_kitti/spvcnn_mk18_cr10.yaml",
                 "pcseg.model.segmentor.fusion.spvcnn.spvcnn", "SPVCNN"),
    "cylinder480": ("voxel/semantic_kitti/cylinder_cy480_cr10.yaml",
                    "pcseg.model.segmentor.voxel.cylinder3d.cylinder_ts", "Cylinder_TS"),
    "rpvnet34": ("fusion/semantic_kitti/rpvnet_mk34_cr17_5.yaml",
                 "pcseg.model.segmentor.fusion.rpvnet.rpvnet", "RPVNet"),
}
_PURGE = ("torchsparse", "range_utils", "rangelib_cuda", "torch_scatter", "pcseg", "tools", "easydict")


class Cfg(dict):
    """EasyDict stand-in (easydict is not installed): attribute access on a dict."""
    __getattr__ = dict.__getitem__

    def __setattr__(self, k, v):
        self[k] = v


def _wrap(d):
    return Cfg({k: (_wrap(v) if isinstance(v, dict) else v) for k, v in d.items()})


def staged() -> bool:
    return os.path.isfile(os.path.join(PY, "pcseg/model/segmentor/voxel/minkunet/minkunet.py"))


def _load_so(name: str, directory: str):
    hits = glob.glob(os.path.join(directory, name + ".*so"))
    if not hits:
        raise FileNotFoundError(f"{name} is not built under {directory} (run oracle/stage_ref.py --cuda "
                                f"or oracle/build_ref.py where the reference is available)")
    import torch  # noqa: F401  (libtorch first)
    spec = importlib.util.spec_from_file_location(name, hits[0])
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def _torch_scatter_standin():
    """torch_scatter.scatter_max for the reference arms (third-party package, not in this image):
    values via ``scatter_reduce_('amax')``; argmax = smallest contributing row, like torch_scatter."""
    import torch
    m = types.ModuleType("torch_scatter")

    def scatter_max(src, index, dim=0, out=None, dim_size=None):
        assert dim == 0 and out is None and src.ndim == 2
        if index.ndim == 2:
            index = index[:, 0]
        index = index.long()
        n = int(dim_size) if dim_size is not None else int(index.max()) + 1
        idx = index[:, None].expand_as(src)
        val = torch.full((n, src.shape[1]), float("-inf"), dtype=src.dtype, device=src.device)
        val = val.scatter_reduce(0, idx, src, "amax", include_self=True)
        rows = torch.arange(src.shape[0], device=src.device)[:, None].expand_as(src)
        cand = torch.where(src == val.gather(0, idx), rows, torch.full_like(rows, src.shape[0]))
        arg = torch.full((n, src.shape[1]), src.shape[0], dtype=torch.long, device=src.device)
        arg = arg.scatter_reduce(0, idx, cand, "amin", include_self=True)
        val = torch.where(torch.isinf(val) & (val < 0), torch.zeros_like(val), val)
        return val, arg

    m.scatter_max = scatter_max
    return m


def _rangelib_cpu_standin():
    """``rangelib_cuda`` for the CPU golden arm only (range_lib ships no CPU build): torch restatement
    of map_count_gpu.cu:5-14 and denselize_gpu.cu:5-34."""
    import torch
    m = types.ModuleType("rangelib_cuda")

    def _pos(pxpy, h, w):
        p = pxpy.long()
        return (p[:, 0] * h + p[:, 2]) * w + p[:, 1]

    def map_count_forward(pxpy, max_bs, h, w):
        out = torch.zeros(max_bs * h * w, dtype=torch.int32)
        out.index_add_(0, _pos(pxpy, h, w), torch.ones(pxpy.shape[0], dtype=torch.int32))
        return out.view(max_bs, h, w)

    def denselize_forward(feat, count_map, pxpy):
        b, h, w = count_map.shape
        c = feat.shape[1]
        pos = _pos(pxpy, h, w)
        cnt = count_map.reshape(-1)[pos].float()
        out = torch.zeros(b * h * w, c)
        out.index_add_(0, pos, feat.float() / cnt[:, None])
        return out.view(b, h, w, c).permute(0, 3, 1, 2).contiguous()

    def denselize_backward(top_grad, count_map, pxpy):
        b, h, w = count_map.shape
        pos = _pos(pxpy, h, w)
        g = top_grad.permute(0, 2, 3, 1).reshape(b * h * w, -1)
        return g[pos] / count_map.reshape(-1)[pos].float()[:, None]

    m.map_count_forward, m.denselize_forward, m.denselize_backward = \
        map_count_forward, denselize_forward, denselize_backward
    return m


def _cpu_backend_proxy(real):
    """The reference's CPU backend with ONE function replaced: ``devoxelize_backward_cpu`` indexes
    ``top_grad`` by voxel index and writes for idx < 0 (TS/backend/devoxelize/devoxelize_cpu.cpp:48-53) - it
    reads out of bounds and segfaults on real scans.  The stand-in restates the CUDA twin
    (devoxelize_cuda.cu:37-58: grad_feat[idx[i,k]] += w[i,k] * g[i]) with index_add_.  Everything else
    (conv fwd/bwd, hash, query, count, voxelize, devoxelize fwd) is the reference's compiled code."""
    import torch
    proxy = types.ModuleType(real.__name__ + "_proxy")
    for k in dir(real):
        if not k.startswith("__"):
            setattr(proxy, k, getattr(real, k))

    def devoxelize_backward_cpu(top_grad, idx, weight, n):
        out = torch.zeros(n, top_grad.shape[1], dtype=top_grad.dtype)
        for k in range(idx.shape[1]):
            ok = idx[:, k] >= 0
            out.index_add_(0, idx[ok, k].long(), top_grad[ok] * weight[ok, k:k + 1].to(top_grad.dtype))
        return out

    proxy.devoxelize_backward_cpu = devoxelize_backward_cpu
    return proxy


class Namespace:
    def __init__(self, kind, torchsparse):
        self.kind, self.torchsparse = kind, torchsparse
        self.SparseTensor, self.PointTensor = torchsparse.SparseTensor, torchsparse.PointTensor

    def model_cfg(self, name: str, **over):
        import yaml
        with open(os.path.join(PY, "tools/cfgs", MODELS[name][0])) as f:
            cfg = _wrap(yaml.safe_load(f)["MODEL"])
        # IF_DIST False = plain BatchNorm1d (one process); RPVNet keeps the yaml's True because its
        # IF_DIST False branch applies the sparse BatchNorm wrapper to dense point features and
        # raises in the reference itself (rpvnet.py:574,261-263); without an initialised process
        # group nn.SyncBatchNorm computes plain batch statistics.
        cfg["IF_DIST"] = name.startswith("rpvnet")
        cfg.update(over)
        return cfg

    def model_class(self, name: str):
        _, module, cls = MODELS[name]
        return getattr(importlib.import_module(module), cls)

    def build_model(self, name: str, num_class: int = 20, **over):
        return self.model_class(name)(self.model_cfg(name, **over), num_class)

    def batch_dict(self, arrays: dict, device):
        """numpy / tensor arrays of ``openpcseg_b200.synthetic.make_model_batch`` -> the reference's batch_dict."""
        import numpy as np
        import torch

        def T(v):
            t = torch.from_numpy(v) if isinstance(v, np.ndarray) else v
            return t.to(device, non_blocking=True)

        a = {k: (T(v) if isinstance(v, (np.ndarray, torch.Tensor)) else v) for k, v in arrays.items()}
        if "coords" in a:                                          # voxel / fusion models
            d = {"lidar": self.SparseTensor(a["feats"], a["coords"]),
                 "targets": self.SparseTensor(a["labels"], a["coords"]),
                 "offset": a["offset"]}
            for k in ("range_image", "range_pxpy"):
                if k in a:
                    d[k] = a[k]
            return d
        return {k: a[k] for k in ("point_feature", "point_coord", "point_label", "voxel_coord", "voxel_label",
                                  "offset")}


def activate(kind: str = "b2s") -> Namespace:
    assert kind in ("b2s", "ref_cuda", "ref_cpu"), kind
    if not staged():
        raise FileNotFoundError("reference sources are not staged under oracle/_ref/py "
                                "(python oracle/stage_ref.py where the reference is available)")
    for name in [m for m in sys.modules if m.split(".")[0] in _PURGE]:
        del sys.modules[name]
    for p in (ROOT, PY):
        if p in sys.path:
            sys.path.remove(p)
    sys.path.insert(0, PY)
    sys.path.insert(0, ROOT)
    easy = types.ModuleType("easydict")
    easy.EasyDict = Cfg
    sys.modules["easydict"] = easy
    if kind == "b2s":
        import openpcseg_b200
        openpcseg_b200.install_as_torchsparse()
    else:
        if kind == "ref_cuda":
            backend = _load_so("ts_ref_backend_cuda", REF_DIR)
            sys.modules["rangelib_cuda"] = _load_so("rangelib_cuda", REF_DIR)
        else:
            backend = _cpu_backend_proxy(_load_so("ts_ref_backend", REF_DIR))
            sys.modules["rangelib_cuda"] = _rangelib_cpu_standin()
        sys.modules["torchsparse.backend"] = backend
        sys.modules["torch_scatter"] = _torch_scatter_standin()
        import warnings
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            ts = importlib.import_module("torchsparse")          # the reference's python package (staged)
        ts.backend = backend
        assert os.path.realpath(ts.__file__).startswith(os.path.realpath(PY)), ts.__file__
    return Namespace(kind, importlib.import_module("torchsparse"))
