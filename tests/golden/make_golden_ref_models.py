#!/usr/bin/env python
"""Run the reference's OWN four sparse segmentors (staged unmodified by oracle/stage_ref.py) on the CPU
build of its bundled torchsparse (oracle/_ref) and freeze their outputs (build container only).

    python tests/golden/make_golden_ref_models.py  ->  tests/golden/ref_models.npz

Per model (MinkUNet-34 cr1.0, SPVCNN-18 cr1.0, Cylinder3D cy480, RPVNet-34 cr1.75; MODEL block of the
reference yaml, key-seeded weights from oracle/det_weights.py, train mode = batch statistics, every
Dropout / Dropout2d instance set to p = 0 so the outputs are deterministic):
one synthetic scan (seed 3, 64 beams x 60 azimuths) -> training loss + the logits of the classifier head.
What is NOT the reference in this arm, and why:
  * ``Tensor.cuda`` is patched to the identity (the models call ``.cuda()`` on targets, rpvnet.py:86, minkunet.py:425);
  * ``torch_scatter.scatter_max`` (third-party, absent) and ``rangelib_cuda`` (CUDA-only in the reference) are torch
    stand-ins (baseline/loader.py);
  * single scan per batch: the reference's CPU kernel-hash reads point 0's batch word for every point
    (TS/backend/hash/hash_cpu.cpp:29);
  * forward only: the reference's devoxelize_backward_cpu is wrong (devoxelize_cpu.cpp:48-53), so gradients of
    this arm are not truth.  Gradients are compared on the GPU box against the reference's CUDA build instead
    (tests/test_gpu_ref_models.py).
Inputs are regenerated from the seed at test time (openpcseg_b200.synthetic.make_model_batch); their CRC32 is
stored so that a drifted generator fails loudly instead of comparing different scans.
"""
import os
import sys
import time
import warnings
import zlib

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
warnings.filterwarnings("ignore")

CASES = [("minkunet34", "voxel"), ("spvcnn18", "voxel"), ("cylinder480", "cylinder"), ("rpvnet34", "fusion")]
SEED, N_AZIMUTH = 3, 60


def input_crc(arrays: dict) -> int:
    c = 0
    for k in sorted(arrays):
        v = arrays[k]
        if isinstance(v, np.ndarray):
            c = zlib.crc32(np.ascontiguousarray(v).tobytes(), c)
    return c


def head_module(name, net):
    return net.logits if name == "cylinder480" else net.classifier


def main():
    torch.Tensor.cuda = lambda self, *a, **k: self
    from baseline import loader
    from openpcseg_b200.synthetic import make_model_batch
    from oracle.det_weights import fill_
    ns = loader.activate("ref_cpu")
    torch.set_num_threads(8)
    out = {}
    for name, kind in CASES:
        t0 = time.time()
        net = ns.build_model(name)
        net.load_state_dict(fill_(net.state_dict()), strict=True)
        net.train()
        for m in net.modules():                    # RPVNet's range branch carries Dropout2d(0.2): random
            if isinstance(m, (torch.nn.Dropout, torch.nn.Dropout2d)):
                m.p = 0.0
        arrays = make_model_batch(kind, [SEED], n_azimuth=N_AZIMUTH)
        cap = {}

        def hook(m, i, o):
            cap["logits"] = (o.F if hasattr(o, "F") else o).detach().clone()
            if hasattr(o, "C"):
                cap["coords"] = o.C.detach().clone()
        h = head_module(name, net).register_forward_hook(hook)
        with torch.no_grad():
            ret, _, _ = net(ns.batch_dict(arrays, "cpu"))
        h.remove()
        out[name + "/loss"] = np.float32(float(ret["loss"]))
        out[name + "/logits"] = cap["logits"].numpy().astype(np.float32)
        if "coords" in cap:
            out[name + "/coords"] = cap["coords"].numpy().astype(np.int32)
        out[name + "/input_crc"] = np.uint32(input_crc(arrays))
        print(f"{name}: loss {float(ret['loss']):.6f} logits {tuple(cap['logits'].shape)} "
              f"|max| {float(cap['logits'].abs().max()):.3f}  {time.time() - t0:.1f}s")
    np.savez_compressed(os.path.join(HERE, "ref_models.npz"), **out)


if __name__ == "__main__":
    main()
