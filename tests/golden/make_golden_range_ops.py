#!/usr/bin/env python
"""Run the reference's own range_lib CUDA build (``rangelib_cuda``, recompiled for sm_100a by
oracle/build_ref_cuda.py) on the inputs of tests/test_gpu_ref_models.py::test_range_ops_match_reference_cuda_build
and freeze its outputs (needs a GPU and oracle/_ref).

    python tests/golden/make_golden_range_ops.py  ->  tests/golden/range_ops.npz

Stored: the full count map (uint8; it holds small counts and compresses well), and for a fixed seeded sample of
occupied pixels / of points the dense image and the feature gradient, with the maxima of the full arrays that the
test's relative bars are taken against.  The CRC32 of the inputs makes a drifted input generator fail loudly.
"""
import os
import sys
import zlib

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)

N_PIXELS, N_POINTS = 3072, 3072


def inputs():
    """pxpy [n, 3] int32 (batch, x, y), feat [n, c], top [b, c, h, w]: 200 k points on every third column of a
    3 x 64 x 2048 image, so that many pixels receive several points."""
    g = torch.Generator().manual_seed(5)
    n, c, b, h, w = 200_000, 24, 3, 64, 2048
    pxpy = torch.stack([torch.randint(0, b, (n,), generator=g), torch.randint(0, w // 4, (n,), generator=g) * 3,
                        torch.randint(0, h, (n,), generator=g)], 1).int()
    feat = torch.randn(n, c, generator=g)
    top = torch.randn(b, c, h, w, generator=g)
    return pxpy, feat, top, (b, h, w)


def input_crc(*tensors) -> int:
    c = 0
    for t in tensors:
        c = zlib.crc32(t.contiguous().numpy().tobytes(), c)
    return c


def main():
    from baseline import loader
    ref = loader._load_so("rangelib_cuda", loader.REF_DIR)
    pxpy, feat, top, (b, h, w) = inputs()
    cm = ref.map_count_forward(pxpy.cuda(), b, h, w)
    img = ref.denselize_forward(feat.cuda(), cm, pxpy.cuda()).cpu()
    grad = ref.denselize_backward(top.cuda(), cm, pxpy.cuda()).cpu()
    cm = cm.cpu()
    assert int(cm.max()) < 256
    g = torch.Generator().manual_seed(0)
    occupied = torch.nonzero(cm.reshape(-1)).view(-1)
    pix = occupied[torch.randperm(len(occupied), generator=g)[:N_PIXELS]].sort().values
    pts = torch.randperm(len(feat), generator=g)[:N_POINTS].sort().values
    img_px = img.permute(0, 2, 3, 1).reshape(b * h * w, -1)[pix]
    np.savez_compressed(
        os.path.join(HERE, "range_ops.npz"),
        input_crc=np.uint32(input_crc(pxpy, feat, top)), count_map=cm.numpy().astype(np.uint8),
        pixels=pix.numpy(), img_at_pixels=img_px.numpy(), img_absmax=np.float32(img.abs().max()),
        points=pts.numpy(), grad_at_points=grad[pts].numpy(), grad_absmax=np.float32(grad.abs().max()))
    print(f"range_ops: {len(occupied)} occupied pixels, max count {int(cm.max())}")


if __name__ == "__main__":
    main()
