"""CPU checks around the reference-arm plumbing: golden inputs reproducible from the seed, the staged
reference segmentors import and construct unmodified on the shim, and the range_utils / torch_scatter
names resolve to this backend."""
import os
import sys
import zlib

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from baseline import loader                                          # noqa: E402

CASES = [("minkunet34", "voxel", 37882900, 63), ("spvcnn18", "voxel", 21785780, 49),
         ("cylinder480", "cylinder", 55892042, 48), ("rpvnet34", "fusion", 123021828, 63)]


def _crc(arrays):
    c = 0
    for k in sorted(arrays):
        if isinstance(arrays[k], np.ndarray):
            c = zlib.crc32(np.ascontiguousarray(arrays[k]).tobytes(), c)
    return c


@pytest.mark.parametrize("name,kind", [(c[0], c[1]) for c in CASES])
def test_golden_inputs_regenerate_from_seed(name, kind, golden):
    from openpcseg_b200.synthetic import make_model_batch
    arrays = make_model_batch(kind, [3], n_azimuth=60)
    assert np.uint32(_crc(arrays)) == golden("ref_models")[name + "/input_crc"]


def test_model_batches_have_the_reference_collate_layout():
    from openpcseg_b200.synthetic import make_model_batch
    v = make_model_batch("voxel", [0, 1], n_azimuth=40)
    assert v["coords"].dtype == np.int32 and v["coords"].shape[1] == 4 and v["feats"].shape[1] == 4
    assert v["offset"].tolist() == np.cumsum(np.bincount(v["coords"][:, 3])).tolist()
    f = make_model_batch("fusion", [0, 1], n_azimuth=40)
    assert f["feats"].shape[1] == 5 and f["range_image"].shape == (2, 5, 64, 2048)
    assert f["range_pxpy"].shape == (len(f["feats"]), 3) and np.abs(f["range_pxpy"][:, 1:]).max() <= 1.0
    assert set(np.unique(f["range_pxpy"][:, 0])) == {0.0, 1.0}
    c = make_model_batch("cylinder", [0, 1], n_azimuth=40)
    assert c["point_feature"].shape == (2 * 64 * 40, 9) and c["point_coord"].dtype == np.int64
    assert (c["point_coord"][:, :3].max(0) < np.array([480, 360, 32])).all() and c["point_coord"].min() >= 0
    assert c["offset"][-1] == len(c["voxel_coord"]) == len(c["voxel_label"])


@pytest.mark.skipif(not loader.staged(), reason="oracle/_ref/py not staged (the reference is not available)")
@pytest.mark.parametrize("name,kind,n_params,n_conv", CASES)
def test_reference_segmentors_construct_unmodified_on_the_shim(name, kind, n_params, n_conv):
    ns = loader.activate("b2s")
    import torchsparse
    import torchsparse.nn as spnn
    import range_utils.nn.functional as rnf
    import torch_scatter
    assert torchsparse.__name__ == "openpcseg_b200.torchsparse"
    assert rnf.__name__ == "openpcseg_b200.range_utils.nn.functional"
    assert torch_scatter.__name__.endswith("torch_scatter")
    net = ns.build_model(name)
    assert type(net).__module__ == loader.MODELS[name][1]
    src = sys.modules[type(net).__module__].__file__
    assert os.path.realpath(src).startswith(os.path.realpath(loader.PY))
    assert sum(p.numel() for p in net.parameters()) == n_params
    assert sum(isinstance(m, spnn.Conv3d) for m in net.modules()) == n_conv
