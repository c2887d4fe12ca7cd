"""Oracle and host mirror vs the reference itself: the reference's outputs on these exact inputs are stored in
tests/golden/oracle_vs_reference.npz (tests/golden/make_golden.py)."""
import os

import numpy as np
import pytest
import torch

from conftest import GOLDEN, rel_err

from oracle import vol_oracle as O  # noqa: E402
from lt_b200 import testing, torch_ops  # noqa: E402
from lt_b200 import v2v as lt_v2v, pose_resnet as lt_pose_resnet  # noqa: E402


@pytest.fixture(scope="module")
def ref():
    return np.load(os.path.join(GOLDEN, "oracle_vs_reference.npz"))


SHAPES = [(1, 2, 3, 9, 13, 5), (2, 8, 4, 12, 12, 6), (1, 9, 2, 8, 6, 4)]


@pytest.mark.parametrize("shape", SHAPES)
@pytest.mark.parametrize("agg", ["sum", "max", "softmax", "conf"])
def test_unproject_random(ref, shape, agg):
    B, V, C, h, w, n = shape
    rng = np.random.RandomState(B * 100 + V)
    heat = rng.randn(B, V, C, h, w).astype(np.float32)
    cams = testing.make_cameras(V, image_size=48, radius=3000.0)
    proj = np.stack([np.stack([O.projection_after_resize(c.K, c.R, c.t, (48, 48), (h, w)) for c in cams])] * B)
    coord = np.stack([O.coord_volume(rng.randn(3) * 100 + [0, 0, 900], 2600.0, n) for _ in range(B)])
    conf = rng.rand(B, V, C).astype(np.float32)
    i = SHAPES.index(shape)
    assert [testing.array_digest(a) for a in (heat, proj, coord, conf)] == list(ref["unp%d_inputs" % i]), \
        "inputs differ from those the reference was run on"
    want = ref["unp%d_out_%s" % (i, agg)]
    assert rel_err(O.unproject_heatmaps(heat, proj, coord, agg, conf), want) < 2e-5
    got_t = torch_ops.unproject_heatmaps(torch.from_numpy(heat), torch.from_numpy(proj), torch.from_numpy(coord), agg,
                                         torch.from_numpy(conf)).numpy()
    assert rel_err(got_t, want) < 2e-5


def test_coord_volume_and_projection_bit_exact(ref):
    base = ref["coord_base"]
    # the reference volume is stored as its three axes: coordinate c of voxel (i, j, k) depends on index (i, j, k)[c] only
    x, y, z = ref["coord_x"], ref["coord_y"], ref["coord_z"]
    coords = np.stack(np.broadcast_arrays(x[:, None, None], y[None, :, None], z[None, None, :]), -1)
    mine = O.coord_volume(base, 2500.0, 32)
    assert np.array_equal(mine, coords)
    assert np.array_equal(O.projection_after_resize(ref["cam_K"], ref["cam_R"], ref["cam_t"], (64, 64), (16, 16)),
                          ref["cam_projection_16"])


def _checksum(tensors):
    return float(sum(torch.as_tensor(t).double().abs().sum() for t in tensors))


def _close_to_reference(got, ref, key, channel_axes):
    got = got.detach().numpy()
    denom = float(ref[key + "_absmax"][0])
    assert float(np.abs(np.abs(got).max() - denom)) <= 1e-5 * denom
    assert float(np.abs(testing.golden_sample(got, int(ref["sample_k"][0])) - ref[key + "_sample"]).max()) < 1e-5 * denom
    if channel_axes is not None:
        mean = got.astype(np.float64).mean(channel_axes)
        assert float(np.abs(mean - ref[key + "_channel_mean"]).max()) < 1e-5 * denom


def test_v2v_and_backbone_functional_restatement(ref):
    # weights and inputs: the same seeded sequence the reference models were built from (their checksums are stored)
    torch.manual_seed(0)
    v = lt_v2v.V2VModel(32, 17).eval()
    for m in v.modules():
        if isinstance(m, torch.nn.BatchNorm3d):
            m.running_mean.normal_(0, 0.1)
            m.running_var.uniform_(0.5, 1.5)
    x = torch.randn(1, 32, 32, 32, 32)
    assert np.allclose([_checksum(v.state_dict().values()), _checksum([x])], ref["v2v_checksum"], rtol=1e-12, atol=0)
    _close_to_reference(O.v2v_forward(v.state_dict(), x), ref, "v2v", (0, 2, 3, 4))
    cfg = testing.AttrDict(num_layers=34, style="simple", num_joints=17, alg_confidences=False, vol_confidences=False,
                           init_weights=False)
    bb = lt_pose_resnet.get_pose_net(cfg, device="cpu").eval()
    xi = torch.randn(2, 3, 64, 64)
    assert np.allclose([_checksum(bb.state_dict().values()), _checksum([xi])], ref["backbone_checksum"], rtol=1e-12, atol=0)
    ohm, ofe = O.pose_resnet_forward(bb.state_dict(), xi)
    _close_to_reference(ofe, ref, "backbone_features", (0, 2, 3))
    _close_to_reference(ohm, ref, "backbone_heatmaps", None)
