"""Generate the golden fixtures in this directory from the UNMODIFIED reference.

Needs a checkout of karfly/learnable-triangulation-pytorch (the tests themselves never do):
    python tests/golden/make_golden.py <reference checkout> [fixture ...]
It imports the reference read-only, feeds it seeded synthetic inputs and the
seeded weight recipe of lt_b200.testing (loaded with strict=True -- which also proves state_dict
compatibility), and stores small input/output vectors as .npz.  Nothing is copied from the reference.
With fixture names (e.g. `oracle_vs_reference collate`) only those files are regenerated.
"""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
if len(sys.argv) < 2 or not os.path.isdir(os.path.join(sys.argv[1], "mvn")):
    raise SystemExit("usage: python tests/golden/make_golden.py <reference checkout> [fixture ...]")
sys.path.insert(0, os.path.abspath(sys.argv[1]))

import lt_b200  # noqa: E402
from lt_b200 import testing  # noqa: E402
from mvn.models.triangulation import VolumetricTriangulationNet as RefNet  # noqa: E402
from mvn.utils import multiview as ref_multiview  # noqa: E402
from mvn.utils import op as ref_op  # noqa: E402


def scene(B, V, C, h, w, n, seed):
    """Small unprojection problem with voxels behind cameras / outside the maps (edge cases of op.py:121-141)."""
    rng = np.random.RandomState(seed)
    heat = rng.randn(B, V, C, h, w).astype(np.float32)
    cams = testing.make_cameras(V, image_size=64, radius=2600.0, height=1200.0)
    proj = np.zeros((B, V, 3, 4), dtype=np.float32)
    for b in range(B):
        for v in range(V):
            c = testing.Camera(cams[v].R, cams[v].t, cams[v].K)
            c.update_after_resize((64, 64), (h, w))
            proj[b, v] = c.projection.astype(np.float32)
    proj[0, 0, 2, :] *= -1.0          # view 0 of sample 0 sees everything behind the camera (depth <= 0)
    side = 3000.0                      # cuboid larger than the field of view -> out-of-image taps
    idx = np.arange(n, dtype=np.float32)
    g = np.stack(np.meshgrid(idx, idx, idx, indexing="ij"), -1)
    coord = np.stack([(-side / 2 + side / (n - 1) * g + np.array([0, 0, 900.0]) + rng.randn(3) * 50).astype(np.float32)
                      for _ in range(B)])
    coord[-1, 0, 0, 0] = -np.linalg.inv(cams[-1].R) @ cams[-1].t.ravel()   # a voxel exactly at a camera centre (z == 0)
    conf = rng.rand(B, V, C).astype(np.float32)
    return heat, proj, coord, conf


def gen_unproject():
    out = {}
    for tag, (B, V, C, h, w, n) in {"a": (2, 3, 4, 12, 16, 8), "b": (1, 4, 32, 10, 10, 6), "c": (1, 1, 5, 7, 9, 5)}.items():
        heat, proj, coord, conf = scene(B, V, C, h, w, n, seed=ord(tag))
        out[tag + "_heat"], out[tag + "_proj"], out[tag + "_coord"], out[tag + "_conf"] = heat, proj, coord, conf
        for agg in ("sum", "max", "softmax", "conf"):
            r = ref_op.unproject_heatmaps(torch.from_numpy(heat), torch.from_numpy(proj), torch.from_numpy(coord), agg,
                                          torch.from_numpy(conf))
            out["%s_out_%s" % (tag, agg)] = r.numpy()
    np.savez_compressed(os.path.join(HERE, "unproject.npz"), **out)


def gen_softargmax():
    rng = np.random.RandomState(7)
    B, J, n = 2, 3, 6
    vols = (rng.randn(B, J, n, n, n) * 3).astype(np.float32)
    coord = (rng.randn(B, n, n, n, 3) * 500).astype(np.float32)
    out = {"vols": vols, "coord": coord}
    for sm in (True, False):
        kp, v = ref_op.integrate_tensor_3d_with_coordinates(torch.from_numpy(vols), torch.from_numpy(coord), softmax=sm)
        out["kp_%d" % sm], out["v_%d" % sm] = kp.numpy(), v.numpy()
    np.savez_compressed(os.path.join(HERE, "softargmax.npz"), **out)


def gen_forward():
    """Whole eval forward: B=2, V=2, 128x128, ResNet-50, 32^3 grid (BASELINE config #1 flavour)."""
    torch.manual_seed(0)
    np.random.seed(0)
    B, V, S, n = 2, 2, 128, 32
    cfg = testing.make_config(num_layers=50, volume_size=n, volume_multiplier=1.0)
    mine = lt_b200.VolumetricTriangulationNet(cfg, device="cpu", backend="torch")
    testing.randomize_weights(mine, seed=1, calib_size=S)
    sd = mine.state_dict()
    ref = RefNet(testing.make_config(num_layers=50, volume_size=n, volume_multiplier=1.0), device="cpu")
    ref.load_state_dict(sd, strict=True)
    ref.eval()
    images, batch = testing.make_batch(B, V, image_size=S, seed=3, camera_cls=ref_multiview.Camera)
    grabbed = {}
    h1 = ref.volume_net.register_forward_hook(lambda m, i, o: grabbed.update(vol_in=i[0].detach(), logits=o.detach()))
    with torch.no_grad():
        kp, feats, vols, conf, cuboids, coords, base = ref(images, None, batch)
    h1.remove()
    assert conf is None
    flat = vols.reshape(B, 17, -1)
    out = {
        "sd_checksum": np.array([float(sum(v.double().abs().sum() for v in sd.values()))]),
        "keypoints": kp.numpy(), "base_points": base.numpy(),
        "features_sub": feats[:, :, ::4, ::3, ::3].numpy(),
        "coord_sub": coords[:, ::5, ::5, ::5].numpy(),
        "vol_in_sub": grabbed["vol_in"][:, ::4, ::3, ::3, ::3].numpy(),
        "logits_sub": grabbed["logits"][:, :, ::3, ::3, ::3].numpy(),
        "volumes_sub": vols[:, :, ::3, ::3, ::3].numpy(),
        "volumes_argmax": flat.argmax(-1).numpy(), "volumes_max": flat.max(-1)[0].numpy(),
        "cuboid_position": np.stack([c.position for c in cuboids]), "cuboid_sides": np.stack([c.sides for c in cuboids]),
    }
    np.savez_compressed(os.path.join(HERE, "forward_r50.npz"), **out)
    print("forward_r50: max prob", float(flat.max()), "uniform", 1.0 / n ** 3, "kp spread", kp.std(dim=1))


def gen_algebraic():
    """AlgebraicTriangulationNet (config #5 flavour): B=2, V=4, 128x128, ResNet-50, with confidences."""
    from mvn.models.triangulation import AlgebraicTriangulationNet as RefAlg
    B, V, S = 2, 4, 128
    mine = lt_b200.AlgebraicTriangulationNet(testing.make_alg_config(num_layers=50), device="cpu", backend="torch")
    testing.randomize_backbone_weights(mine, seed=5, calib_size=S)
    sd = mine.state_dict()
    ref = RefAlg(testing.make_alg_config(num_layers=50), device="cpu")
    ref.load_state_dict(sd, strict=True)
    ref.eval()
    images, batch = testing.make_batch(B, V, image_size=S, seed=9, camera_cls=ref_multiview.Camera)
    proj = torch.from_numpy(testing.image_projections(batch))
    with torch.no_grad():
        kp3d, kp2d, heat, conf = ref(images, proj, batch)
    out = {"sd_checksum": np.array([float(sum(v.double().abs().sum() for v in sd.values()))]),
           "proj": proj.numpy(), "keypoints_3d": kp3d.numpy(), "keypoints_2d": kp2d.numpy(), "confidences": conf.numpy(),
           "heatmaps_sub": heat[:, :, :, ::2, ::2].numpy(), "heatmaps_argmax": heat.reshape(B, V, 17, -1).argmax(-1).numpy()}
    np.savez_compressed(os.path.join(HERE, "algebraic_r50.npz"), **out)
    print("algebraic_r50: heat max", float(heat.max()), "kp3d", kp3d[0, :3])


def gen_state_dict_keys():
    """Key -> shape table of the reference ResNet-152 volumetric model (1311 tensors)."""
    import json
    ref = RefNet(testing.make_config(num_layers=152), device="cpu")
    with open(os.path.join(HERE, "state_dict_r152.json"), "w") as f:
        json.dump({k: list(v.shape) for k, v in ref.state_dict().items()}, f)


def gen_state_dict_r18():
    """Key -> shape table of the reference ResNet-18 volumetric model at a 32^3 grid (the train.py drop-in test's model)."""
    import json
    ref = RefNet(testing.make_config(num_layers=18, volume_size=32), device="cpu")
    with open(os.path.join(HERE, "state_dict_r18.json"), "w") as f:
        json.dump({k: list(v.shape) for k, v in ref.state_dict().items()}, f)


def _checksum(tensors):
    return float(sum(torch.as_tensor(t).double().abs().sum() for t in tensors))


def gen_oracle_vs_reference():
    """Reference outputs for tests/test_oracle_vs_reference.py: unprojection on random scenes, the coordinate volume and
    projection of a ResNet-18 forward, and V2V / pose-ResNet-34 forwards (weights and inputs from torch.manual_seed(0)).
    Large outputs are stored as a fixed seeded sample of SAMPLE draws (testing.golden_sample) plus per-channel means."""
    from oracle import vol_oracle as O
    from mvn.models import v2v as ref_v2v, pose_resnet as ref_pose_resnet
    SAMPLE = 16384
    out = {"sample_k": np.array([SAMPLE])}
    for i, (B, V, C, h, w, n) in enumerate([(1, 2, 3, 9, 13, 5), (2, 8, 4, 12, 12, 6), (1, 9, 2, 8, 6, 4)]):
        rng = np.random.RandomState(B * 100 + V)
        heat = rng.randn(B, V, C, h, w).astype(np.float32)
        cams = testing.make_cameras(V, image_size=48, radius=3000.0)
        proj = np.stack([np.stack([O.projection_after_resize(c.K, c.R, c.t, (48, 48), (h, w)) for c in cams])] * B)
        coord = np.stack([O.coord_volume(rng.randn(3) * 100 + [0, 0, 900], 2600.0, n) for _ in range(B)])
        conf = rng.rand(B, V, C).astype(np.float32)
        out["unp%d_inputs" % i] = np.array([testing.array_digest(a) for a in (heat, proj, coord, conf)])
        for agg in ("sum", "max", "softmax", "conf"):
            out["unp%d_out_%s" % (i, agg)] = ref_op.unproject_heatmaps(torch.from_numpy(heat), torch.from_numpy(proj),
                                                                       torch.from_numpy(coord), agg, torch.from_numpy(conf)).numpy()

    base = np.array([123.4, -56.7, 910.1])
    net = RefNet(testing.make_config(num_layers=18, volume_size=32), device="cpu").eval()
    images, batch = testing.make_batch(1, 2, image_size=64, seed=5, camera_cls=ref_multiview.Camera)
    batch["keypoints_3d"][0][6, :3] = base
    with torch.no_grad():
        coords = net(images, None, batch)[5].numpy()[0]
    # each coordinate depends on its own voxel index only, so three axes hold the whole volume bit for bit
    axes = [coords[:, 0, 0, 0], coords[0, :, 0, 1], coords[0, 0, :, 2]]
    full = np.stack(np.broadcast_arrays(axes[0][:, None, None], axes[1][None, :, None], axes[2][None, None, :]), -1)
    assert np.array_equal(full, coords)
    out["coord_base"] = base
    out["coord_x"], out["coord_y"], out["coord_z"] = axes
    cam = batch["cameras"][1][0]
    c2 = ref_multiview.Camera(cam.R, cam.t, cam.K)
    c2.update_after_resize((64, 64), (16, 16))
    out["cam_K"], out["cam_R"], out["cam_t"] = cam.K, cam.R, cam.t
    out["cam_projection_16"] = c2.projection.astype(np.float32)

    torch.manual_seed(0)
    v = ref_v2v.V2VModel(32, 17).eval()
    for m in v.modules():
        if isinstance(m, torch.nn.BatchNorm3d):
            m.running_mean.normal_(0, 0.1)
            m.running_var.uniform_(0.5, 1.5)
    x = torch.randn(1, 32, 32, 32, 32)
    with torch.no_grad():
        want = v(x)
    out["v2v_checksum"] = np.array([_checksum(v.state_dict().values()), _checksum([x])])
    out["v2v_sample"] = testing.golden_sample(want.numpy(), SAMPLE)
    out["v2v_channel_mean"] = want.double().mean((0, 2, 3, 4)).numpy()
    out["v2v_absmax"] = np.array([float(want.abs().max())])
    cfg = testing.AttrDict(num_layers=34, style="simple", num_joints=17, alg_confidences=False, vol_confidences=False,
                           init_weights=False)
    bb = ref_pose_resnet.get_pose_net(cfg, device="cpu").eval()
    xi = torch.randn(2, 3, 64, 64)
    with torch.no_grad():
        hm, feats, _, _ = bb(xi)
    out["backbone_checksum"] = np.array([_checksum(bb.state_dict().values()), _checksum([xi])])
    out["backbone_heatmaps_sample"] = testing.golden_sample(hm.numpy(), SAMPLE)
    out["backbone_heatmaps_absmax"] = np.array([float(hm.abs().max())])
    out["backbone_features_sample"] = testing.golden_sample(feats.numpy(), SAMPLE)
    out["backbone_features_channel_mean"] = feats.double().mean((0, 2, 3)).numpy()
    out["backbone_features_absmax"] = np.array([float(feats.abs().max())])
    np.savez_compressed(os.path.join(HERE, "oracle_vs_reference.npz"), **out)


def gen_collate():
    """Reference collate_fn / prepare_batch / normalize_image outputs for tests/test_pipeline_cpu.py, all compared for
    exact equality there, so only their digests (testing.array_digest) are stored."""
    from mvn.datasets import utils as ref_utils
    from mvn.utils import img as ref_img
    out = {}
    for randomize in (False, True):
        items = testing.dataset_items(3, 5, seed=9, camera_cls=ref_multiview.Camera)
        np.random.seed(11)
        want = ref_utils.make_collate_fn(randomize_n_views=randomize, min_n_views=2, max_n_views=4)(list(items))
        key = "r%d_" % randomize
        for name in ("images", "detections", "pred_keypoints_3d"):
            out[key + name] = testing.array_digest(want[name])
        # which item / view each collated camera is, [view][batch] -> (item, view)
        where = {id(c): (b, v) for b, it in enumerate(items) for v, c in enumerate(it["cameras"])}
        out[key + "camera_index"] = np.array([[where[id(c)] for c in row] for row in want["cameras"]])
        out[key + "prepared"] = np.array([testing.array_digest(t.numpy()) for t in ref_utils.prepare_batch(want, "cpu", None)])
    u8 = np.random.RandomState(1).randint(0, 256, size=(2, 2, 6, 7, 3)).astype(np.uint8)
    ref_norm = np.stack([np.stack([ref_img.normalize_image(im) for im in row]) for row in u8])
    out["u8_normalized"] = testing.array_digest(torch.stack([ref_img.image_batch_to_torch(x) for x in ref_norm]).numpy())
    np.savez_compressed(os.path.join(HERE, "collate.npz"), **out)


if __name__ == "__main__":
    fixtures = {"state_dict_r152": gen_state_dict_keys, "state_dict_r18": gen_state_dict_r18, "unproject": gen_unproject, "softargmax": gen_softargmax,
                "forward_r50": gen_forward, "algebraic_r50": gen_algebraic, "oracle_vs_reference": gen_oracle_vs_reference,
                "collate": gen_collate}
    for name in sys.argv[2:] or fixtures:
        fixtures[name]()
    for f in sorted(os.listdir(HERE)):
        print(f, os.path.getsize(os.path.join(HERE, f)))
