"""Drop-in proof for the reference's training script, without the reference itself.

`lt_b200.install()` rebinds the names `train.py` imports (tested on a stand-in `mvn` package); then the statements of
`train.py` that touch the model run against lt_b200's class as `train.py` would call it: construction from the experiment
config with the backend chosen by LT_B200_BACKEND (train.py:400-404), strict `load_state_dict` of a checkpoint with DDP's
`module.` prefixes and the reference's key set (:406-413, key/shape table in tests/golden/state_dict_r18.json), the three
optimizer parameter groups (:430-437), `DistributedDataParallel` wrapping (:452-453, gloo, world_size 2) and one
forward/backward/step of the loop body (:189-243) on the CPU.
"""
import json
import os
import socket
import sys
import types

import numpy as np
import pytest
import torch
import torch.multiprocessing as mp

from conftest import GOLDEN


def _tiny_config():
    """experiments/human36m/train/human36m_vol_softmax.yaml shrunk for a CPU test: ResNet-18 backbone, 32^3 grid, no
    pretrained weights.  The yaml differs from testing.make_config only in use_gt_pelvis; `opt` holds its learning rates."""
    from lt_b200 import testing
    config = testing.make_config(num_layers=18, volume_size=32, use_gt_pelvis=False)
    config.opt = testing.AttrDict(lr=1e-4, process_features_lr=1e-3, volume_net_lr=1e-3)
    return config


def _build_model(config, device="cpu"):
    """train.py:400-404: the class is called with (config, device) only; the backend comes from the environment."""
    import lt_b200
    os.environ["LT_B200_BACKEND"] = "torch"
    try:
        return lt_b200.VolumetricTriangulationNet(config, device=device).to(device)
    finally:
        os.environ.pop("LT_B200_BACKEND")


def _keypoints_mae(pred, gt, validity):
    """The MAE criterion train.py selects (opt.criterion: MAE): masked mean absolute error over joints and coordinates."""
    return torch.sum(torch.abs(gt - pred) * validity) / (pred.shape[-1] * max(1, float(validity.sum())))


@pytest.fixture
def stand_in_mvn():
    """A package shaped like the reference's `mvn`, holding placeholders where install() must put lt_b200's objects."""
    name = "mvn_stand_in"
    mods = {}
    for sub in ("", ".models", ".models.triangulation", ".utils", ".utils.op"):
        mods[name + sub] = types.ModuleType(name + sub)
    tri, op = mods[name + ".models.triangulation"], mods[name + ".utils.op"]
    for attr in ("VolumetricTriangulationNet", "AlgebraicTriangulationNet", "RANSACTriangulationNet"):
        setattr(tri, attr, type(attr, (), {}))
    for attr in ("integrate_tensor_2d", "unproject_heatmaps", "integrate_tensor_3d_with_coordinates"):
        setattr(op, attr, lambda *a, **k: None)
    mods[name].models, mods[name].utils = mods[name + ".models"], mods[name + ".utils"]
    mods[name + ".models"].triangulation, mods[name + ".utils"].op = tri, op
    sys.modules.update(mods)
    try:
        yield mods[name]
    finally:
        for key in mods:
            sys.modules.pop(key, None)


def test_install_patches_the_names_train_py_binds(stand_in_mvn):
    import lt_b200
    ransac = stand_in_mvn.models.triangulation.RANSACTriangulationNet
    assert lt_b200.install(stand_in_mvn) is stand_in_mvn
    tri, ref_op = stand_in_mvn.models.triangulation, stand_in_mvn.utils.op
    assert tri.VolumetricTriangulationNet is lt_b200.VolumetricTriangulationNet
    assert tri.AlgebraicTriangulationNet is lt_b200.AlgebraicTriangulationNet
    assert tri.RANSACTriangulationNet is ransac                       # not replaced: no native implementation
    assert ref_op.integrate_tensor_2d is lt_b200.op.integrate_tensor_2d
    assert ref_op.unproject_heatmaps is lt_b200.op.unproject_heatmaps
    assert ref_op.integrate_tensor_3d_with_coordinates is lt_b200.op.integrate_tensor_3d_with_coordinates
    # what train.py does at import time, after install()
    scope = {}
    exec("from mvn_stand_in.models.triangulation import VolumetricTriangulationNet, AlgebraicTriangulationNet", scope)
    assert scope["VolumetricTriangulationNet"] is lt_b200.VolumetricTriangulationNet
    assert scope["AlgebraicTriangulationNet"] is lt_b200.AlgebraicTriangulationNet


def test_train_py_model_setup_statements():
    """train.py:400-413 (construct + strict load of a DDP-prefixed checkpoint) and :430-437 (optimizer parameter groups)."""
    import lt_b200
    config = _tiny_config()
    model = _build_model(config)
    assert isinstance(model, lt_b200.VolumetricTriangulationNet) and model.backend == "torch"
    # a checkpoint with the reference model's key set, as saved under DDP (train.py:465-469)
    shapes = json.load(open(os.path.join(GOLDEN, "state_dict_r18.json")))
    g = torch.Generator().manual_seed(0)
    saved = {k: torch.randn(s, generator=g) if s else torch.randint(0, 100, (), generator=g) for k, s in shapes.items()}
    state_dict = {"module." + k: v for k, v in saved.items()}
    for key in list(state_dict.keys()):                                                  # train.py:408-410
        new_key = key.replace("module.", "")
        state_dict[new_key] = state_dict.pop(key)
    model.load_state_dict(state_dict, strict=True)                                       # train.py:412
    have = model.state_dict()
    assert set(have) == set(saved)
    for k, v in saved.items():
        assert torch.equal(have[k], v.to(have[k].dtype)), k
    opt = torch.optim.Adam(                                                              # train.py:430-437
        [{'params': model.backbone.parameters()},
         {'params': model.process_features.parameters(), 'lr': config.opt.process_features_lr if hasattr(config.opt, "process_features_lr") else config.opt.lr},
         {'params': model.volume_net.parameters(), 'lr': config.opt.volume_net_lr if hasattr(config.opt, "volume_net_lr") else config.opt.lr}],
        lr=config.opt.lr)
    assert [g["lr"] for g in opt.param_groups] == [1e-4, 1e-3, 1e-3]
    in_groups = [p for g in opt.param_groups for p in g["params"]]
    assert len({id(p) for p in in_groups}) == len(in_groups)                             # no parameter in two groups
    assert {id(p) for p in in_groups} == {id(p) for p in model.parameters()}             # and none left out
    assert not any(p.requires_grad for p in model.backbone.final_layer.parameters())     # frozen head, triangulation.py:235-236


def _free_port():
    s = socket.socket(); s.bind(("127.0.0.1", 0)); p = s.getsockname()[1]; s.close(); return p


def _ddp_worker(rank, world, port, ret):
    import torch.distributed as dist
    from torch.nn.parallel import DistributedDataParallel
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        from lt_b200 import testing
        torch.manual_seed(0)
        model = _build_model(_tiny_config())
        model = DistributedDataParallel(model)                                           # train.py:452-453 (device_ids=None on CPU)
        opt = torch.optim.Adam(filter(lambda p: p.requires_grad, model.parameters()), lr=1e-4)
        images, batch = testing.make_batch(2, 2, image_size=64, seed=10 + rank)   # 2 samples: train-mode BN at the 1^3 V2V level
        model.train()
        keypoints_3d_pred, heatmaps_pred, volumes_pred, confidences_pred, cuboids_pred, coord_volumes_pred, base_points_pred = \
            model(images, None, batch)                                                   # train.py:189-191
        gt = torch.from_numpy(np.stack(batch["keypoints_3d"])[:, :, :3]).float()
        validity = torch.ones(2, 17, 1)
        loss = _keypoints_mae(keypoints_3d_pred * 0.1, gt * 0.1, validity)               # train.py:219-221 (scale_keypoints_3d)
        opt.zero_grad()
        loss.backward()                                                                  # train.py:236
        g = model.module.process_features[0].weight.grad.clone()
        opt.step()
        # DDP averaged the gradient: identical on both ranks although the inputs differ
        gathered = [torch.zeros_like(g) for _ in range(world)]
        dist.all_gather(gathered, g)
        ret[rank] = (float(loss), bool(torch.equal(gathered[0], gathered[1])), tuple(keypoints_3d_pred.shape),
                     float(g.abs().sum()))
    finally:
        dist.destroy_process_group()


def test_ddp_wrap_and_one_training_step_gloo():
    """train.py:452-453 + one pass of the loop body: forward 7-tuple, loss, backward, optimizer step, gradients all-reduced."""
    world = 2
    ret = mp.get_context("spawn").Manager().dict()
    mp.spawn(_ddp_worker, args=(world, _free_port(), ret), nprocs=world, join=True)
    assert len(ret) == world
    for rank, (loss, same_grad, shape, grad_mass) in ret.items():
        assert np.isfinite(loss) and same_grad and shape == (2, 17, 3) and grad_mass > 0
