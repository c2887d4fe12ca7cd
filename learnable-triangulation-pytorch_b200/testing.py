"""Synthetic workload factory shared by tests, bench.py and __graft_entry__.smoke().

Nothing here is on the product path: it builds the experiment config (same schema as
experiments/human36m/*/human36m_vol_softmax.yaml), a ring of pinhole cameras, the `batch` dict in
the collate layout (mvn/datasets/utils.py:8-37) and a seeded, well-conditioned weight set.
(SURVEY.md section 8d defines the rig; Human3.6M and the released weights are not obtainable offline.)
"""
import numpy as np
import torch
from torch import nn

from .multiview import Camera


class AttrDict(dict):
    """10-line EasyDict stand-in: attribute access, AttributeError for missing keys (hasattr probes work)."""

    def __init__(self, d=None, **kw):
        super().__init__()
        for k, v in dict(d or {}, **kw).items():
            self[k] = AttrDict(v) if isinstance(v, dict) else v

    def __getattr__(self, k):
        try:
            return self[k]
        except KeyError:
            raise AttributeError(k)

    def __setattr__(self, k, v):
        self[k] = v


def make_config(num_layers=152, volume_size=64, aggregation="softmax", volume_multiplier=1.0, volume_softmax=True,
                use_gt_pelvis=True, kind="mpii", cuboid_side=2500.0, num_joints=17, style="simple"):
    """The `model:` section of human36m_vol_softmax.yaml with init_weights off (random init, BASELINE.json)."""
    return AttrDict({
        "image_shape": [384, 384],
        "model": {
            "name": "vol", "kind": kind, "volume_aggregation_method": aggregation,
            "init_weights": False, "use_gt_pelvis": use_gt_pelvis, "cuboid_side": cuboid_side,
            "volume_size": volume_size, "volume_multiplier": volume_multiplier, "volume_softmax": volume_softmax,
            "heatmap_softmax": True, "heatmap_multiplier": 100.0,
            "backbone": {"name": "resnet%d" % num_layers, "style": style, "init_weights": False,
                         "num_joints": num_joints, "num_layers": num_layers},
        },
    })


def _look_at(eye, target=(0.0, 0.0, 900.0)):
    """World->camera rotation for a camera at `eye` looking at `target`, z up (H3.6M-like, mm)."""
    eye, target = np.asarray(eye, dtype=np.float64), np.asarray(target, dtype=np.float64)
    fwd = target - eye
    fwd /= np.linalg.norm(fwd)
    right = np.cross(fwd, np.array([0.0, 0.0, 1.0]))
    right /= np.linalg.norm(right)
    down = np.cross(fwd, right)
    return np.stack([right, down, fwd], axis=0)


def make_cameras(n_views, image_size=384, radius=4500.0, height=1500.0, focal=None, phase=0.3, camera_cls=Camera):
    """n_views pinhole cameras on a ring looking at the subject; the 2.5 m cuboid fills the crop."""
    focal = focal if focal is not None else 520.0 * image_size / 384.0
    cams = []
    for v in range(n_views):
        a = phase + 2 * np.pi * v / n_views
        eye = np.array([radius * np.cos(a), radius * np.sin(a), height])
        R = _look_at(eye)
        t = -R @ eye
        K = np.array([[focal, 0.0, image_size / 2.0], [0.0, focal, image_size / 2.0], [0.0, 0.0, 1.0]])
        cams.append(camera_cls(R, t, K, name="cam%d" % v))
    return cams


def make_batch(batch_size, n_views, image_size=384, seed=0, camera_cls=Camera, device="cpu"):
    """-> images (B, V, 3, H, W) float32, batch dict with cameras[v][b], keypoints_3d, pred_keypoints_3d."""
    rng = np.random.RandomState(seed)
    g = torch.Generator().manual_seed(seed)
    images = torch.randn(batch_size, n_views, 3, image_size, image_size, generator=g)
    cams = make_cameras(n_views, image_size, camera_cls=camera_cls)
    cameras = [[camera_cls(c.R, c.t, c.K, name=c.name) for _ in range(batch_size)] for c in cams]
    kps = []
    for _ in range(batch_size):
        kp = np.concatenate([rng.normal(0.0, 200.0, size=(17, 3)) + np.array([0.0, 0.0, 900.0]), np.ones((17, 1))], axis=1)
        kps.append(kp)
    batch = {"cameras": cameras, "keypoints_3d": kps,
             "pred_keypoints_3d": np.stack([k[:, :3] for k in kps], axis=0)}
    return images.to(device), batch


def dataset_items(n_items, n_views, size=8, dtype=np.float64, seed=0, camera_cls=None):
    """Seeded dataset items (the per-sample dicts a collate_fn receives) with size x (size + 2) images of `dtype`."""
    rng = np.random.RandomState(seed)
    cams = make_cameras(n_views, image_size=size)
    if camera_cls is not None:
        cams = [camera_cls(c.R, c.t, c.K) for c in cams]
    items = []
    for i in range(n_items):
        if dtype == np.uint8:
            imgs = [rng.randint(0, 256, size=(size, size + 2, 3)).astype(np.uint8) for _ in range(n_views)]
        else:
            imgs = [rng.randn(size, size + 2, 3).astype(dtype) for _ in range(n_views)]
        items.append({"images": imgs, "detections": [rng.rand(5) for _ in range(n_views)], "cameras": list(cams),
                      "keypoints_3d": rng.randn(17, 4).astype(np.float32), "indexes": i,
                      "pred_keypoints_3d": rng.randn(17, 3)})
    return items


@torch.no_grad()
def randomize_weights(model, seed=0, calib_size=64, calib_views=2, feat_gain=4.0, branch_gain=0.2):
    """Seeded, non-degenerate weights (SURVEY.md hard part H1).

    Default inits in eval mode collapse the signal (BN running stats are 0/1, deconv outputs ~5e-3),
    which would make any parity check vacuous.  Recipe: Kaiming-normal conv filters, BatchNorm running
    affine gamma ~ U(0.75, 1.25), beta ~ N(0, 0.2), then running statistics calibrated by one train-mode
    pass of the torch formulation over seeded noise (momentum 1) and the output layer rescaled.  Deterministic for a given torch build.
    """
    g = torch.Generator().manual_seed(seed)
    dev = next(model.parameters()).device
    model_cpu = model.to("cpu")
    for mod in model_cpu.modules():
        if isinstance(mod, (nn.Conv2d, nn.Conv3d, nn.ConvTranspose2d, nn.ConvTranspose3d)):
            fan_in = mod.weight[0].numel() if not isinstance(mod, (nn.ConvTranspose2d, nn.ConvTranspose3d)) \
                else mod.weight.shape[0] * mod.weight[0, 0].numel() / (mod.stride[0] ** (mod.weight.dim() - 2))
            mod.weight.copy_(torch.randn(mod.weight.shape, generator=g) * (2.0 / fan_in) ** 0.5)
            if mod.bias is not None:
                mod.bias.copy_(torch.randn(mod.bias.shape, generator=g) * 0.05)
    bns = [m for m in model_cpu.modules() if isinstance(m, (nn.BatchNorm2d, nn.BatchNorm3d))]
    saved = [(m.momentum, m.training) for m in bns]
    # last BatchNorm of every residual branch: small gain, so that the identity path dominates (as in trained
    # residual nets; a random ResNet with unit-gain branches amplifies a 1e-5 perturbation ~250x, which would turn
    # the parity check into a test of fp32 summation order)
    last_of_branch = set()
    for mod in model_cpu.modules():
        if hasattr(mod, "stages") and hasattr(mod, "downsample"):
            last_of_branch.add(mod.stages()[-1][1])
        if hasattr(mod, "res_branch"):
            last_of_branch.add(mod.res_branch[4])
    for m in bns:
        # affine parameters first, so that the calibration below sees the final network
        lo, hi = (branch_gain * 0.5, branch_gain * 1.5) if m in last_of_branch else (0.75, 1.25)
        m.weight.copy_(torch.rand(m.weight.shape, generator=g) * (hi - lo) + lo)
        m.bias.copy_(torch.randn(m.bias.shape, generator=g) * 0.2)
        m.momentum = 1.0
        m.train()
    # calibration pass: the whole torch formulation (backbone -> process_features -> unprojection -> V2V) on a
    # synthetic scene, so every BatchNorm sees the activation statistics it will see at test time
    model_cpu.process_features[0].weight.mul_(feat_gain)   # wider feature range: view-softmax becomes selective
    # enough samples that the deepest V2V level (1^3 voxels per sample at volume_size 32) has stable statistics
    calib_batch = 2 if model_cpu.volume_size >= 64 else 6
    images, batch = make_batch(calib_batch, calib_views, image_size=calib_size, seed=seed + 1000)
    grabbed = {}
    hook = model_cpu.volume_net.output_layer.register_forward_hook(lambda m, i, o: grabbed.update(logits=o))
    top_training = model_cpu.training
    model_cpu.training = False                               # theta = 0; only the BatchNorms are in train mode
    backend, model_cpu.backend = getattr(model_cpu, "backend", "torch"), "torch"    # CPU calibration: torch ops whatever the backend
    model_cpu._forward_torch(images, batch)
    model_cpu.backend = backend
    model_cpu.training = top_training
    hook.remove()
    logits = grabbed["logits"]
    for m, (mom, tr) in zip(bns, saved):
        m.momentum = mom
        m.train(tr)
        m.running_var.clamp_(min=1e-3)
    # logits with a spread of ~2.5: the 3-D softmax is peaked but not saturated
    model_cpu.volume_net.output_layer.weight.mul_(2.5 / float(logits.std()))
    model_cpu.eval()
    return model_cpu.to(dev)


def make_alg_config(num_layers=152, use_confidences=True, heatmap_multiplier=100.0, num_joints=17):
    """The `model:` section of experiments/human36m/*/human36m_alg.yaml with init_weights off."""
    return AttrDict({
        "image_shape": [384, 384],
        "model": {"name": "alg", "init_weights": False, "use_confidences": use_confidences,
                  "heatmap_multiplier": heatmap_multiplier, "heatmap_softmax": True,
                  "backbone": {"name": "resnet%d" % num_layers, "style": "simple", "init_weights": False,
                               "num_joints": num_joints, "num_layers": num_layers}},
    })


def image_projections(batch):
    """(B, V, 3, 4) float32 image-space projection matrices of a make_batch() dict (datasets/utils.py:61-63)."""
    from .multiview import stack_projections
    return stack_projections(batch["cameras"])


@torch.no_grad()
def randomize_backbone_weights(model, seed=0, calib_size=128, calib_images=4, branch_gain=0.2, heat_spread=3.0):
    """Seeded well-conditioned weights for a model that only has `.backbone` (algebraic model): same recipe as
    randomize_weights; the heatmap head is rescaled so that heatmaps * heatmap_multiplier has a spread of ~3."""
    g = torch.Generator().manual_seed(seed)
    dev = next(model.parameters()).device
    m = model.to("cpu")
    bb = m.backbone
    for mod in bb.modules():
        if isinstance(mod, (nn.Conv2d, nn.ConvTranspose2d)):
            fan_in = mod.weight[0].numel() if isinstance(mod, nn.Conv2d) else mod.weight.shape[0] * mod.weight[0, 0].numel() / 4
            mod.weight.copy_(torch.randn(mod.weight.shape, generator=g) * (2.0 / fan_in) ** 0.5)
            if mod.bias is not None:
                mod.bias.copy_(torch.randn(mod.bias.shape, generator=g) * 0.05)
        if isinstance(mod, nn.Linear):
            mod.weight.copy_(torch.randn(mod.weight.shape, generator=g) * (1.0 / mod.weight.shape[1]) ** 0.5)
            mod.bias.copy_(torch.randn(mod.bias.shape, generator=g) * 0.3)
    last = {u.stages()[-1][1] for u in bb.modules() if hasattr(u, "stages")}
    bns = [x for x in bb.modules() if isinstance(x, nn.BatchNorm2d)]
    for x in bns:
        lo, hi = (branch_gain * 0.5, branch_gain * 1.5) if x in last else (0.75, 1.25)
        x.weight.copy_(torch.rand(x.weight.shape, generator=g) * (hi - lo) + lo)
        x.bias.copy_(torch.randn(x.bias.shape, generator=g) * 0.2)
        x.momentum = 1.0
        x.train()
    heat, _, _, _ = bb(torch.randn(calib_images, 3, calib_size, calib_size, generator=g))
    for x in bns:
        x.momentum = BN_MOMENTUM
        x.eval()
        x.running_var.clamp_(min=1e-3)
    scale = heat_spread / (float(heat.std()) * float(m.heatmap_multiplier))
    bb.final_layer.weight.mul_(scale)
    bb.final_layer.bias.mul_(scale)
    m.eval()
    return m.to(dev)


BN_MOMENTUM = 0.1


def golden_sample(a, k=2048, seed=0):
    """A fixed, seeded sample of at most k elements of `a` (all of them when it is no larger), flattened and in index order:
    stored golden data and dumped benchmark outputs shrink large arrays this way, so both sides draw the same indices."""
    a = np.asarray(a).reshape(-1)
    if a.size <= k:
        return a.copy()
    return a[np.unique(np.random.RandomState(seed).randint(0, a.size, size=k))]


def array_digest(a):
    """sha256 of an array's dtype, shape and bytes: stored instead of arrays that a test compares for exact equality."""
    import hashlib
    a = np.ascontiguousarray(a)
    return hashlib.sha256(("%s%s" % (a.dtype.str, a.shape)).encode() + a.tobytes()).hexdigest()
