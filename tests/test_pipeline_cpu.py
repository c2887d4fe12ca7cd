"""Host batch contract (lt_b200.pipeline): collate, normalisation table, prepare_batch (torch backend on CPU).
Reference behaviours mirrored: mvn/datasets/utils.py:6-65, mvn/utils/img.py:96-110.  What the reference functions return
for the same inputs is stored as digests in tests/golden/collate.npz (tests/golden/make_golden.py)."""
import os

import numpy as np
import pytest
import torch

from conftest import GOLDEN
from lt_b200 import pipeline, testing


def test_normalization_table_is_normalize_image_rounded_once():
    lut = pipeline.normalization_table()
    assert lut.shape == (3, 256) and lut.dtype == np.float32
    img = np.arange(256, dtype=np.uint8).reshape(16, 16, 1).repeat(3, axis=2)
    want = ((img / 255.0 - pipeline.IMAGENET_MEAN) / pipeline.IMAGENET_STD).astype(np.float32)      # img.py:102-110
    got = lut[np.arange(3)[None, None, :], img]
    assert np.array_equal(got, want)


def test_collate_layout_and_none_filtering(capsys):
    items = testing.dataset_items(3, 4)
    fn = pipeline.make_collate_fn(randomize_n_views=False)
    batch = fn([items[0], None, items[1], items[2]])
    assert batch["images"].shape == (3, 4, 8, 10, 3) and batch["images"].flags["C_CONTIGUOUS"]
    for b in range(3):
        for v in range(4):
            assert np.array_equal(batch["images"][b, v], items[b]["images"][v])
    assert len(batch["cameras"]) == 4 and len(batch["cameras"][0]) == 3            # [view][batch]
    assert batch["detections"].shape == (3, 4, 5)
    assert batch["pred_keypoints_3d"].shape == (3, 17, 3)
    assert batch["indexes"] == [0, 1, 2]
    assert fn([None, None]) is None
    assert "All items in batch are None" in capsys.readouterr().out


def test_collate_random_views_within_bounds():
    items = testing.dataset_items(2, 6)
    fn = pipeline.make_collate_fn(randomize_n_views=True, min_n_views=2, max_n_views=4)
    np.random.seed(3)
    seen = set()
    for _ in range(20):
        b = fn(items)
        V = b["images"].shape[1]
        assert 2 <= V <= 4 and len(b["cameras"]) == V
        seen.add(V)
    assert len(seen) > 1


@pytest.mark.parametrize("dtype", [np.float64, np.float32, np.uint8])
def test_prepare_batch_torch_backend(dtype):
    items = testing.dataset_items(2, 3, dtype=dtype, seed=4)
    batch = pipeline.make_collate_fn(randomize_n_views=False)(items)
    images, kp, valid, proj = pipeline.prepare_batch(batch, "cpu", None, backend="torch")
    assert images.shape == (2, 3, 3, 8, 10) and images.dtype == torch.float32
    want = torch.from_numpy(batch["images"]).permute(0, 1, 4, 2, 3).float()
    assert torch.equal(images, want)
    assert kp.shape == (2, 17, 3) and valid.shape == (2, 17, 1) and proj.shape == (2, 3, 3, 4)
    for b in range(2):
        for v in range(3):
            assert np.array_equal(proj[b, v].numpy(), batch["cameras"][v][b].projection.astype(np.float32))
    if dtype == np.uint8:
        normed = pipeline.prepare_batch(batch, "cpu", None, normalize_u8=True, backend="torch")[0]
        ref = ((batch["images"] / 255.0 - pipeline.IMAGENET_MEAN) / pipeline.IMAGENET_STD).astype(np.float32)
        assert np.array_equal(normed.numpy(), ref.transpose(0, 1, 4, 2, 3))


def test_native_backend_refuses_cpu_device():
    batch = pipeline.make_collate_fn(randomize_n_views=False)(testing.dataset_items(1, 2))
    with pytest.raises(RuntimeError):
        pipeline.prepare_batch(batch, "cpu", None)          # default backend is the CUDA path: no silent CPU route


@pytest.mark.parametrize("randomize", [False, True])
def test_collate_and_prepare_batch_equal_reference(randomize):
    ref = np.load(os.path.join(GOLDEN, "collate.npz"))
    key = "r%d_" % randomize
    items = testing.dataset_items(3, 5, seed=9)
    np.random.seed(11)
    got = pipeline.make_collate_fn(randomize_n_views=randomize, min_n_views=2, max_n_views=4)(list(items))
    for name in ("images", "detections", "pred_keypoints_3d"):
        assert testing.array_digest(got[name]) == ref[key + name], name
    where = {id(c): (b, v) for b, it in enumerate(items) for v, c in enumerate(it["cameras"])}
    assert np.array_equal([[where[id(c)] for c in row] for row in got["cameras"]], ref[key + "camera_index"])
    m = pipeline.prepare_batch(got, "cpu", None, backend="torch")
    assert [testing.array_digest(t.numpy()) for t in m] == list(ref[key + "prepared"])
    # uint8 crops normalised through the table == normalize_image on the CPU, then the reference upload path
    u8 = np.random.RandomState(1).randint(0, 256, size=(2, 2, 6, 7, 3)).astype(np.uint8)
    got_t = pipeline.images_to_device(u8, "cpu", normalize_u8=True, backend="torch")
    assert testing.array_digest(got_t.numpy()) == ref["u8_normalized"]
