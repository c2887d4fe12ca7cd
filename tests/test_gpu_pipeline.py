"""GPU tests of the batch ingest path (lt_images_hwc_to_nchw_fwd through prepare_batch) and of the pipelined
InferenceStream: same values as the torch formulation / as one synchronous forward per batch."""
import numpy as np
import pytest
import torch

import lt_b200
from lt_b200 import pipeline, testing

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


@pytest.mark.parametrize("dtype", [np.uint8, np.float32, np.float64])
@pytest.mark.parametrize("shape", [(1, 1, 6, 10, 3), (2, 3, 33, 47, 3), (2, 2, 128, 128, 3), (1, 2, 17, 9, 1)])
def test_images_to_device_native_equals_torch(dtype, shape):
    rng = np.random.RandomState(shape[2])
    imgs = rng.randint(0, 256, size=shape).astype(np.uint8) if dtype == np.uint8 else (rng.randn(*shape) * 3).astype(dtype)
    want = pipeline.images_to_device(imgs, "cpu", backend="torch")
    got = pipeline.images_to_device(imgs, DEV)
    assert got.is_cuda and got.dtype == torch.float32 and tuple(got.shape) == tuple(want.shape)
    assert torch.equal(got.cpu(), want)
    if dtype == np.uint8 and shape[-1] == 3:
        want_n = pipeline.images_to_device(imgs, "cpu", normalize_u8=True, backend="torch")
        got_n = pipeline.images_to_device(imgs, DEV, normalize_u8=True)
        assert torch.equal(got_n.cpu(), want_n)          # table lookup: bit-exact normalize_image (img.py:102-110)


def test_pinned_collate_and_prepare_batch():
    items = testing.dataset_items(3, 4, size=16, dtype=np.float64, seed=2)
    batch = pipeline.make_collate_fn(randomize_n_views=False, pinned=True)(items)
    assert torch.from_numpy(batch["images"]).is_pinned()
    native = pipeline.prepare_batch(batch, DEV, None)
    ref = pipeline.prepare_batch(batch, "cpu", None, backend="torch")
    for a, b in zip(native, ref):
        assert a.is_cuda and torch.equal(a.cpu(), b)


def test_inference_stream_equals_synchronous_forward():
    B, V, S, n = 2, 2, 128, 32
    cfg = testing.make_config(num_layers=50, volume_size=n)
    model = lt_b200.VolumetricTriangulationNet(cfg, device=DEV, backend="native", conv_mode="tc")
    testing.randomize_weights(model, seed=1, calib_size=S)
    model = model.to(DEV).eval()
    batches, want = [], []
    for i in range(5):
        images, batch = testing.make_batch(B, V, image_size=S, seed=20 + i)
        hwc = np.ascontiguousarray(images.permute(0, 1, 3, 4, 2).numpy())
        if i % 2 == 0:                                   # mix pinned and pageable submissions
            pinned = pipeline.pinned_empty(hwc.shape, hwc.dtype)
            pinned[...] = hwc
            hwc = pinned
        batch["images"] = hwc
        batches.append(batch)
        with torch.no_grad():
            want.append(model(images.to(DEV), None, batch)[0].cpu().numpy().copy())
    stream = pipeline.InferenceStream(model)
    got = list(stream.run(batches))
    assert len(got) == len(want)
    for g, w in zip(got, want):
        assert g.shape == (B, 17, 3) and np.array_equal(g, w)      # same kernels, same inputs, in order
    assert stream.h2d_bytes == sum(b["images"].nbytes for b in batches)
    assert stream.d2h_bytes == 5 * B * 17 * 3 * 4
    assert list(stream.run([])) == []
