"""GPU tests of the input step (csrc/image_prep.cu, data.resize_images / prepare_batch, unipose.forward_images):
cv2.resize bit for bit against the stored cv2 outputs and the numpy oracle, the three output modes against each other,
the network on device-resized images against forward_uint8, and the training labels against the reference's path."""
import hashlib
import os
import warnings

import numpy as np
import pytest
import torch

from conftest import GOLDEN
from oracle import evaluate_oracle as E
from oracle import image_prep_oracle as P
from oracle import unipose_oracle as O

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def golden():
    return np.load(os.path.join(GOLDEN, "resize_cv2.npz"))


def _sources(golden):
    return [P.synth_image(int(s), int(h), int(w)) for h, w, s in golden["sizes"]]


def _padded(img: np.ndarray, pitch: int) -> torch.Tensor:
    """A device image whose rows are `pitch` bytes apart (a view into a wider buffer)."""
    h, w, _ = img.shape
    buf = torch.zeros((h, pitch), dtype=torch.uint8)
    buf[:, :3 * w] = torch.from_numpy(img.reshape(h, 3 * w))
    return buf.cuda().as_strided((h, w, 3), (pitch, 3, 1))


@pytest.mark.parametrize("flip", [False, True])
def test_u8_bit_exact_vs_cv2_fixture_and_oracle(golden, flip):
    from unipose_b200 import data
    imgs = _sources(golden)
    dev = [torch.from_numpy(i).cuda() for i in imgs]
    fl = torch.full((len(dev),), flip, dtype=torch.bool, device="cuda")
    out = data.resize_images(dev, 368, flip=fl).cpu().numpy()
    for i, img in enumerate(imgs):
        ref = P.resize_u8(img, 368, 368)
        assert hashlib.sha256(ref.tobytes()).hexdigest() == str(golden["sha368"][i])
        if flip:
            ref = ref[:, ::-1]
        assert np.array_equal(out[i], ref), (img.shape, int((out[i] != ref).sum()))
    small = data.resize_images(dev, 96, flip=fl).cpu().numpy()
    for i in range(len(imgs)):
        ref = golden["r96_%d" % i][:, ::-1] if flip else golden["r96_%d" % i]
        assert np.array_equal(small[i], ref), imgs[i].shape
    idx = [int(i) for i in golden["r128x160_idx"]]
    rect = data.resize_images([dev[i] for i in idx], (128, 160), flip=fl[:len(idx)]).cpu().numpy()
    for j, i in enumerate(idx):
        ref = golden["r128x160_%d" % i][:, ::-1] if flip else golden["r128x160_%d" % i]
        assert np.array_equal(rect[j], ref), imgs[i].shape


def test_f32_is_normalised_u8(golden):
    from unipose_b200 import data
    dev = [torch.from_numpy(i).cuda() for i in _sources(golden)]
    flip = torch.tensor([i % 2 for i in range(len(dev))], device="cuda")
    u8 = data.resize_images(dev, 368, flip=flip)
    f32 = data.resize_images(dev, 368, flip=flip, out="f32")
    ref = (u8.permute(0, 3, 1, 2).float() - 128.0) / 256.0
    assert f32.shape == ref.shape and torch.equal(f32, ref)


@pytest.mark.parametrize("precision", ["fp16", "bf16", "fp32"])
def test_s2d_equals_pack_of_u8(golden, precision):
    from unipose_b200 import data, ops
    dev = [torch.from_numpy(i).cuda() for i in _sources(golden)]
    flip = torch.tensor([(i // 2) % 2 for i in range(len(dev))], device="cuda")
    n, s = len(dev), 368
    mode = ops.mode_of(precision)
    u8 = data.resize_images(dev, s, flip=flip)
    a = ops.Act(n, s // 2, s // 8 + 1, 64, mode, "cuda", zero=True)
    b = ops.Act(n, s // 2, s // 8 + 1, 64, mode, "cuda", zero=True)
    ops.pack_input_u8_s2d(u8, a, wpad_left=2)
    batch = data.ImageBatch(dev)
    batch.set_flip(flip)
    data.resize_into_s2d(batch, b, s, wpad_left=2)
    assert torch.equal(a.t.view(torch.int16), b.t.view(torch.int16))


def test_ragged_packed_batch_with_odd_pitches():
    """32 images of 4 sizes in one buffer, row pitches that are not multiples of 16 (byte-load staging)."""
    from unipose_b200 import data
    sizes = [(720, 1280, 3 * 1280 + 5), (333, 401, 3 * 401 + 1), (150, 200, 3 * 200 + 7), (480, 640, 3 * 640)]
    imgs, shapes, chunks = [], [], []
    for i in range(32):
        h, w, pitch = sizes[i % 4]
        img = P.synth_image(100 + i, h, w)
        rows = np.zeros((h, pitch), np.uint8)
        rows[:, :3 * w] = img.reshape(h, 3 * w)
        imgs.append(img)
        shapes.append((h, w, pitch))
        chunks.append(rows.reshape(-1))
    buf = torch.from_numpy(np.concatenate(chunks)).cuda()
    flip = torch.tensor([(i * 7) % 3 == 0 for i in range(32)], device="cuda")
    out = data.resize_images(buf, 368, flip=flip, shapes=shapes).cpu().numpy()
    for i, img in enumerate(imgs):
        ref, _, _ = P.prepare(img, 368, 368, flip=bool(flip[i]))
        assert np.array_equal(out[i], ref), (i, img.shape)
    # the same images as padded views of separate buffers
    views = [_padded(img, shapes[i][2]) for i, img in enumerate(imgs[:8])]
    out = data.resize_images(views, 368, flip=flip[:8]).cpu().numpy()
    for i in range(8):
        assert np.array_equal(out[i], P.prepare(imgs[i], 368, 368, flip=bool(flip[i]))[0]), i


@pytest.mark.parametrize("precision", ["fp16", "fp32"])
def test_forward_images_equals_forward_uint8_of_resized(precision):
    from unipose_b200 import data
    from unipose_b200.model.unipose import unipose
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        m = unipose(dataset="MPII", num_classes=16, precision=precision)
    m.load_state_dict(O.synth_state_dict(16, seed=0))
    m = m.cuda().eval()
    imgs = [P.synth_image(50 + i, h, w) for i, (h, w) in enumerate([(720, 1280), (150, 200), (257, 255)])]
    dev = [torch.from_numpy(i).cuda() for i in imgs]
    resized = torch.from_numpy(np.stack([P.resize_u8(i, 128, 128) for i in imgs])).cuda()
    assert torch.equal(data.resize_images(dev, 128), resized)
    a = m.forward_uint8(resized)
    for _ in range(2):       # the second call replays the captured plan
        b = m.forward_images(dev, size=128)
        assert torch.equal(a, b)


def test_prepare_batch_labels_vs_reference_path():
    from unipose_b200 import data
    sizes = [(720, 1280), (150, 200), (333, 401), (368, 368)]
    imgs = [P.synth_image(70 + i, h, w) for i, (h, w) in enumerate(sizes)]
    pts = [P.synth_points(70 + i, h, w, 14) for i, (h, w) in enumerate(sizes)]
    kpt = torch.from_numpy(np.stack([k for k, _ in pts])).cuda()
    center = torch.from_numpy(np.stack([c for _, c in pts])).cuda()
    flip = torch.tensor([True, False, True, True], device="cuda")
    res = data.prepare_batch([torch.from_numpy(i).cuda() for i in imgs], 368, flip=flip, kpts=kpt, center=center)
    assert res.heatmaps.shape == (4, 15, 46, 46) and res.centermap.shape == (4, 1, 46, 46)
    bad = 0
    for b, (img, (k, c)) in enumerate(zip(imgs, pts)):
        ref_img, rk, rc = P.prepare(img, 368, 368, flip=bool(flip[b]), kpt=k, center=c)
        assert np.array_equal(res.images[b].cpu().numpy(), ref_img)
        assert np.array_equal(res.kpts[b].cpu().numpy(), rk)
        assert np.array_equal(res.center[b].cpu().numpy(), rc)
        rh, rcm = E.reference_labels(rk, rc, 368, 368, 8, 3.0)
        heat = res.heatmaps[b].cpu().numpy()
        # as test_gpu_data: CUDA's and glibc's double exp may differ by 1 fp32 ulp after the store, very rarely
        assert np.abs(heat.astype(np.float64) - rh).max() <= 6e-8
        bad += int((heat != rh).sum())
        assert np.array_equal(res.centermap[b].cpu().numpy(), rcm)
    assert bad <= 2, bad
