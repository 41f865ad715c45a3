"""GPU input / label pipeline - the steps either side of the hot path (SURVEY.md 8f3).

* `gaussian_heatmaps` / `center_map`: the ground-truth synthesis of the reference's datasets
  (utils/mpii_data.py:165-181, same code in lsp_lspet_data.py / bbc_data.py / penn_action_data.py) on the device,
  bit-for-bit (float64 Gaussian, clipping, fp32 store, background channel).
* uint8 images go straight into the network through `unipose.forward_uint8` (model/unipose.py): normalisation
  `(x - 128) / 256` (mpii_data.py:184-185) is fused into the stem's input packing.
* `resize_images` / `prepare_batch`: the step in front of both - decoded uint8 images of any sizes ->
  `cv2.resize(img, (368, 368))` (mpii_data.py:159-162, lsp_lspet_data.py:211) bit for bit, the optional
  Mytransforms.hflip (Mytransforms.py:501-519), and the matching key-point / centre transform, in one launch
  (csrc/image_prep.cu).  `unipose.forward_images` writes the same resize straight into the stem's input.
"""
from __future__ import annotations

import ctypes
from typing import NamedTuple, Optional, Sequence

import torch

from . import _lib, ops

SWAP_PAIRS = ((0, 5), (1, 4), (2, 3), (6, 11), (7, 10), (8, 9))   # Mytransforms.hflip / hflip_NTID (LSP order)
SWAP_PAIRS_BBC = ((1, 2), (3, 4), (5, 6))                           # Mytransforms.hflip_BBC
_OUT_FORMATS = {"u8": _lib.UP_RESIZE_OUT_U8, "f32": _lib.UP_RESIZE_OUT_F32}


def _out_size(size) -> tuple:
    s_h, s_w = (size, size) if isinstance(size, int) else (int(size[0]), int(size[1]))
    if s_h <= 0 or s_w <= 0 or s_h % 16 or s_w % 16:
        raise ValueError("output size must be positive multiples of 16 (the stem's requirement); got %dx%d" % (s_h, s_w))
    return s_h, s_w


class ImageBatch:
    """A ragged batch of uint8 HWC (3-channel) device images as the kernel's job table.

    `images` is a list of CUDA tensors [h, w, 3] (rows may be padded: strides (pitch, 3, 1)), or one uint8 CUDA
    buffer with `shapes` = [(h, w) or (h, w, pitch), ...] of images stored back to back (each h * pitch bytes,
    pitch = 3 * w when omitted).  The caller keeps the source memory alive until the launches that read it have run."""

    def __init__(self, images, shapes: Optional[Sequence] = None):
        entries = []
        if shapes is None:
            if isinstance(images, torch.Tensor):
                raise TypeError("pass a list of [h, w, 3] images, or a packed buffer together with `shapes`")
            for i, t in enumerate(images):
                ops.require_cuda(t, "image %d" % i)
                if t.dtype != torch.uint8 or t.dim() != 3 or t.shape[2] != 3 or t.stride(2) != 1 or t.stride(1) != 3:
                    raise ValueError("image %d must be uint8 [h, w, 3] with packed pixels; got %s %s strides %s"
                                     % (i, t.dtype, tuple(t.shape), t.stride()))
                entries.append((t.data_ptr(), t.shape[0], t.shape[1], t.stride(0) if t.shape[0] > 1 else 3 * t.shape[1]))
            device = images[0].device if len(images) else None
        else:
            ops.require_cuda(images, "image buffer")
            if images.dtype != torch.uint8 or not images.is_contiguous():
                raise ValueError("the packed image buffer must be a contiguous uint8 tensor")
            off, base, end = 0, images.data_ptr(), images.numel()
            for i, s in enumerate(shapes):
                h, w = int(s[0]), int(s[1])
                pitch = int(s[2]) if len(s) > 2 else 3 * w
                if off + max(h, 0) * pitch > end:
                    raise ValueError("image %d (%dx%d, pitch %d) runs past the end of the buffer" % (i, h, w, pitch))
                entries.append((base + off, h, w, pitch))
                off += max(h, 0) * pitch
            device = images.device
        if not entries:
            raise ValueError("empty image batch")
        self.n = len(entries)
        self.device = device
        self.sizes = [(h, w) for _p, h, w, _q in entries]
        self.host = (_lib.UpImageJob * self.n)()
        for j, (p, h, w, pitch) in zip(self.host, entries):
            j.src, j.h, j.w, j.pitch, j.flip = p, h, w, pitch, 0
        raw = torch.frombuffer(bytearray(bytes(self.host)), dtype=torch.int32).view(self.n, ctypes.sizeof(_lib.UpImageJob) // 4)
        self.dev = raw.to(device)

    def set_flip(self, flip) -> None:
        """Per-image mirror flags (bool / int tensor or sequence of n); stays on the device, no host round trip."""
        if flip is None:
            self.dev[:, 5] = 0
            return
        f = torch.as_tensor(flip, device=self.device).reshape(-1)
        if f.numel() != self.n:
            raise ValueError("flip has %d entries for %d images" % (f.numel(), self.n))
        self.dev[:, 5] = (f != 0).to(torch.int32)

    def launch(self, out_h: int, out_w: int, out_format: int, y_ptr, plane_stride: int = 0, wpitch: int = 0,
               wpad_left: int = 0, mean: float = 128.0, std: float = 256.0) -> None:
        with torch.cuda.device(self.device):
            _lib.call("up_resize_pack_u8", self.host, ops._ptr(self.dev), self.n, out_h, out_w, out_format, y_ptr,
                      plane_stride, wpitch, wpad_left, float(mean), float(std), ops._stream())


def resize_images(images, size=368, flip=None, out: str = "u8", shapes: Optional[Sequence] = None,
                  mean: float = 128.0, std: float = 256.0) -> torch.Tensor:
    """cv2.resize(img, (S_w, S_h)) of every image, bit for bit, then the mirror where `flip` is set.
    out="u8": uint8 [n, S_h, S_w, 3]; out="f32": (x - mean) / std as fp32 NCHW [n, 3, S_h, S_w] (the reference's
    network input, Mytransforms.normalize)."""
    s_h, s_w = _out_size(size)
    if out not in _OUT_FORMATS:
        raise ValueError("out must be one of %s (got %r)" % (sorted(_OUT_FORMATS), out))
    batch = images if isinstance(images, ImageBatch) else ImageBatch(images, shapes)
    batch.set_flip(flip)
    if out == "u8":
        y = torch.empty((batch.n, s_h, s_w, 3), dtype=torch.uint8, device=batch.device)
    else:
        y = torch.empty((batch.n, 3, s_h, s_w), dtype=torch.float32, device=batch.device)
    batch.launch(s_h, s_w, _OUT_FORMATS[out], ops._ptr(y), mean=mean, std=std)
    return y


def resize_into_s2d(batch: ImageBatch, y: "ops.Act", size, wpad_left: int = 0, mean: float = 128.0,
                    std: float = 256.0) -> None:
    """The resize written as the stem's normalised space-to-depth input (the layout of ops.pack_input_u8_s2d)."""
    s_h, s_w = _out_size(size)
    assert (y.n, y.h) == (batch.n, s_h // 2) and y.c % 16 == 0
    wpitch = y.w * (y.c // 16)
    assert wpitch >= s_w // 2 + wpad_left
    batch.launch(s_h, s_w, y.mode, y.ptr(), y.plane_stride, wpitch, wpad_left, mean, std)


def transform_points(pts: torch.Tensor, sizes, size, flip=None, swap_pairs=SWAP_PAIRS,
                     flip_invisible: bool = False) -> torch.Tensor:
    """Key-points [n, k, 2 or 3] (x, y(, visibility)) or centres [n, 2] in source pixels -> network-input pixels.

    Scale as mpii_data.py:159-161 (float32 x * float32(S_w / w)), then, for the images with `flip`, Mytransforms.hflip:
    x = S_w - 1 - x where visibility == 1 (every point with `flip_invisible`, as hflip_NTID / hflip_BBC, and every
    point of a tensor without a visibility column), then swap the `swap_pairs` (key-points only: a [n, 2] centre is
    always mirrored and never swapped)."""
    ops.require_cuda(pts, "points")
    s_h, s_w = _out_size(size)
    center = pts.dim() == 2
    p = pts.detach().to(torch.float32).clone()
    if center:
        p = p.unsqueeze(1)
    if p.dim() != 3 or p.shape[2] < 2 or p.shape[0] != len(sizes):
        raise ValueError("points must be [n, k, >=2] or [n, 2] with n = %d; got %s" % (len(sizes), tuple(pts.shape)))
    fx = torch.tensor([s_w / w for _h, w in sizes], dtype=torch.float32, device=p.device)
    fy = torch.tensor([s_h / h for h, _w in sizes], dtype=torch.float32, device=p.device)
    p[:, :, 0] *= fx[:, None]
    p[:, :, 1] *= fy[:, None]
    if flip is not None:
        f = torch.as_tensor(flip, device=p.device).reshape(-1, 1) != 0
        mirror = f
        if not center and not flip_invisible and p.shape[2] > 2:
            mirror = f & (p[:, :, 2] == 1)
        p[:, :, 0] = torch.where(mirror, (s_w - 1) - p[:, :, 0], p[:, :, 0])
        if not center and swap_pairs:
            perm = list(range(p.shape[1]))
            for a, b in swap_pairs:
                perm[a], perm[b] = perm[b], perm[a]
            p = torch.where(f[:, :, None], p[:, perm], p)
    return p[:, 0] if center else p


class PreparedBatch(NamedTuple):
    images: torch.Tensor                    # uint8 [n, S_h, S_w, 3] or fp32 [n, 3, S_h, S_w]
    kpts: Optional[torch.Tensor]            # [n, k, >=2] in network-input pixels
    center: Optional[torch.Tensor]          # [n, 2]
    heatmaps: Optional[torch.Tensor]        # [n, k + 1, S_h / stride, S_w / stride] (background channel 0)
    centermap: Optional[torch.Tensor]       # [n, 1, S_h / stride, S_w / stride]


def prepare_batch(images, size=368, flip=None, kpts=None, center=None, swap_pairs=SWAP_PAIRS,
                  flip_invisible: bool = False, out: str = "u8", shapes: Optional[Sequence] = None,
                  stride: int = 8, sigma: float = 3.0) -> PreparedBatch:
    """A batch of decoded images of any sizes -> the network input and its training labels, all on the device:
    resize (+ flip) as `resize_images`, key-points / centres as `transform_points`, then the heat-maps
    (`gaussian_heatmaps`) and the centre map (`center_map`) of mpii_data.py:165-181.  `flip` is a per-image bool
    tensor drawn by the caller (RandomHorizontalFlip's coin, Mytransforms.py:564-587)."""
    s_h, s_w = _out_size(size)
    batch = ImageBatch(images, shapes)
    out_images = resize_images(batch, (s_h, s_w), flip=flip, out=out)
    k = c = heat = cmap = None
    if kpts is not None:
        k = transform_points(kpts, batch.sizes, (s_h, s_w), flip, swap_pairs, flip_invisible)
        heat = gaussian_heatmaps(k, s_h, s_w, stride, sigma)
    if center is not None:
        c = transform_points(center, batch.sizes, (s_h, s_w), flip)
        cmap = center_map(c, s_h, s_w, stride)
    return PreparedBatch(out_images, k, c, heat, cmap)


def _kpts(t: torch.Tensor) -> torch.Tensor:
    ops.require_cuda(t, "key-points")
    t = t.detach().float().contiguous()
    if t.dim() != 3 or t.shape[2] < 2:
        raise ValueError("key-points must be [n, k, 2(+)] (x, y in input-image pixels); got %s" % (tuple(t.shape),))
    return t[:, :, :2].contiguous()


def gaussian_heatmaps(kpts: torch.Tensor, height: int, width: int, stride: int = 8, sigma: float = 3.0,
                      background: bool = True) -> torch.Tensor:
    """[n, k(+1), height/stride, width/stride] fp32 heat-maps for key-points given in input-image pixels
    (height x width = the network input, 368 x 368 in the reference)."""
    k = _kpts(kpts)
    n, nk = k.shape[:2]
    h, w = int(height / stride), int(width / stride)
    out = torch.empty((n, nk + (1 if background else 0), h, w), dtype=torch.float32, device=k.device)
    with torch.cuda.device(k.device):
        _lib.call("up_gaussian_labels", ops._ptr(k), ops._ptr(out), n, nk, h, w, float(stride), float(sigma),
                  1 if background else 0, 1, ops._stream())
    return out


def center_map(center: torch.Tensor, height: int, width: int, stride: int = 8, sigma: float = 3.0) -> torch.Tensor:
    """[n, 1, height/stride, width/stride] centre map (mpii_data.py:177-181: Gaussian at int(center / stride))."""
    c = center.detach().float().reshape(center.shape[0], 1, -1)
    k = _kpts(c)
    n = k.shape[0]
    h, w = int(height / stride), int(width / stride)
    out = torch.empty((n, 1, h, w), dtype=torch.float32, device=k.device)
    with torch.cuda.device(k.device):
        _lib.call("up_gaussian_labels", ops._ptr(k), ops._ptr(out), n, 1, h, w, float(stride), float(sigma), 0, 2,
                  ops._stream())
    return out
