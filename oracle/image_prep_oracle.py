"""numpy restatement of the reference's input step (the thing csrc/image_prep.cu reproduces on the device):

* `resize_u8`: `cv2.resize(img, (S_w, S_h))` of an 8-bit HWC image, i.e. OpenCV's INTER_LINEAR fixed-point path, bit
  for bit (utils/mpii_data.py:159-162, utils/lsp_lspet_data.py:211).  The rules, settled against cv2 4.13:
    - coordinates: scale = 1 / (dst / src) in double, f = float32((d + 0.5) * scale - 0.5), s = floor(f), f -= s;
    - columns: s < 0 -> (s, f) = (0, 0); s >= w - 1 -> (s, f) = (w - 1, 0);
    - rows keep their fraction; only the two source row indices are clamped to [0, h - 1];
    - weights: c0 = round((1 - f) * 2048), c1 = round(f * 2048) (round half to even, float32 products);
    - horizontal pass in int32: row = S[s] * a0 + S[s + 1] * a1;
    - vertical pass, the SIMD formula: ((row0 >> 4) * b0 >> 16) + ((row1 >> 4) * b1 >> 16), then (v + 2) >> 2,
      saturated to uint8;
    - a source exactly twice the target in both dimensions takes cv2's INTER_AREA fast path instead:
      (sum of the 2x2 block + 2) >> 2;
    - a source of the target's size is copied.
* `hflip_points` (+ the image mirror in `prepare`): Mytransforms.hflip / hflip_NTID / hflip_BBC
  (utils/Mytransforms.py:501-562) applied after the resize: mirror the image, x = S_w - 1 - x (visible joints only
  unless `flip_invisible`), swap the left/right pairs, always mirror the centre.
* `scale_points`: kpt[:, 0] *= S_w / w, kpt[:, 1] *= S_h / h in float32 (mpii_data.py:159-161), the centre alike.
"""
from __future__ import annotations

import numpy as np

COEF_BITS = 11
COEF_ONE = 1 << COEF_BITS          # INTER_RESIZE_COEF_SCALE
SWAP_PAIRS = ((0, 5), (1, 4), (2, 3), (6, 11), (7, 10), (8, 9))   # Mytransforms.hflip / hflip_NTID
SWAP_PAIRS_BBC = ((1, 2), (3, 4), (5, 6))                           # Mytransforms.hflip_BBC


def coords(src: int, dst: int, clamp_fraction: bool):
    """Source index and fixed-point weights (c0, c1) per destination index along one axis."""
    scale = 1.0 / (float(dst) / float(src))
    f = ((np.arange(dst, dtype=np.float64) + 0.5) * scale - 0.5).astype(np.float32)
    s = np.floor(f).astype(np.int64)
    f = (f - s.astype(np.float32)).astype(np.float32)
    if clamp_fraction:
        lo = s < 0
        f[lo], s[lo] = 0, 0
        hi = s >= src - 1
        f[hi], s[hi] = 0, src - 1
    c0 = np.rint((np.float32(1) - f) * np.float32(COEF_ONE)).astype(np.int64)
    c1 = np.rint(f * np.float32(COEF_ONE)).astype(np.int64)
    return s, c0, c1


def resize_u8(img: np.ndarray, out_h: int, out_w: int) -> np.ndarray:
    """cv2.resize(img, (out_w, out_h)) for uint8 [h, w, c] (INTER_LINEAR)."""
    assert img.dtype == np.uint8 and img.ndim == 3
    h, w, _ = img.shape
    if (h, w) == (out_h, out_w):
        return img.copy()
    if (h, w) == (2 * out_h, 2 * out_w):
        s = img.astype(np.int64)
        v = s[0::2, 0::2] + s[0::2, 1::2] + s[1::2, 0::2] + s[1::2, 1::2]
        return ((v + 2) >> 2).astype(np.uint8)
    sx, a0, a1 = coords(w, out_w, clamp_fraction=True)
    sy, b0, b1 = coords(h, out_h, clamp_fraction=False)
    sx1 = np.minimum(sx + 1, w - 1)             # a1 == 0 wherever sx + 1 would leave the image
    src = img.astype(np.int64)
    rows = src[:, sx] * a0[None, :, None] + src[:, sx1] * a1[None, :, None]       # [h, out_w, c] int32 range
    r0 = rows[np.clip(sy, 0, h - 1)] >> 4
    r1 = rows[np.clip(sy + 1, 0, h - 1)] >> 4
    v = ((r0 * b0[:, None, None]) >> 16) + ((r1 * b1[:, None, None]) >> 16)
    return np.clip((v + 2) >> 2, 0, 255).astype(np.uint8)


def scale_points(pts: np.ndarray, h: int, w: int, out_h: int, out_w: int) -> np.ndarray:
    """[..., >=2] float32 points in source pixels -> network-input pixels (float32 product, as the reference's
    float32 tensor times a Python float)."""
    p = np.array(pts, dtype=np.float32, copy=True)
    p[..., 0] = p[..., 0] * np.float32(out_w / w)
    p[..., 1] = p[..., 1] * np.float32(out_h / h)
    return p


def hflip_points(kpt, center, width: int, swap_pairs=SWAP_PAIRS, flip_invisible=False):
    """Mytransforms.hflip (flip_invisible=False) / hflip_NTID, hflip_BBC (True) on float32 key-points [k, 3]
    (x, y, visibility) and centre [2] of an image `width` pixels wide; returns new arrays."""
    k = np.array(kpt, dtype=np.float32, copy=True)
    c = np.array(center, dtype=np.float32, copy=True)
    m = np.ones(len(k), dtype=bool) if flip_invisible else (k[:, 2] == 1)
    k[m, 0] = np.float32(width - 1) - k[m, 0]
    c[0] = np.float32(width - 1) - c[0]
    for a, b in swap_pairs:
        k[[a, b]] = k[[b, a]]
    return k, c


def prepare(img, out_h, out_w, flip=False, kpt=None, center=None, swap_pairs=SWAP_PAIRS, flip_invisible=False):
    """One image through the whole step: resize, scale the points, then (optionally) flip both."""
    h, w = img.shape[:2]
    out = resize_u8(img, out_h, out_w)
    k = None if kpt is None else scale_points(kpt, h, w, out_h, out_w)
    c = None if center is None else scale_points(center, h, w, out_h, out_w)
    if flip:
        out = np.ascontiguousarray(out[:, ::-1])
        if k is not None:
            k, c = hflip_points(k, c if c is not None else np.zeros(2, np.float32), out_w, swap_pairs, flip_invisible)
    return out, k, c


def synth_image(seed: int, h: int, w: int) -> np.ndarray:
    """Seeded uint8 HWC test image: a smooth gradient plus noise, so both flat and busy regions are exercised."""
    rng = np.random.default_rng(seed)
    yy, xx = np.mgrid[0:h, 0:w]
    base = (xx * 255.0 / max(w - 1, 1))[..., None] * np.array([1.0, 0.5, 0.0]) + \
        (yy * 255.0 / max(h - 1, 1))[..., None] * np.array([0.0, 0.5, 1.0])
    noise = rng.integers(-40, 41, size=(h, w, 3))
    return np.clip(base + noise, 0, 255).astype(np.uint8)


def synth_points(seed: int, h: int, w: int, k: int = 14):
    """Seeded key-points [k, 3] (x, y, visibility in {0, 1}) inside an h x w image, and a centre [2]."""
    rng = np.random.default_rng(seed + 1000)
    kpt = np.zeros((k, 3), dtype=np.float32)
    kpt[:, 0] = rng.uniform(0, w - 1, k)
    kpt[:, 1] = rng.uniform(0, h - 1, k)
    kpt[:, 2] = (rng.random(k) < 0.75).astype(np.float32)
    center = np.array([rng.uniform(0, w - 1), rng.uniform(0, h - 1)], dtype=np.float32)
    return kpt, center
