"""Write tests/golden/resize_cv2.npz: what cv2.resize and the reference's hflip transforms produce on seeded inputs.
Run where cv2 and the reference sources are importable:

    python oracle/make_resize_golden.py

Source images are not stored: the tests regenerate them with image_prep_oracle.synth_image(seed, h, w).  Stored:
  sizes          [m, 3] (h, w, seed) of the sources
  r96_<i>        cv2.resize(img_i, (96, 96)) for every source
  r128x160_<i>   cv2.resize(img_i, (160, 128)) for the sources listed in r128x160_idx
  sha368         [m] SHA-256 (hex) of cv2.resize(img_i, (368, 368)).tobytes()
  kpt_<name>, center_<name>, width_<name>   inputs of the key-point flips (float32; visibility 0 / 1)
  hflip_<name>_kpt, hflip_<name>_center     Mytransforms.hflip / hflip_NTID / hflip_BBC on those inputs
"""
from __future__ import annotations

import hashlib
import importlib.util
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = "/root/reference"
OUT = os.path.join(ROOT, "tests", "golden", "resize_cv2.npz")
sys.path.insert(0, ROOT)

from oracle import image_prep_oracle as P  # noqa: E402

# downscales (MPII 1280x720, 1080p, odd), upscales, odd and degenerate sizes, the target size itself, exactly twice it
SIZES = [(720, 1280, 1), (1080, 1920, 2), (333, 401, 3), (150, 200, 4), (368, 368, 5), (736, 736, 6), (97, 1, 7),
         (1, 75, 8), (41, 59, 9), (500, 300, 10), (192, 320, 11), (257, 255, 12)]
R128_IDX = [0, 3, 8]


def _mytransforms():
    spec = importlib.util.spec_from_file_location("ref_mytransforms", os.path.join(REF, "utils", "Mytransforms.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def main() -> None:
    import cv2
    out = {"sizes": np.array(SIZES, dtype=np.int64), "r128x160_idx": np.array(R128_IDX, dtype=np.int64)}
    sha = []
    for i, (h, w, seed) in enumerate(SIZES):
        img = P.synth_image(seed, h, w)
        out["r96_%d" % i] = cv2.resize(img, (96, 96))
        if i in R128_IDX:
            out["r128x160_%d" % i] = cv2.resize(img, (160, 128))
        sha.append(hashlib.sha256(np.ascontiguousarray(cv2.resize(img, (368, 368))).tobytes()).hexdigest())
    out["sha368"] = np.array(sha)
    T = _mytransforms()
    # The loaders keep key-points as lists (lsp_lspet_data.read_mat_file: .tolist()); float32 elements keep the
    # arithmetic in float32.  A dummy image carries the width.
    for name, fn, k, seed in (("lsp", T.hflip, 14, 20), ("ntid", T.hflip_NTID, 14, 21), ("bbc", T.hflip_BBC, 7, 22)):
        kpt, center = P.synth_points(seed, 368, 368, k)
        kpt[0, 2], kpt[1, 2] = 0, 1            # at least one invisible and one visible joint
        img = np.zeros((4, 368, 3), np.uint8)
        klist = [[np.float32(v) for v in row] for row in kpt]
        clist = [np.float32(v) for v in center]
        _img, k2, c2 = fn(img, klist, clist)
        out["kpt_" + name], out["center_" + name] = kpt, center
        out["hflip_%s_kpt" % name] = np.array(k2, dtype=np.float32)
        out["hflip_%s_center" % name] = np.array(c2, dtype=np.float32)
    np.savez_compressed(OUT, **out)
    print("wrote %s (%d bytes)" % (OUT, os.path.getsize(OUT)))


if __name__ == "__main__":
    main()
