"""CPU checks of the input step's oracle (oracle/image_prep_oracle.py) against cv2.resize and the reference's hflip
transforms (stored in tests/golden/resize_cv2.npz, and live where cv2 is importable), and of the UpImageJob layout
the device kernel (csrc/image_prep.cu) reads."""
import ctypes
import hashlib
import os
import re

import numpy as np
import pytest
import torch

from conftest import GOLDEN, ROOT
from oracle import image_prep_oracle as P
from unipose_b200 import _lib


@pytest.fixture(scope="module")
def golden():
    return np.load(os.path.join(GOLDEN, "resize_cv2.npz"))


def test_oracle_resize_equals_cv2_fixture(golden):
    idx128 = set(int(i) for i in golden["r128x160_idx"])
    for i, (h, w, seed) in enumerate(golden["sizes"]):
        img = P.synth_image(int(seed), int(h), int(w))
        assert np.array_equal(P.resize_u8(img, 96, 96), golden["r96_%d" % i]), (h, w)
        if i in idx128:
            assert np.array_equal(P.resize_u8(img, 128, 160), golden["r128x160_%d" % i]), (h, w)
        sha = hashlib.sha256(P.resize_u8(img, 368, 368).tobytes()).hexdigest()
        assert sha == str(golden["sha368"][i]), (h, w)


@pytest.mark.parametrize("name,pairs,invisible", [("lsp", P.SWAP_PAIRS, False), ("ntid", P.SWAP_PAIRS, True),
                                                  ("bbc", P.SWAP_PAIRS_BBC, True)])
def test_oracle_hflip_equals_reference_fixture(golden, name, pairs, invisible):
    kpt, center = golden["kpt_" + name], golden["center_" + name]
    assert (kpt[:, 2] == 0).any() and (kpt[:, 2] == 1).any()
    k, c = P.hflip_points(kpt, center, 368, pairs, invisible)
    assert np.array_equal(k, golden["hflip_%s_kpt" % name])
    assert np.array_equal(c, golden["hflip_%s_center" % name])


def test_oracle_point_scaling_matches_torch_float32():
    """mpii_data.py:160-161 multiplies a float32 tensor by a Python float: float32(x) * float32(368 / w)."""
    kpt, _ = P.synth_points(3, 720, 1280, 16)
    ref = torch.from_numpy(kpt.copy())
    ref[:, 0] = ref[:, 0] * (368 / 1280)
    ref[:, 1] = ref[:, 1] * (368 / 720)
    assert np.array_equal(P.scale_points(kpt, 720, 1280, 368, 368), ref.numpy())


def test_oracle_resize_equals_live_cv2():
    cv2 = pytest.importorskip("cv2")
    rng = np.random.default_rng(1234)
    cases = [(int(rng.integers(1, 1100)), int(rng.integers(1, 1100)), 16 * int(rng.integers(1, 30)),
              16 * int(rng.integers(1, 30))) for _ in range(40)]
    cases += [(2 * 48, 2 * 64, 48, 64), (48, 64, 48, 64), (1, 1, 16, 16), (3, 2, 32, 48)]
    for h, w, oh, ow in cases:
        img = P.synth_image(h * 7 + w, h, w)
        assert np.array_equal(P.resize_u8(img, oh, ow), cv2.resize(img, (ow, oh))), (h, w, oh, ow)


def test_image_job_layout_matches_header():
    src = open(os.path.join(ROOT, "include", "unipose_b200.h")).read()
    body = re.search(r"typedef struct UpImageJob \{(.*?)\} UpImageJob;", src, re.S).group(1)
    fields = re.findall(r"(\S+)\s*\*?\s*(\w+(?:\s*,\s*\w+)*);", re.sub(r"/\*.*?\*/", "", body, flags=re.S))
    names = [n.strip() for _t, ns in fields for n in ns.split(",")]
    assert names == [f for f, _ in _lib.UpImageJob._fields_]
    assert ctypes.sizeof(_lib.UpImageJob) == 24
    assert _lib.UpImageJob.flip.offset == 20 and _lib.UpImageJob.h.offset == 8


def test_resize_rejects_bad_jobs_before_launch():
    """Argument checks run on the host copy of the table, so they need no GPU."""
    lib = _lib.load()
    jobs = (_lib.UpImageJob * 2)()
    for j in jobs:
        j.src, j.h, j.w, j.pitch = 4096, 10, 10, 30
    dev = ctypes.c_void_p(4096)
    y = ctypes.c_void_p(4096)

    def call(n=2, oh=368, ow=368, fmt=_lib.UP_RESIZE_OUT_U8):
        return lib.up_resize_pack_u8(jobs, dev, n, oh, ow, fmt, y, 0, 0, 0, 128.0, 256.0, None)

    jobs[1].w = 0
    assert call() == -1 and b"image 1 is empty" in lib.up_last_error()
    jobs[1].w, jobs[1].src = 10, None
    assert call() == -1 and b"null source" in lib.up_last_error()
    jobs[1].src, jobs[1].pitch = 4096, 29
    assert call() == -1 and b"pitch" in lib.up_last_error()
    jobs[1].pitch = 30
    assert call(oh=360) == -1 and b"multiples of 16" in lib.up_last_error()
    assert call(fmt=5) == -1 and b"out_format" in lib.up_last_error()
    assert lib.up_resize_pack_u8(None, dev, 2, 368, 368, 8, y, 0, 0, 0, 128.0, 256.0, None) == -1
    assert b"null argument" in lib.up_last_error()
