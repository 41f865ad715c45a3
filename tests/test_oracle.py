"""CPU tests: the oracle (oracle/*.py) against the committed golden fixtures produced by the real reference
(oracle/make_golden.py)."""
import json
import os

import numpy as np
import pytest
import torch

from oracle import evaluate_oracle as E
from oracle import unipose_oracle as O

from conftest import GOLDEN


def _load(name):
    return np.load(os.path.join(GOLDEN, name))


def _close(a, b, rtol=2e-4, atol=2e-5):
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    scale = max(np.abs(b).mean(), 1e-6)
    assert a.shape == b.shape
    err = np.abs(a - b).max()
    assert err <= atol + rtol * scale, "max err %g (scale %g)" % (err, scale)


def test_state_dict_keys_match_reference_fixture():
    meta = json.load(open(os.path.join(GOLDEN, "state_dict_keys.json")))
    for video, key, k in ((False, "image_mpii_keys", 16), (True, "video_keys", 13)):
        specs = O.param_specs(k, video)
        assert [s[0] for s in specs] == list(meta[key].keys())
        for name, shape, _ in specs:
            assert list(shape) == meta[key][name], name
    assert len(meta["image_mpii_keys"]) == 687   # SURVEY.md §2: 687 state_dict entries


def test_oracle_image_model_vs_golden():
    g = _load("image_mpii_96.npz")
    sd = O.synth_state_dict(16, seed=0)
    x = O.synth_input(2, 96, 96, seed=0)
    with torch.no_grad():
        feat, low = O.resnet101_forward(x, sd)
        w = O.wasp_forward(feat, sd)
        heat = O.decoder_forward(w, low, sd)
    _close(feat[:, ::16].numpy(), g["feat_s"])
    _close(low[:, ::16, ::2, ::2].numpy(), g["low_s"])
    _close(w.numpy(), g["wasp"])
    _close(heat.numpy(), g["heat"])
    full = O.unipose_forward(x, sd, stride=4)
    _close(full[:, :, ::4, ::4].numpy(), _load("image_mpii_96_fullres.npz")["heat"])


def test_oracle_lsp_config1_vs_golden():
    sd = O.synth_state_dict(14, seed=1)
    with torch.no_grad():
        heat = O.unipose_forward(O.synth_input(1, 256, 256, seed=1), sd)
    assert heat.shape == (1, 15, 32, 32)
    _close(heat.numpy(), _load("image_lsp_256.npz")["heat"])


def test_oracle_config5_512_and_output_stride8_vs_golden():
    """Round-2 fixtures from the real reference: BASELINE.json configs[4] geometry (512x512, 17 joints) and the
    output_stride=8 variant (WASP dilations 48/36/24/12, layer3/4 dilated)."""
    with torch.no_grad():
        h5 = O.unipose_forward(O.synth_input(1, 512, 512, seed=5), O.synth_state_dict(17, seed=5))
        assert h5.shape == (1, 18, 64, 64)
        _close(h5.numpy(), _load("image_c5_512.npz")["heat"])
        sd8 = O.synth_state_dict(16, seed=8, output_stride=8)
        x8 = O.synth_input(2, 128, 128, seed=8)
        g8 = _load("image_os8_128.npz")
        f8, _ = O.resnet101_forward(x8, sd8, output_stride=8)
        _close(f8[:, ::16].numpy(), g8["feat_s"])
        _close(O.unipose_forward(x8, sd8, output_stride=8).numpy(), g8["heat"])


def _check_vs_crosscheck(forward, accuracy, seed, eval_seed):
    """forward(state_dict, x) and accuracy() against the reference's own MPII 64x64 forward and accuracy() outputs,
    stored by `oracle/make_golden.py --crosscheck`."""
    g = _load("crosscheck_mpii_64.npz")
    sd = O.synth_state_dict(16, seed=seed)
    with torch.no_grad():
        _close(forward(sd, O.synth_input(1, 64, 64, seed=seed)).numpy(), g["heat_seed%d" % seed], rtol=1e-5, atol=1e-6)
    gt, pred = E.synth_eval_inputs(4, 16, 48, seed=eval_seed)
    got = accuracy(pred, gt, 0.2, 0.5, "MPII")
    assert len(got) == 6
    for i, v in enumerate(got):
        np.testing.assert_allclose(np.asarray(v, dtype=np.float64), g["accuracy_seed%d_%d" % (eval_seed, i)],
                                   rtol=0, atol=1e-12)


def _oracle_forward(sd, x):
    return O.unipose_forward(x, sd)


def test_oracle_and_compiled_reference_vs_crosscheck_fixture():
    """The oracle port == the reference's outputs; so is oracle/_ref (the reference's own modules as byte-code, what
    bench.py's CPU arm times) where `oracle/build_ref.py` has built it."""
    from oracle import build_ref
    _check_vs_crosscheck(_oracle_forward, E.accuracy, 6, 22)
    if build_ref.have_ref():
        RefUnipose, _, ref_eval = build_ref.import_reference()

        def compiled_forward(sd, x):
            m = RefUnipose(dataset="MPII", num_classes=16).eval()
            m.load_state_dict(sd, strict=True)
            return m(x)

        _check_vs_crosscheck(compiled_forward, ref_eval.accuracy, 6, 22)


def test_oracle_video_vs_golden():
    g = _load("video_penn_368.npz")
    sd = O.synth_state_dict(13, video=True, seed=2)
    inp = O.synth_input(3, 368, 368, seed=2).view(1, 3, 3, 368, 368)
    cm = torch.from_numpy(E.gaussian_heatmaps(1, 3, 368, 368, seed=5, sigma=21.0)[:, 1:4]).view(1, 3, 1, 368, 368)
    heat = hide = cell = None
    with torch.no_grad():
        for it in range(2):
            heat, cell, hide = O.unipose_lstm_forward(inp, cm, it, heat, hide, cell, sd)
            _close(heat.numpy(), g["heat%d" % it])
            _close(cell.numpy(), g["cell%d" % it])
            _close(hide.numpy(), g["hide%d" % it])


@pytest.mark.parametrize("name,dataset,k,hw,n", [("mpii", "MPII", 16, 48, 8), ("lsp", "LSP", 14, 32, 4),
                                                 ("penn", "Penn_Action", 13, 46, 4)])
def test_evaluate_oracle_vs_golden(name, dataset, k, hw, n):
    g = _load("evaluate.npz")
    gt, pred = E.synth_eval_inputs(n, k, hw)
    acc, PCK, PCKh, cnt, p, vis = E.accuracy(pred, gt, 0.2, 0.5, dataset)
    preds, maxvals = E.get_max_preds(pred)
    assert np.array_equal(preds, g[name + "_preds"])          # integer joint indices: bit exact
    assert np.array_equal(maxvals, g[name + "_maxvals"])
    assert np.array_equal(p, g[name + "_preds"])
    assert cnt == int(g[name + "_cnt"])
    np.testing.assert_allclose(acc, g[name + "_acc"], rtol=0, atol=1e-12)
    np.testing.assert_allclose(PCK, g[name + "_PCK"], rtol=0, atol=1e-12)
    np.testing.assert_allclose(PCKh, g[name + "_PCKh"], rtol=0, atol=1e-12)
    np.testing.assert_array_equal(vis, g[name + "_visible"])
    # planted edge cases: all-zero map is masked, tie resolves to the first occurrence
    assert preds[0, 3].tolist() == [0.0, 0.0]
    assert preds[1, 5].tolist() == [9.0, 7.0]


def test_label_oracle_vs_reference_golden():
    """reference_labels restates utils/mpii_data.py:165-181; the fixture was produced with the reference's own
    guassian_kernel (oracle/make_golden.py --round2)."""
    g = _load("labels_mpii.npz")
    kpts, center = E.synth_keypoints(4, 16, 368, 368, seed=40)
    for b in range(4):
        heat, cm = E.reference_labels(kpts[b], center[b], 368, 368, 8, 3)
        assert np.array_equal(heat, g["heat"][b]) and np.array_equal(cm, g["centermap"][b])
    assert g["heat"].shape == (4, 17, 46, 46) and float(g["heat"][:, 1:].max()) == 1.0


def test_get_kpts_oracle():
    m = np.zeros((1, 3, 46, 46), np.float32)
    m[0, 1, 10, 20] = 1
    m[0, 2, 45, 0] = 2
    assert E.get_kpts(m) == [[int(20 * 368.0 / 46), int(10 * 368.0 / 46)], [0, int(45 * 368.0 / 46)]]


def test_oracle_vs_reference_crosscheck_fixture():
    _check_vs_crosscheck(_oracle_forward, E.accuracy, 3, 21)
