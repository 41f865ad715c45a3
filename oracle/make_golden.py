"""Generate tests/golden/*.npz by running the UNMODIFIED reference (imported read-only from
/root/reference) on seeded synthetic weights / inputs.  Run in the build container only:

    python oracle/make_golden.py

The GPU box has no /root/reference; tests there compare against the committed fixtures.
Inputs and weights are NOT stored: they are regenerated from seeds by oracle.unipose_oracle
(synth_state_dict / synth_input), which is itself checked here key-for-key against the reference
modules' own state_dict.
"""
from __future__ import annotations

import importlib.util
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = "/root/reference"
OUT = os.path.join(ROOT, "tests", "golden")
sys.path.insert(0, ROOT)

from oracle import evaluate_oracle as E  # noqa: E402
from oracle import unipose_oracle as O  # noqa: E402


def import_reference():
    if REF not in sys.path:
        sys.path.insert(0, REF)
    from model.modules.backbone import resnet
    resnet.model_zoo.load_url = lambda *a, **k: {}  # offline: resnet.py:142 would download ImageNet weights
    from model.unipose import unipose as RefUnipose
    import model.uniposeLSTM as ref_lstm
    spec = importlib.util.spec_from_file_location("ref_evaluate", os.path.join(REF, "utils", "evaluate.py"))
    ref_eval = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(ref_eval)
    return RefUnipose, ref_lstm, ref_eval


def check_specs(model, num_classes, video):
    ref_sd = model.state_dict()
    specs = O.param_specs(num_classes, video)
    keys = [k for k, _, _ in specs]
    assert keys == list(ref_sd.keys()), "state_dict key order differs from the reference"
    for k, shape, _ in specs:
        assert tuple(ref_sd[k].shape) == tuple(shape), (k, tuple(ref_sd[k].shape), shape)
    return {k: list(s) for k, s, _ in specs}


def round2_fixtures():
    """Fixtures added in round 2 (the round-1 files are left untouched): BASELINE.json configs[4] geometry
    (512x512, 17 joints -> 32x32 WASP map, 64x64 heat-maps) and the output_stride=8 variant (layer3/4 dilated,
    WASP dilations 48/36/24/12: wasp.py:41-42, resnet.py:54-56)."""
    os.makedirs(OUT, exist_ok=True)
    torch.set_grad_enabled(False)
    RefUnipose, _ref_lstm, _ref_eval = import_reference()
    m5 = RefUnipose(dataset="COCO", num_classes=17).eval()
    m5.load_state_dict(O.synth_state_dict(17, seed=5), strict=True)
    x5 = O.synth_input(1, 512, 512, seed=5)
    np.savez_compressed(os.path.join(OUT, "image_c5_512.npz"), heat=m5(x5).numpy())
    m8 = RefUnipose(dataset="MPII", num_classes=16, output_stride=8).eval()
    sd8 = O.synth_state_dict(16, seed=8, output_stride=8)
    assert list(sd8.keys()) == list(m8.state_dict().keys())
    m8.load_state_dict(sd8, strict=True)
    x8 = O.synth_input(2, 128, 128, seed=8)
    f8, l8 = m8.backbone(x8)
    np.savez_compressed(os.path.join(OUT, "image_os8_128.npz"), heat=m8(x8).numpy(), feat_s=f8[:, ::16].numpy())
    # ---- label synthesis: the reference's own guassian_kernel (utils/mpii_data.py:62-65) driven through the loop of
    # mpii.__getitem__ (:165-181).  The module imports utils.Mytransforms (whose package pulls matplotlib): stubbed.
    import types
    pkg = types.ModuleType("utils")
    pkg.__path__ = []
    sys.modules.setdefault("utils", pkg)
    sys.modules.setdefault("utils.Mytransforms", types.ModuleType("utils.Mytransforms"))
    spec = importlib.util.spec_from_file_location("ref_mpii_data", os.path.join(REF, "utils", "mpii_data.py"))
    ref_data = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(ref_data)
    kpts, center = E.synth_keypoints(4, 16, 368, 368, seed=40)
    heat = np.zeros((4, 17, 46, 46), np.float32)
    cmap = np.zeros((4, 1, 46, 46), np.float32)
    for b in range(4):
        hm = np.zeros((46, 46, 17), dtype=np.float32)
        kp = torch.Tensor(kpts[b])
        ce = torch.Tensor(center[b])
        for i in range(len(kp)):                                     # mpii_data.py:166-173
            x = int(kp[i][0]) * 1.0 / 8
            y = int(kp[i][1]) * 1.0 / 8
            g = ref_data.guassian_kernel(size_h=46, size_w=46, center_x=x, center_y=y, sigma=3)
            g[g > 1] = 1
            g[g < 0.0099] = 0
            hm[:, :, i + 1] = g
        hm[:, :, 0] = 1.0 - np.max(hm[:, :, 1:], axis=2)             # :175
        c = ref_data.guassian_kernel(size_h=46, size_w=46, center_x=int(ce[0] / 8), center_y=int(ce[1] / 8), sigma=3)
        c[c > 1] = 1
        c[c < 0.0099] = 0
        heat[b] = hm.transpose(2, 0, 1)
        cmap[b, 0] = c
    np.savez_compressed(os.path.join(OUT, "labels_mpii.npz"), heat=heat, centermap=cmap)
    for fn in ("image_c5_512.npz", "image_os8_128.npz", "labels_mpii.npz"):
        print("%-32s %8.1f KB" % (fn, os.path.getsize(os.path.join(OUT, fn)) / 1024))


def crosscheck_fixtures():
    """The reference's own outputs for the oracle cross-checks of tests/test_oracle.py, so that they run without the
    reference: MPII forward at 64x64 (seeds 3 and 6) and utils/evaluate.py accuracy() (seeds 21 and 22)."""
    os.makedirs(OUT, exist_ok=True)
    torch.set_grad_enabled(False)
    RefUnipose, _ref_lstm, ref_eval = import_reference()
    out = {}
    for seed in (3, 6):
        torch.manual_seed(0)
        m = RefUnipose(dataset="MPII", num_classes=16).eval()
        m.load_state_dict(O.synth_state_dict(16, seed=seed), strict=True)
        out["heat_seed%d" % seed] = m(O.synth_input(1, 64, 64, seed=seed)).numpy()
    for seed in (21, 22):
        gt, pred = E.synth_eval_inputs(4, 16, 48, seed=seed)
        for i, v in enumerate(ref_eval.accuracy(pred, gt, 0.2, 0.5, "MPII")):
            out["accuracy_seed%d_%d" % (seed, i)] = np.asarray(v, dtype=np.float64)
    np.savez_compressed(os.path.join(OUT, "crosscheck_mpii_64.npz"), **out)
    print("%-32s %8.1f KB" % ("crosscheck_mpii_64.npz", os.path.getsize(os.path.join(OUT, "crosscheck_mpii_64.npz")) / 1024))


def main():
    if "--round2" in sys.argv:
        return round2_fixtures()
    if "--crosscheck" in sys.argv:
        return crosscheck_fixtures()
    os.makedirs(OUT, exist_ok=True)
    torch.manual_seed(0)
    torch.set_grad_enabled(False)
    RefUnipose, ref_lstm, ref_eval = import_reference()
    meta = {}

    # ---- image model, MPII (16 joints) ----
    m = RefUnipose(dataset="MPII", num_classes=16).eval()
    meta["image_mpii_keys"] = check_specs(m, 16, False)
    sd = O.synth_state_dict(16, video=False, seed=0)
    m.load_state_dict(sd, strict=True)
    x = O.synth_input(2, 96, 96, seed=0)
    feat, low = m.backbone(x)
    w = m.wasp(feat)
    heat = m.decoder(w, low)
    assert torch.equal(heat, m(x))
    np.savez_compressed(os.path.join(OUT, "image_mpii_96.npz"),
                        heat=heat.numpy(), wasp=w.numpy(),
                        feat_s=feat[:, ::16].numpy(), low_s=low[:, ::16, ::2, ::2].numpy())
    # stride != 8 path (model/unipose.py:31-32)
    m.stride = 4
    np.savez_compressed(os.path.join(OUT, "image_mpii_96_fullres.npz"), heat=m(x)[:, :, ::4, ::4].numpy())
    m.stride = 8

    # ---- config 1: LSP 256x256 bs1 (14 joints) ----
    m1 = RefUnipose(dataset="LSP", num_classes=14).eval()
    sd1 = O.synth_state_dict(14, video=False, seed=1)
    m1.load_state_dict(sd1, strict=True)
    x1 = O.synth_input(1, 256, 256, seed=1)
    np.savez_compressed(os.path.join(OUT, "image_lsp_256.npz"), heat=m1(x1).numpy())

    # ---- video model (13 joints), two frames, composed from the reference's own sub-modules because
    # uniposeLSTM.unipose.forward hard-codes .cuda() (model/uniposeLSTM.py:99-104) ----
    mv = ref_lstm.unipose(num_classes=13).eval()
    meta["video_keys"] = check_specs(mv, 13, True)
    sdv = O.synth_state_dict(13, video=True, seed=2)
    mv.load_state_dict(sdv, strict=True)
    inp = O.synth_input(3, 368, 368, seed=2).view(1, 3, 3, 368, 368)  # [B=1, T=3, 3, H, W]
    cm = torch.from_numpy(E.gaussian_heatmaps(1, 3, 368, 368, seed=5, sigma=21.0)[:, 1:4]).view(1, 3, 1, 368, 368)
    outs = {}
    hide = cell = None
    F = torch.nn.functional
    for it in range(3):
        fx, flow = mv.backbone(inp[:, it])
        t = mv.decoder(mv.wasp(fx), flow)
        c = mv.pool_center(cm[:, it])
        cat = torch.cat((t, c), dim=1)
        if it == 0:
            cell, hide = mv.lstm_0(cat)
        else:
            cell, hide = mv.lstm(cat, hide, cell)
        hm = F.relu(mv.conv1(hide))
        hm = F.relu(mv.conv2(hm))
        hm = F.relu(mv.conv3(hm))
        hm = F.relu(mv.conv4(hm))
        hm = F.relu(mv.conv5(hm))
        outs["heat%d" % it] = hm.numpy()
        outs["cell%d" % it] = cell.numpy()
        outs["hide%d" % it] = hide.numpy()
        # the trunk heat-maps only scale the state tolerance of the GPU test: their max-abs keeps the file under 1 MB
        outs["trunk%d_absmax" % it] = np.float32(t.abs().max())
    np.savez_compressed(os.path.join(OUT, "video_penn_368.npz"), **outs)

    # ---- evaluation path: utils/evaluate.py on identical synthetic heat-maps ----
    ev = {}
    for name, dataset, k, hw, n in [("mpii", "MPII", 16, 48, 8), ("lsp", "LSP", 14, 32, 4),
                                    ("penn", "Penn_Action", 13, 46, 4)]:
        gt, pred = E.synth_eval_inputs(n, k, hw)
        acc, PCK, PCKh, cnt, p, vis = ref_eval.accuracy(pred, gt, 0.2, 0.5, dataset)
        preds, maxvals = ref_eval.get_max_preds(pred)
        ev.update({name + "_acc": acc, name + "_PCK": PCK,
                   name + "_PCKh": PCKh, name + "_cnt": np.int64(cnt), name + "_preds": preds,
                   name + "_maxvals": maxvals, name + "_visible": vis})
    np.savez_compressed(os.path.join(OUT, "evaluate.npz"), **ev)

    with open(os.path.join(OUT, "state_dict_keys.json"), "w") as f:
        json.dump(meta, f)
    for fn in sorted(os.listdir(OUT)):
        print("%-32s %8.1f KB" % (fn, os.path.getsize(os.path.join(OUT, fn)) / 1024))


if __name__ == "__main__":
    main()
