"""In-kernel phase timeline of the fused bottleneck run (UP_DEBUG_TIMING=1 -> globaltimer stamps per CTA) and its
total time against the layer-wise launches."""
import os, sys, warnings, ctypes
os.environ["UP_DEBUG_TIMING"] = "1"
os.environ.setdefault("UNIPOSE_B200_GRAPH", "0")
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch
from unipose_b200 import _lib, engine, synth
from unipose_b200.model.unipose import unipose

n = int(sys.argv[1]) if len(sys.argv) > 1 else 32
hw = int(sys.argv[2]) if len(sys.argv) > 2 else 24
with warnings.catch_warnings():
    warnings.simplefilter("ignore")
    m = unipose(dataset="MPII", num_classes=16, precision="fp16")
synth.trained_like_init_(m, 0)
m = m.cuda().eval()
blocks = list(m.backbone.layer3)[1:]


def build(chain):
    os.environ["UNIPOSE_B200_BNECK_CHAIN"] = "1" if chain else "0"
    plan = engine.Plan(torch.device("cuda:0"), "fp16", use_graph=False)
    b = plan.builder
    x = b.act(n, hw, hw, 1024)
    x.t.copy_(torch.randn(x.t.shape, device="cuda").clamp_min_(0) * 0.5)
    if chain:
        out = m.backbone._emit_chain(b, x, blocks)
    else:
        out = x
        for blk in blocks:
            out = blk._emit(b, out)
    plan.finalize([])
    return plan


flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
for chain in (False, True):
    plan = build(chain)
    for _ in range(3):
        plan.run()
    torch.cuda.synchronize()
    tot = 0.0
    for _ in range(5):
        flush.zero_()
        a, b_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        plan.run()
        b_.record()
        torch.cuda.synchronize()
        tot += a.elapsed_time(b_)
    print("%s: %d launches, %.1f us for %d blocks (eager launches, L2 flushed)" % (
        "chain" if chain else "layer-wise", plan.launches, tot / 5 * 1e3, len(blocks)))
names = {0: "entry", 1: "deps", 31: "exit"}
for b in range(3):
    names[23 + b] = "b%d_conv2_first_mma" % b      # centre tap of chunks 0-1 issued (staged t1 tile)
    names[26 + b] = "b%d_halo_c0_mma" % b          # first halo MMA (chunk 0) issued: counter[b][0] complete + TMA
    names[5 + b] = "b%d_conv2_issued" % b
    names[8 + b] = "b%d_p3_issued" % b
    names[11 + b] = "b%d_t2_epi_done" % b
    names[14 + b] = "b%d_p3_epi_done" % b
    names[17 + b] = "b%d_t1next_epi_done" % b
buf = (ctypes.c_ulonglong * (160 * 32))()
_lib.call("up_debug_bneck_timing", buf)
t = np.array(buf, dtype=np.float64).reshape(160, 32)
t = t[t[:, 0] > 0]
t0 = t[:, 0].min()
print("CTAs", len(t))
order = [0, 1] + [k + b for b in range(3) for k in (23, 26, 5, 11, 8, 14, 17)] + [31]
for k in order:
    col = t[:, k]
    col = col[col > 0]
    if len(col) == 0:
        continue
    r = (col - t0) / 1e3
    print("%-20s n=%3d  min %8.2f  med %8.2f  max %8.2f us" % (names[k], len(r), r.min(), np.median(r), r.max()))
