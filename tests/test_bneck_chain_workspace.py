"""CPU test of the fused bottleneck run's workspace (csrc/bneck_chain.cu): it holds one release/acquire counter per
(image group, block, 64-channel chunk of T1) plus the exit counter, for the layer3 shapes the GPU tests and the
benchmark run.  up_bneck_chain_workspace_bytes is host-only code, so no GPU is needed."""
import ctypes

import pytest

from unipose_b200 import _lib

NBLOCKS = 22      # layer3 blocks 1..22 of the ResNet-101


def _pick_tile(n, h, w, tile_px=128):
    """Python mirror of pick_tile (csrc/up_conv_host.h): images per 128-pixel tile."""
    best, bn, bh, bw = -1, 1, 8, 16
    cw = 1
    while cw <= tile_px:
        chh = 1
        while cw * chh <= tile_px:
            cn = tile_px // (cw * chh)
            if cn <= 256:
                cost = -(-w // cw) * -(-h // chh) * -(-n // cn)
                if best < 0 or cost < best or (cost == best and (cw > bw or (cw == bw and chh > bh))):
                    best, bn, bh, bw = cost, cn, chh, cw
            chh *= 2
        cw *= 2
    return bn


def _desc(n, hw, dil, dtype):
    d = _lib.UpBneckChainDesc()
    d.n, d.h, d.w, d.planes, d.nblocks, d.dil, d.dtype = n, hw, hw, 256, NBLOCKS, dil, dtype
    return d


# (batch, layer3 map, dilation): the network inputs of tests/test_gpu_bneck_chain.py at output stride 16 / 8, and the
# benchmark's batch 32 at 384^2
@pytest.mark.parametrize("n,hw,dil", [(4, 24, 1), (2, 32, 1), (2, 16, 1), (2, 48, 2), (4, 23, 1), (32, 24, 1)])
@pytest.mark.parametrize("dtype", [_lib.UP_FP16, _lib.UP_BF16])
def test_workspace_holds_a_counter_per_block_and_chunk(n, hw, dil, dtype):
    lib = _lib.load()
    d = _desc(n, hw, dil, dtype)
    got = int(lib.up_bneck_chain_workspace_bytes(ctypes.byref(d)))
    tiles_n = n // _pick_tile(n, hw, hw)
    need = (tiles_n * (NBLOCKS + 1) * 4 + 1) * 4
    assert got >= need, (n, hw, tiles_n, got, need)
    assert got % 256 == 0 and got < need + 256, (got, need)
