"""Dilated ResNet-101 backbone on tcgen05 implicit-GEMM convs.

Mirrors model/modules/backbone/resnet.py of the reference (Bottleneck :5-42, ResNet :44-150,
ResNet101 :152-160): same attribute names -> same state_dict keys; same initialisation
(normal(0, sqrt(2/(k*k*out))) convs, BN weight 1 / bias 0, resnet.py:126-136).  forward() does not run
torch ops: every conv+BN(+residual)+ReLU is ONE fused kernel launch recorded into an engine.Plan.
"""
import math
import os
import warnings

import torch
import torch.nn as nn

from ....plan_module import PlanModule

_IMAGENET_FILE = 'resnet101-5d3b4d8f.pth'   # what resnet.py:142 downloads


def _gather_like(loops_fn, name, w):
    """Apply a pure regrouping of filter elements (defined by slice copies in `loops_fn`) as ONE gather: the index map
    (0 = structural zero) is derived once per (co, device) by pushing element numbers through the definition, so a call
    costs three kernels instead of ~100 - it runs at every weight refresh, i.e. every step of a training plan."""
    key = (name, w.shape[0], str(w.device))
    idx = _GATHER_INDEX.get(key)
    if idx is None:
        numbered = torch.arange(1, w.numel() + 1, dtype=torch.float64).reshape(w.shape)
        idx = loops_fn(numbered).long().to(w.device)
        _GATHER_INDEX[key] = idx
    return torch.cat([w.new_zeros(1), w.reshape(-1)])[idx]


_GATHER_INDEX = {}


def stem_s2d_weight(w):
    """[co,3,7,7] stride-2 stem filter -> [co,16,4,4] stride-1 filter over the 2x2 space-to-depth image
    (channel order (ph,pw,c), taps at offsets -2..1; up_pack_input_s2d produces the matching activations)."""
    return _gather_like(_stem_s2d_loops, "s2d", w)


def _stem_s2d_loops(w):
    w2 = w.new_zeros((w.shape[0], 16, 4, 4))
    for a in range(4):
        for ph in range(2):
            kh = 2 * (a - 2) + ph + 3
            if not 0 <= kh < 7:
                continue
            for bb in range(4):
                for pw in range(2):
                    kw = 2 * (bb - 2) + pw + 3
                    if 0 <= kw < 7:
                        c0 = (ph * 2 + pw) * 3
                        w2[:, c0:c0 + 3, a, bb] = w[:, :, kh, kw]
    return w2


def stem_window_weight(w):
    """[co,3,7,7] -> [co,64,4,1]: filter rows stay taps, the 4 horizontal taps x 16 s2d channels become the K-chunk."""
    w2 = stem_s2d_weight(w)                                    # [co, 16, kh', kw']
    return w2.permute(0, 3, 1, 2).reshape(w.shape[0], 64, 4, 1).contiguous()   # cin index = kw' * 16 + ch


def _stem_superpixel_loops(w):
    """Definition of the super-pixel regrouping (see stem_superpixel_weight) as explicit slice copies."""
    w2 = _stem_s2d_loops(w)                                    # [co, 16, a, b]
    co = w.shape[0]
    out = w.new_zeros((4 * co, 64, 4, 2))
    for j in range(4):
        for kw in range(2):
            for pp in range(4):
                b = 4 * kw + pp - j
                if 0 <= b < 4:
                    out[j * co:(j + 1) * co, pp * 16:(pp + 1) * 16, :, kw] = w2[:, :, :, b]
    return out


def stem_superpixel_weight(w):
    """[co,3,7,7] stride-2 stem filter -> [4*co, 64, 4, 2]: an ORDINARY 4x2 stride-1 convolution that produces four
    horizontally adjacent output pixels (x = 4s .. 4s+3) at once from the space-to-depth image regrouped into
    "super pixels" of 4 s2d pixels x 16 channels = 64 contiguous elements (128 aligned bytes).

    Output channel j*co + o is output pixel 4s+j, channel o; input element p*16 + ch of tap (a, kw) is s2d pixel
    4(s+kw) + p - 2 (the rows carry 2 zero pixels of left padding), i.e. horizontal s2d tap b = 4*kw + p - j."""
    return _gather_like(_stem_superpixel_loops, "superpixel", w)


class Bottleneck(PlanModule):
    expansion = 4

    def __init__(self, inplanes, planes, stride=1, dilation=1, downsample=None, BatchNorm=None):
        super().__init__()
        self.conv1 = nn.Conv2d(inplanes, planes, kernel_size=1, bias=False)
        self.bn1 = BatchNorm(planes)
        self.conv2 = nn.Conv2d(planes, planes, kernel_size=3, stride=stride, dilation=dilation,
                               padding=dilation, bias=False)
        self.bn2 = BatchNorm(planes)
        self.conv3 = nn.Conv2d(planes, planes * 4, kernel_size=1, bias=False)
        self.bn3 = BatchNorm(planes * 4)
        self.downsample = downsample
        self.stride, self.dilation = stride, dilation
        self._out_channels = (planes * 4,)

    def _emit(self, b, x, t1=None, nxt=None):
        """t1: this block's conv1 output when the PREVIOUS block's tail kernel already produced it; nxt: the following
        bottleneck - when this block ends in the tail kernel and qualifies, that kernel also runs nxt.conv1 and the
        result is left in self._next_t1 for the caller to hand on."""
        n, h, w = x.n, x.h, x.w
        planes = self.conv1.out_channels
        s, d = self.stride, self.dilation
        ho, wo = (h - 1) // s + 1, (w - 1) // s + 1
        self._next_t1 = None
        if t1 is None:
            t1 = b.act(n, h, w, planes)
            b.conv(x, b.packed_conv(self.conv1, self.bn1), t1, "bottleneck.conv1", relu=True)
        out = b.act(n, ho, wo, planes * 4)
        if self.downsample is not None and s == 1 and self._emit_tail(b, t1, x, out, proj=self.downsample, nxt=nxt):
            return out          # projection shortcut folded into the tail kernel: Wd x never goes to memory
        res = x
        pcp = self._packed_conv3_proj(b, x) if self.downsample is not None else None
        if pcp is not None:
            t2 = b.act(n, ho, wo, planes)
            b.conv(t1, b.packed_conv(self.conv2, self.bn2), t2, "bottleneck.conv2", stride=s, dil=d, pad=d, relu=True)
            b.conv(t2, pcp, out, "bottleneck.conv3+proj", relu=True, proj=(x, s))
            return out
        if self.downsample is not None:
            res = b.act(n, ho, wo, planes * 4)
            b.conv(x, b.packed_conv(self.downsample[0], self.downsample[1]), res, "bottleneck.downsample",
                   stride=s, pad=0)
        if self._emit_tail(b, t1, res, out, nxt=nxt):
            return out
        t2 = b.act(n, ho, wo, planes)
        b.conv(t1, b.packed_conv(self.conv2, self.bn2), t2, "bottleneck.conv2", stride=s, dil=d, pad=d, relu=True)
        b.conv(t2, b.packed_conv(self.conv3, self.bn3), out, "bottleneck.conv3", relu=True, residual=res)
        return out

    def _packed_conv3_proj(self, b, x):
        """conv3 and the projection shortcut (`downsample`: 1x1 conv of stride s + BN, resnet.py:36-37,75-79) as ONE
        GEMM: out = ReLU([W3*s3 | Wd*sd] . [t2 ; x_strided] + (shift3 + shiftd)) - K grows by the block's input
        channels, the shortcut tensor and the downsample launch disappear (UP_FLAG_PROJ).  Returns the packed filter
        [1 + inplanes / planes][cout][planes] or None when the shape does not qualify."""
        from .... import engine, ops
        conv_d, bn_d = self.downsample[0], self.downsample[1]
        planes, s = self.conv1.out_channels, self.stride
        cout = 4 * planes
        if (os.environ.get("UNIPOSE_B200_PROJ_FUSE", "1") == "0" or b.mode == ops.UP_SPLIT or planes % 64 or
                not isinstance(x, ops.Act) or x.c != conv_d.in_channels or x.c % planes or s not in (1, 2) or
                x.h % s or x.w % s or conv_d.kernel_size != (1, 1) or conv_d.stride != (s, s) or
                conv_d.bias is not None or conv_d.out_channels != cout):
            return None
        pt = x.c // planes
        dev, f32 = b.device, torch.float32
        wbuf = torch.empty((1, 1 + pt, cout, planes), dtype=torch.float16 if b.mode == ops.UP_FP16 else torch.bfloat16,
                           device=dev)
        pc3 = b.packed_conv(self.conv3, self.bn3, wbuf=wbuf[:, 0:1])
        fold_d = torch.empty(bn_d.num_features, dtype=f32, device=dev)
        scale_d, shift_d, shift_sum = (torch.empty(cout, dtype=f32, device=dev) for _ in range(3))
        wt = b.plan.weights
        wt.add_epilogue(scale_d, shift_d, cout, bn=bn_d, fold_scale=fold_d)
        for j in range(pt):          # slice j of the projection's input channels = filter "tap" 1 + j
            wt.add_pack(lambda: engine._param(conv_d, "weight"), wbuf[0, 1 + j], cout, planes, ci_off=j * planes, cin_slice=planes,
                        row_scale=fold_d, scale_period=bn_d.num_features)
        # both shifts are table outputs: the sum follows every table refresh (changed or replaced BatchNorm tensors)
        b.plan.pack_jobs.append(engine._PackJob((), lambda: torch.add(pc3.shift, shift_d, out=shift_sum), with_table=True))
        b.plan.buffers.append((wbuf, scale_d, shift_d, fold_d))
        return ops.PackedConv(wbuf, pc3.scale, shift_sum, 1, 1, cout, planes, cout, planes, b.mode)

    def _emit_tail(self, b, t1, res, out, proj=None, nxt=None):
        """conv2 (3x3) + conv3 (1x1 expansion) + residual + ReLU as ONE launch (csrc/bneck_tail.cu) for the
        bandwidth-bound layers (planes 64 / 128, stride 1, fp16 / bf16): t2 never leaves shared memory.
        proj = the block's `downsample` (1x1 conv + BN, stride 1): `res` is the block INPUT and the projection is
        computed inside the kernel (UNIPOSE_B200_BNECK_TAIL_PROJ=0: separate launch as before).
        nxt = the following bottleneck: at planes 64 its conv1 + bn1 + ReLU (1x1, stride 1, 64 or 128 outputs) runs in
        the same kernel on the output tile while it is on chip (UNIPOSE_B200_TAIL_CONV1=0: its own launch)."""
        import ctypes
        from .... import _lib, ops
        planes = self.conv1.out_channels
        if (os.environ.get("UNIPOSE_B200_BNECK_TAIL", "1") == "0" or b.mode == ops.UP_SPLIT or self.stride != 1 or
                planes not in (64, 128) or not isinstance(res, ops.Act) or t1.c != planes):
            return False
        if proj is None:
            if res.c != 4 * planes:
                return False
        elif (os.environ.get("UNIPOSE_B200_BNECK_TAIL_PROJ", "1") == "0" or res.c % 64 != 0 or
              proj[0].in_channels != res.c or proj[0].kernel_size != (1, 1) or proj[0].stride != (1, 1)):
            return False
        d = _lib.UpBneckTailDesc()
        d.n, d.h, d.w, d.planes, d.dil, d.dtype = t1.n, t1.h, t1.w, planes, self.dilation, b.mode
        d.proj_cin = res.c if proj is not None else 0
        c1n = nxt.conv1 if nxt is not None else None
        if (c1n is not None and os.environ.get("UNIPOSE_B200_TAIL_CONV1", "1") != "0" and planes == 64 and
                c1n.kernel_size == (1, 1) and c1n.stride == (1, 1) and c1n.in_channels == 4 * planes and
                c1n.out_channels in (64, 128) and c1n.bias is None):
            d.next_planes = c1n.out_channels
        if _lib.load().up_bneck_tail_supported(ctypes.byref(d)) != 0:
            return False
        pc2 = b.packed_conv(self.conv2, self.bn2)
        pc3 = b.packed_conv(self.conv3, self.bn3)
        pcd = b.packed_conv(proj[0], proj[1]) if proj is not None else None
        pc1n = t1n = None
        if d.next_planes:
            pc1n = b.packed_conv(nxt.conv1, nxt.bn1)
            t1n = b.act(t1.n, t1.h, t1.w, d.next_planes)
            self._next_t1 = t1n

        def launch(keep=(pc2, pc3, pcd, pc1n)):
            _lib.call("up_bneck_tail_fwd", ctypes.byref(d), t1.ptr(), ops._ptr(pc2.w), ops._ptr(pc2.shift), ops._ptr(pc3.w),
                      ops._ptr(pc3.shift), res.ptr(), ops._ptr(pcd.w) if pcd else None,
                      ops._ptr(pcd.shift) if pcd else None, out.ptr(), ops._ptr(pc1n.w) if pc1n else None,
                      ops._ptr(pc1n.shift) if pc1n else None, t1n.ptr() if t1n is not None else None, ops._stream())
        b.add(launch, "bottleneck.tail+conv1" if pc1n else "bottleneck.tail")
        return True


class ResNet(PlanModule):
    def __init__(self, block, layers, output_stride, BatchNorm, pretrained=True):
        super().__init__()
        self.inplanes = 64
        if output_stride == 16:
            strides, dilations = [1, 2, 2, 1], [1, 1, 1, 2]
        elif output_stride == 8:
            strides, dilations = [1, 2, 1, 1], [1, 1, 2, 4]
        else:
            raise NotImplementedError
        self.conv1 = nn.Conv2d(3, 64, kernel_size=7, stride=2, padding=3, bias=False)
        self.bn1 = BatchNorm(64)
        self.layer1 = self._stack(block, 64, [dilations[0]] * layers[0], strides[0], BatchNorm)
        self.layer2 = self._stack(block, 128, [dilations[1]] * layers[1], strides[1], BatchNorm)
        self.layer3 = self._stack(block, 256, [dilations[2]] * layers[2], strides[2], BatchNorm)
        # multi-grid unit: dilation x [1, 2, 4] (resnet.py:49,70,94-111)
        self.layer4 = self._stack(block, 512, [m * dilations[3] for m in (1, 2, 4)], strides[3], BatchNorm)
        self._out_channels = (2048, 256)
        self._init_weight()
        if pretrained:
            self._load_pretrained_model()

    def _stack(self, block, planes, dils, stride, BatchNorm):
        down = None
        if stride != 1 or self.inplanes != planes * block.expansion:
            down = nn.Sequential(nn.Conv2d(self.inplanes, planes * block.expansion, kernel_size=1, stride=stride,
                                           bias=False), BatchNorm(planes * block.expansion))
        blocks = [block(self.inplanes, planes, stride, dils[0], down, BatchNorm)]
        self.inplanes = planes * block.expansion
        blocks += [block(self.inplanes, planes, 1, d, None, BatchNorm) for d in dils[1:]]
        return nn.Sequential(*blocks)

    def _init_weight(self):
        for m in self.modules():
            if isinstance(m, nn.Conv2d):
                n = m.kernel_size[0] * m.kernel_size[1] * m.out_channels
                m.weight.data.normal_(0, math.sqrt(2. / n))
            elif isinstance(m, nn.BatchNorm2d):
                m.weight.data.fill_(1)
                m.bias.data.zero_()

    def _load_pretrained_model(self):
        """The reference downloads the torchvision ImageNet ResNet-101 here (resnet.py:138-150).  Offline, the
        file is used when it already sits in the torch hub cache; otherwise the random init stays."""
        path = os.path.join(torch.hub.get_dir(), 'checkpoints', _IMAGENET_FILE)
        if not os.path.exists(path):
            warnings.warn('unipose_b200: %s not in the torch hub cache - backbone keeps its random init' % path)
            return
        pretrain = torch.load(path, map_location='cpu')
        own = self.state_dict()
        own.update({k: v for k, v in pretrain.items() if k in own})
        self.load_state_dict(own)

    # image entry point: fp32 NCHW -> 2x2 space-to-depth NHWC (instead of the generic NCHW->NHWC copy)
    def _input_channels_pad(self, idx, c):
        return 16

    def _emit_image(self, b, x_static, s2d_shape=None):
        """x_static: fp32 NCHW [n,3,h,w] (the reference's input) or uint8 NHWC [n,h,w,3] (raw images; normalised
        (x-128)/256 while packing, utils/mpii_data.py:184-185).  x_static None with s2d_shape = (n, h, w): the plan
        starts at the stem convolution and the caller writes its space-to-depth input, b.plan.s2d_input, before each
        run (unipose.forward_images)."""
        from .... import ops
        u8 = x_static is not None and x_static.dtype == torch.uint8
        if x_static is None:
            n, h, w = s2d_shape
        elif u8:
            n, h, w, _ = x_static.shape
        else:
            n, _, h, w = x_static.shape
        if h % 16 or w % 16:
            raise ValueError('unipose_b200: input height/width must be multiples of 16 (got %dx%d)' % (h, w))
        # Super-pixel stem: the 2x2 space-to-depth image (16 channels, rows padded by 2 zero pixels on the left) is
        # read as [n, h/2, w/8 + 1, 64] - four s2d pixels per 128-byte "super pixel" - and the 7x7/s2 conv becomes a
        # plain 4x2 stride-1 conv with 4*64 outputs = four adjacent output pixels (stem_superpixel_weight).  Every
        # activation row the TMA fetches is 128 aligned bytes and is shared by 4 outputs.
        ws = w // 8
        x2 = b.act(n, h // 2, ws + 1, 64, zero=True)
        if x_static is None:
            b.plan.s2d_input = x2
        elif u8:
            b.add(lambda x_static=x_static, x2=x2: ops.pack_input_u8_s2d(x_static, x2, wpad_left=2), "pack_input_u8_s2d")
        else:
            b.add(lambda x_static=x_static, x2=x2: ops.pack_input_s2d(x_static, x2, wpad_left=2), "pack_input_s2d")
        stem = b.act(n, h // 2, w // 2, 64)
        pc = b.packed_conv(self.conv1, self.bn1, cin_pad=64, weight_fn=stem_superpixel_weight)
        b.conv(x2, pc, stem.reshaped(h // 2, ws, 256), "stem", pad=(2, 0), relu=True, ho=h // 2, wo=ws)
        x = b.act(n, h // 4, w // 4, 64)
        b.add(lambda stem=stem, x=x: ops.maxpool3x3s2(stem, x), "maxpool")
        low = None
        names = ('layer1', 'layer2', 'layer3', 'layer4')
        t1 = None          # conv1 output of the block about to be emitted, when the previous tail kernel produced it
        for li, name in enumerate(names):
            blocks = list(getattr(self, name))
            i = 0
            while i < len(blocks):
                run = self._chain_run(blocks, i)
                fused = self._emit_chain(b, x, blocks[i:i + run]) if (run >= 2 and t1 is None) else None
                if fused is not None:
                    x = fused
                    i += run
                else:
                    nxt = blocks[i + 1] if i + 1 < len(blocks) else (
                        getattr(self, names[li + 1])[0] if li + 1 < len(names) else None)
                    blk = blocks[i]
                    x = blk._emit(b, x, t1=t1, nxt=nxt)
                    t1 = blk._next_t1
                    i += 1
            if name == 'layer1':
                low = x
        return x, low

    # ---- runs of identical bottlenecks as one persistent kernel (csrc/bneck_chain.cu) ----
    @staticmethod
    def _chain_run(blocks, i):
        """Length of the run of blocks starting at i that the fused kernel takes: planes 256, stride 1, no downsample
        path, same dilation."""
        def ok(blk):
            return (blk.downsample is None and blk.stride == 1 and blk.conv1.out_channels == 256 and
                    blk.conv1.in_channels == 1024)
        if not ok(blocks[i]):
            return 0
        j = i
        while j < len(blocks) and ok(blocks[j]) and blocks[j].dilation == blocks[i].dilation:
            j += 1
        return j - i

    def _emit_chain(self, b, x, blocks):
        import ctypes
        from .... import _lib, ops
        if os.environ.get("UNIPOSE_B200_BNECK_CHAIN", "1") == "0" or b.mode == ops.UP_SPLIT:
            return None
        nb = len(blocks)
        d = _lib.UpBneckChainDesc()
        d.n, d.h, d.w, d.planes, d.nblocks, d.dil, d.dtype = x.n, x.h, x.w, 256, nb, blocks[0].dilation, b.mode
        if x.c != 1024 or _lib.load().up_bneck_chain_supported(ctypes.byref(d)) != 0:
            return None      # odd batch, tiny maps, more tiles than CTA pairs: the layer-wise plan takes every shape
        dt = torch.float16 if b.mode == ops.UP_FP16 else torch.bfloat16
        dev = b.device
        w1 = torch.empty((nb, 256, 1024), dtype=dt, device=dev)
        w2 = torch.empty((nb, 9, 256, 256), dtype=dt, device=dev)
        w3 = torch.empty((nb, 1024, 256), dtype=dt, device=dev)
        s1, s2, s3 = (torch.empty((nb, c), dtype=torch.float32, device=dev) for c in (256, 256, 1024))
        sc = [torch.empty((nb, c), dtype=torch.float32, device=dev) for c in (256, 256, 1024)]   # epilogue scales (all 1)
        for i, blk in enumerate(blocks):
            b.packed_conv(blk.conv1, blk.bn1, wbuf=w1[i].view(1, 1, 256, 1024), scale=sc[0][i], shift=s1[i])
            b.packed_conv(blk.conv2, blk.bn2, wbuf=w2[i].view(1, 9, 256, 256), scale=sc[1][i], shift=s2[i])
            b.packed_conv(blk.conv3, blk.bn3, wbuf=w3[i].view(1, 1, 1024, 256), scale=sc[2][i], shift=s3[i])
        xb = b.act(x.n, x.h, x.w, 1024)
        t1 = b.act(2 * x.n, x.h, x.w, 256)
        ws_bytes = int(_lib.load().up_bneck_chain_workspace_bytes(ctypes.byref(d)))
        ws = b.tensor((ws_bytes,), dtype=torch.uint8, zero=True)
        wts = _lib.UpBneckChainWeights()
        wts.w1, wts.w2, wts.w3 = w1.data_ptr(), w2.data_ptr(), w3.data_ptr()
        wts.shift1, wts.shift2, wts.shift3 = s1.data_ptr(), s2.data_ptr(), s3.data_ptr()
        keep = (w1, w2, w3, s1, s2, s3, sc, ws)

        def launch(keep=keep):
            _lib.call("up_bneck_chain_fwd", ctypes.byref(d), ctypes.byref(wts), x.ptr(), xb.ptr(), t1.ptr(), ops._ptr(ws),
                      ws_bytes, ops._stream())
        b.add(launch, "bottleneck.chain[%d]" % nb)
        return x if nb % 2 == 0 else xb

    def forward(self, input):
        from .... import engine, ops
        self._check_inputs([input])
        self._bn_eval_only()
        key = (tuple(input.shape), self._precision(), input.device.index)
        plan = self._plans.get(key)
        if plan is None:
            plan = engine.Plan(input.device, self._precision())
            b = plan.builder
            st = plan.static_input(tuple(input.shape))
            x, low = self._emit_image(b, st)
            outs = []
            for a, c in ((x, 2048), (low, 256)):
                dst = b.tensor((a.n, c, a.h, a.w))
                b.add(lambda a=a, c=c, dst=dst: ops.act_to_nchw(a, c, dst), "nhwc_to_nchw")
                outs.append(dst)
            plan.finalize(outs)
            self._plans[key] = plan
        x, low = plan.run(input.detach().float())
        return x.clone(), low.clone()


def ResNet101(output_stride, BatchNorm, pretrained=True):
    return ResNet(Bottleneck, [3, 4, 23, 3], output_stride, BatchNorm, pretrained=pretrained)
