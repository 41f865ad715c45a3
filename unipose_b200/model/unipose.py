"""UniPose single-image model — drop-in for model/unipose.py of the reference (class unipose :8-65):
same constructor, same forward(input) -> [N, num_classes+1, H/8, W/8] fp32 heat-maps, same state_dict.
forward compiles (once per input shape / precision) and replays ONE CUDA graph of hand-written sm_100a
kernels: backbone -> WASP -> decoder; nothing on the path is a torch op."""
import torch
import torch.nn as nn

from .. import engine, ops
from ..plan_module import PlanModule
from .modules.backbone import build_backbone
from .modules.decoder import build_decoder
from .modules.wasp import build_wasp


class unipose(PlanModule):
    def __init__(self, dataset, backbone='resnet', output_stride=16, num_classes=21, sync_bn=True,
                 freeze_bn=False, stride=8, precision=None):
        super().__init__()
        self.stride = stride
        self.num_classes = num_classes
        self.precision = precision
        BatchNorm = nn.BatchNorm2d   # sync_bn is accepted and ignored, as in the reference (unipose.py:9-14)
        self.pool_center = nn.AvgPool2d(kernel_size=9, stride=8, padding=1)   # unused by the image model
        self.backbone = build_backbone(backbone, output_stride, BatchNorm)
        self.wasp = build_wasp(backbone, output_stride, BatchNorm)
        self.decoder = build_decoder(dataset, num_classes, backbone, BatchNorm)
        if freeze_bn:
            self.freeze_bn()

    # ------------------------------------------------------------------------------------------
    def _build_plan(self, shape, device, u8=False, s2d=False):
        plan = engine.Plan(device, self._precision())
        b = plan.builder
        if s2d:
            # shape = (n, 3, h, w): no input tensor, the plan starts at the stem (forward_images fills plan.s2d_input)
            st = None
            x, low = self.backbone._emit_image(b, None, s2d_shape=(shape[0], shape[2], shape[3]))
        else:
            st = plan.static_input(shape, dtype=torch.uint8 if u8 else torch.float32)
            if u8:
                shape = (shape[0], 3, shape[1], shape[2])
            x, low = self.backbone._emit_image(b, st)
        x = self.wasp._emit(b, x)
        heat = self.decoder._emit(b, x, low)
        if self.stride != 8:   # model/unipose.py:31-32
            full = b.tensor((shape[0], heat.shape[1], shape[2], shape[3]))
            b.add(lambda heat=heat, full=full: ops._lib.call(
                "up_upsample_bilinear_ac_nchw_f32", ops._ptr(heat), ops._ptr(full), shape[0], heat.shape[1],
                heat.shape[2], heat.shape[3], shape[2], shape[3], ops._stream()), "upsample_to_input")
            heat = full
        plan.finalize([heat])
        return plan

    def plan_for(self, input):
        """The compiled plan for this input shape (bench / profiling hook)."""
        u8 = input.dtype == torch.uint8
        key = (tuple(input.shape), self._precision(), input.device.index, self.stride, u8)
        plan = self._plans.get(key)
        if plan is None:
            plan = self._build_plan(tuple(input.shape), input.device, u8=u8)
            self._plans[key] = plan
        return plan

    def forward_uint8(self, images):
        """Inference on raw uint8 HWC images [N, H, W, 3] (cv2 / decoder layout, BGR or RGB as the weights expect):
        the reference's `(img - 128) / 256` normalisation (utils/mpii_data.py:184-185) is fused into the stem's input
        packing, so a batch costs a quarter of the host->device bytes of the fp32 NCHW tensor and produces the same
        bits as forward(normalised fp32 input)."""
        self._check_inputs([images])
        if images.dtype != torch.uint8 or images.dim() != 4 or images.shape[3] != 3:
            raise ValueError("forward_uint8 expects uint8 [N, H, W, 3]; got %s %s" % (images.dtype, tuple(images.shape)))
        if self.training:
            raise NotImplementedError("forward_uint8 is an inference entry point (call .eval())")
        self._bn_eval_only()
        return self.plan_for(images).run(images.contiguous())[0].clone()

    def forward_images(self, images, size=368, shapes=None):
        """Inference on a ragged batch of decoded uint8 HWC images of any sizes (a list of [h, w, 3] CUDA tensors, or
        one packed buffer with `shapes`, see data.ImageBatch): the reference's cv2.resize(img, (368, 368))
        (utils/mpii_data.py:159-162) runs on the device, bit for bit, and writes the normalised space-to-depth input
        of the stem directly; the result equals forward_uint8(cv2-resized batch) bit for bit.  The resize is one
        launch on the current stream just before the graph replay of a plan keyed by (n, size, precision, device):
        ragged source addresses change every call, so it is not part of the captured graph."""
        from .. import data
        if self.training:
            raise NotImplementedError("forward_images is an inference entry point (call .eval())")
        batch = data.ImageBatch(images, shapes)
        s_h, s_w = data._out_size(size)
        dev = next(self.parameters()).device
        if batch.device != dev:
            raise RuntimeError("unipose_b200: parameters on %s but images on %s (call .cuda())" % (dev, batch.device))
        self._bn_eval_only()
        key = ("images", batch.n, s_h, s_w, self._precision(), batch.device.index, self.stride)
        plan = self._plans.get(key)
        if plan is None:
            plan = self._build_plan((batch.n, 3, s_h, s_w), batch.device, s2d=True)
            self._plans[key] = plan
        with torch.cuda.device(batch.device):
            data.resize_into_s2d(batch, plan.s2d_input, (s_h, s_w), wpad_left=2)
            return plan.run()[0].clone()

    def forward(self, input):
        self._check_inputs([input])
        if self.training:
            # train mode = the autograd-carrying training plan (dropout live); BatchNorm layers that were put in eval
            # mode - freeze_bn=True / model.freeze_bn(), model/unipose.py:24-25,40-43 - use their running statistics
            from .. import train
            return train.forward_train(self, input)
        self._bn_eval_only()
        plan = self.plan_for(input)
        src = input.detach()
        if src.dtype != torch.float32:
            src = src.float()
        out = plan.run(src)[0]
        return out.clone()

    def forward_static(self, input):
        """Like forward() but returns the plan-owned output buffer (overwritten by the next call)."""
        return self.plan_for(input).run(input)[0]

    # ------------------------------------------------------------------------------------------
    def freeze_bn(self):
        for m in self.modules():
            if isinstance(m, nn.BatchNorm2d):
                m.eval()

    def _lr_params(self, roots):
        for root in roots:
            for m in root.modules():
                if isinstance(m, (nn.Conv2d, nn.BatchNorm2d)):
                    for p in m.parameters(recurse=False):
                        if p.requires_grad:
                            yield p

    def get_1x_lr_params(self):
        return self._lr_params([self.backbone])

    def get_10x_lr_params(self):
        return self._lr_params([self.wasp, self.decoder])
