"""`UNet` with the reference's constructor, attribute names and state_dict layout (robosat/unet.py:76-141),
whose forward pass runs on librsb200.so.

The module tree exists to hold parameters under the reference's names (`resnet.*`, `center`, `dec0..dec5`, `final`)
so checkpoints written by either implementation load into the other (`module.`-prefixed when wrapped in
`nn.DataParallel`, train.py:69). `forward` (eval mode) builds -- and caches per input shape -- a `UNetEngine`
plan from the current parameters and replays it; nothing in it is executed by torch ops.

In training mode (`net.train()`, robosat/tools/train.py:168) the forward runs the train-mode plan (`UNetTrainEngine`:
batch-statistics BatchNorm with running-stat updates, activations saved in fp16) and `loss.backward()` runs its backward
plan (BN / ReLU / max-pool backward kernels, tcgen05 dgrad and wgrad); gradients arrive in `param.grad` as fp32.
"""

import torch
import torch.nn as nn

from robosat_b200 import _lib
from robosat_b200.engine import UNetEngine


class _TrainStep(torch.autograd.Function):
    """logits = net(images) in train mode; backward = the engine's backward plan. Parameters are passed only so that
    autograd routes their gradients (the engine reads the live parameter storage itself)."""

    @staticmethod
    def forward(ctx, x, module, names, *params):
        eng = module._train_engine_for(x)
        logits = eng.forward(x.contiguous())
        # the plan's saved activations / batch statistics are static buffers shared by every forward of this input shape:
        # stamp the forward so that a backward through a graph whose buffers were overwritten fails instead of being wrong
        eng.generation = getattr(eng, "generation", 0) + 1
        ctx.generation, ctx.consumed = eng.generation, False
        ctx.eng, ctx.names, ctx.params, ctx.fused = eng, names, params, module.fused_grad_accumulation
        return logits.clone()

    @staticmethod
    def backward(ctx, grad_out):
        if ctx.consumed:
            raise RuntimeError("robosat_b200.UNet: backward() ran twice through the same forward (retain_graph): the training plan "
                               "keeps one set of saved activations and consumes them in place; run forward again")
        if ctx.eng.generation != ctx.generation:
            raise RuntimeError("robosat_b200.UNet: a second train-mode forward with the same input shape ran before this graph's "
                               "backward() and overwrote its saved activations (one static plan per shape); call backward() "
                               "after each forward (gradient accumulation: forward, backward, forward, backward)")
        ctx.consumed = True
        grads = ctx.eng.backward(grad_out.contiguous().float())
        if ctx.fused:
            # every parameter that already holds a dense fp32 .grad (the usual case after optimizer.zero_grad()) is
            # accumulated in place by one kernel; autograd gets None for it and therefore launches no per-tensor add
            targets = {}
            for n, p in zip(ctx.names, ctx.params):
                g = p.grad
                if n in grads and g is not None and g.dtype == torch.float32 and g.is_contiguous() and g.device == grads[n].device:
                    targets[n] = g
            if targets:
                ctx.eng.accumulate_into(targets)
            return (None, None, None) + tuple(None if n in targets else grads.get(n) for n in ctx.names)
        return (None, None, None) + tuple(grads.get(n) for n in ctx.names)


class ConvRelu(nn.Module):
    """3x3 convolution (no bias) + ReLU parameter holder (unet.py:18-44)."""

    def __init__(self, num_in, num_out):
        super().__init__()
        self.block = nn.Conv2d(num_in, num_out, kernel_size=3, padding=1, bias=False)


class DecoderBlock(nn.Module):
    """Nearest x2 upsample + ConvRelu parameter holder (unet.py:47-73)."""

    def __init__(self, num_in, num_out):
        super().__init__()
        self.block = ConvRelu(num_in, num_out)


def _resnet50_container(pretrained):
    from torchvision.models import resnet50  # parameter container only; its forward is never called

    if pretrained:
        try:
            return resnet50(weights="IMAGENET1K_V1")
        except Exception as exc:  # no network / no cached weights: checkpoints overwrite these anyway
            import warnings

            warnings.warn("ImageNet weights unavailable (%s); the encoder starts from random weights" % exc)
    return resnet50(weights=None)


class UNet(nn.Module):
    def __init__(self, num_classes, num_filters=32, pretrained=True):
        super().__init__()
        assert num_filters == 32, "the B200 plan is built for the reference's num_filters=32"
        self.num_classes = num_classes
        self.resnet = _resnet50_container(pretrained)
        self.center = DecoderBlock(2048, num_filters * 8)
        self.dec0 = DecoderBlock(2048 + num_filters * 8, num_filters * 8)
        self.dec1 = DecoderBlock(1024 + num_filters * 8, num_filters * 8)
        self.dec2 = DecoderBlock(512 + num_filters * 8, num_filters * 2)
        self.dec3 = DecoderBlock(256 + num_filters * 2, num_filters * 2 * 2)
        self.dec4 = DecoderBlock(num_filters * 2 * 2, num_filters)
        self.dec5 = ConvRelu(num_filters, num_filters)
        self.final = nn.Conv2d(num_filters, num_classes, kernel_size=1)
        self._engines = {}
        self._engines_version = None
        self._train_engines = {}
        self.precision = None  # None: RSB_PRECISION or "strict" (see robosat_b200.engine.UNetEngine); eval plans only
        # training plans: None = RSB_TRAIN_PRECISION or "fast"; "strict" = hi/lo fp16 forward (robosat_b200.train_engine.UNetTrainEngine)
        self.train_precision = None
        # loss.backward() adds into existing .grad tensors with one kernel instead of one autograd add per parameter
        # (False: hand every gradient to autograd, e.g. when tensor hooks on parameters must fire)
        self.fused_grad_accumulation = True
        self.loss_scale = 4096.0  # activation gradients are fp16: scaled by this inside the backward plan, unscaled in param.grad

    # any weight change invalidates the packed plans
    def load_state_dict(self, *args, **kwargs):
        out = super().load_state_dict(*args, **kwargs)
        self.invalidate_plans()
        return out

    def invalidate_plans(self):
        self._engines.clear()

    def _weights_version(self):
        """Cheap fingerprint of the weights the inference plans were packed from: tensor identity + torch's in-place version
        counters. It changes on load_state_dict (also through an nn.DataParallel / DDP wrapper, which never reaches this class's
        override), optimizer steps and any other in-place edit, so a cached plan can never serve stale folded weights."""
        v = 0
        for t in list(self.parameters()) + list(self.buffers()):
            v = (v * 1000003 + t._version * 7919 + (t.data_ptr() & 0xFFFFFFFF)) & 0xFFFFFFFFFFFFFFFF
        return v

    def train(self, mode=True):
        if mode:
            self._engines.clear()  # inference plans hold folded copies of the weights: stale once training updates them
        return super().train(mode)

    def _train_engine_for(self, x):
        from robosat_b200.train_engine import UNetTrainEngine, default_train_precision

        precision = self.train_precision or default_train_precision()
        key = (tuple(x.shape), x.dtype, x.device.index, precision)
        eng = self._train_engines.get(key)
        if eng is not None and eng.overflowed():
            # strict plan: the weights outgrew the exponents fixed when it was built (that step's gradients were not finite and
            # the guarded optimiser step skipped it); a new plan takes fresh exponents from the current weights
            eng = None
            del self._train_engines[key]
        if eng is None:
            # live references: the plan reads the current storage of every parameter / buffer at each step
            params = dict(self.named_parameters())
            params.update(dict(self.named_buffers()))
            h, w = (x.shape[2], x.shape[3]) if x.dtype == torch.float32 else (x.shape[1], x.shape[2])
            eng = UNetTrainEngine(params, self.num_classes, x.shape[0], h, w, device=x.device, loss_scale=self.loss_scale,
                                  precision=precision)
            self._train_engines[key] = eng
        return eng

    def _engine_for(self, x):
        version = self._weights_version()
        if version != self._engines_version:
            self._engines.clear()
            self._engines_version = version
        key = (tuple(x.shape), x.dtype, x.device.index, self.precision)
        eng = self._engines.get(key)
        if eng is None:
            n = x.shape[0]
            h, w = (x.shape[2], x.shape[3]) if x.dtype == torch.float32 else (x.shape[1], x.shape[2])
            sd = {k: v.detach().cpu() for k, v in self.state_dict().items()}
            eng = UNetEngine(sd, self.num_classes, n, h, w, device=x.device, precision=self.precision)
            self._engines[key] = eng
        return eng

    def forward(self, x):
        """x: fp32 [N, 3, H, W] normalised (reference API) or uint8 [N, H, W, 3] raw RGB -> fp32 [N, C, H, W] logits."""
        if x.dtype == torch.float32:
            assert x.size(-1) % 32 == 0 and x.size(-2) % 32 == 0, "image resolution has to be divisible by 32 for resnet"
        if not x.is_cuda:
            raise _lib.RsbError("robosat_b200.UNet runs on sm_100a kernels only (no CPU fallback); move the input to a CUDA device")
        if self.training:
            # the reference's normalised fp32 NCHW tensors, or raw uint8 NHWC tiles (normalised by the pre-pass on the device)
            assert x.dtype in (torch.float32, torch.uint8), "training takes fp32 NCHW (normalised) or uint8 NHWC (raw) tiles"
            named = [(n, p) for n, p in self.named_parameters()]
            return _TrainStep.apply(x, self, tuple(n for n, _ in named), *[p for _, p in named])
        return self._engine_for(x).forward(x.contiguous()).clone()
