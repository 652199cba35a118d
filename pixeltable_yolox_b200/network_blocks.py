"""Building blocks with the reference's names, constructor signatures and state_dict layout
(yolox/models/network_blocks.py:27-208), so reference checkpoints load unchanged.

Execution model
  * eval + CUDA : every block lowers itself onto an ``engine.Builder`` (``lower`` methods); the
    launches are hand-written sm_100a kernels called through the C-ABI. ``forward`` on a block
    builds a tiny plan for just that block (NCHW in / NCHW out, like the reference).
  * training    : plain PyTorch ops so that autograd can differentiate the step (SURVEY 8a row 6:
    the SimOTA assignment is the B200-native part of the training step).
  * eval + CPU  : raises. There is deliberately no CPU fallback.
"""
from __future__ import annotations

import os

import torch
import torch.nn as nn
import torch.nn.functional as F


def get_activation(name="silu", inplace=True):
    # yolox/models/network_blocks.py:14-24
    table = {"silu": lambda: nn.SiLU(inplace=inplace), "relu": lambda: nn.ReLU(inplace=inplace),
             "lrelu": lambda: nn.LeakyReLU(0.1, inplace=inplace)}
    if name not in table:
        raise AttributeError("Unsupported act type: {}".format(name))
    return table[name]()


def act_name(module: nn.Module) -> str:
    if isinstance(module, nn.SiLU):
        return "silu"
    if isinstance(module, nn.LeakyReLU):
        return "lrelu"
    if isinstance(module, nn.ReLU):
        return "relu"
    raise AttributeError(f"Unsupported activation module {type(module).__name__}")


class _FusedBnAct(torch.autograd.Function):
    """Training-mode BatchNorm2d + activation of a BaseConv as three launches each way (csrc/yx_train.cu: statistics,
    finalize, apply) instead of torch's collect-statistics / transform / activation and activation-backward /
    batch_norm_backward kernels, which were 52 % of the training step's GPU time at 8 images per GPU
    (tools/gpu_prof_train.py). Running statistics are updated in place like F.batch_norm."""

    @staticmethod
    def forward(ctx, x, gamma, beta, running_mean, running_var, eps, momentum, act, num_batches_tracked=None):
        from . import ops
        from ._lib import ACT_CODES

        if not ops._is_channels_last(x):
            x = x.contiguous()
        code = ACT_CODES[act]
        y, mean, invstd = ops.bn_act_train_fwd(x, gamma, beta, running_mean, running_var, eps, momentum, code, num_batches_tracked)
        ctx.save_for_backward(x, gamma, beta, mean, invstd)
        ctx.act = code
        return y

    @staticmethod
    def backward(ctx, dy):
        from . import ops

        x, gamma, beta, mean, invstd = ctx.saved_tensors
        dy = dy.to(x.dtype)
        if dy.stride() != x.stride():                       # same memory format as x (NCHW or channels_last)
            _, _, H, W = x.shape
            ld = dy.stride(3)
            sliced = (ops._is_channels_last(x) and ld % 8 == 0 and dy.stride() == (H * W * ld, 1, W * ld, ld)
                      and dy.data_ptr() % 16 == 0)           # channel slice of a wider NHWC gradient (backward of cat): read in place
            if not sliced:
                dy = dy.contiguous(memory_format=torch.channels_last) if ops._is_channels_last(x) else dy.contiguous()
        from .train_conv import direct_target

        tg, tb = direct_target(gamma), direct_target(beta)
        if tg is not None and tb is not None:
            # gradient accumulation into .grad inside the finalize launch (see train_conv.direct_target)
            dx, _, _ = ops.bn_act_train_bwd(x, dy, gamma, beta, mean, invstd, ctx.act, tg, tb)
            return dx, None, None, None, None, None, None, None, None
        dx, dgamma, dbeta = ops.bn_act_train_bwd(x, dy, gamma, beta, mean, invstd, ctx.act)
        return dx, dgamma, dbeta, None, None, None, None, None, None


class _SppCat(torch.autograd.Function):
    """cat[x, maxpool5(x), maxpool9(x), maxpool13(x)] of SPPBottleneck (network_blocks.py:137-139) on a channels_last 16-bit
    tensor: forward = the inference pool kernel on the concat buffer, backward = one scatter kernel (torch's channels_last
    max-pool kernels took 1.2 ms of the 8-image training step for these three 20x20 maps)."""

    @staticmethod
    def forward(ctx, x):
        from . import ops

        B, c, H, W = x.shape
        cat = torch.empty((B, 4 * c, H, W), dtype=x.dtype, device=x.device, memory_format=torch.channels_last)
        cat[:, :c] = x
        ops.spp_maxpool(ops._nhwc(cat), c)
        ctx.save_for_backward(cat)
        return cat

    @staticmethod
    def backward(ctx, dout):
        from . import ops

        (cat,) = ctx.saved_tensors
        return ops.spp_maxpool_bwd(cat, dout.to(cat.dtype).contiguous(memory_format=torch.channels_last))


class _B200Block(nn.Module):
    """Shared forward dispatch: training -> torch autograd ops, eval -> B200 plan."""

    def _train_forward(self, x):  # pragma: no cover - overridden
        raise NotImplementedError

    def lower(self, b, x):  # pragma: no cover - overridden
        raise NotImplementedError

    def forward(self, x):
        if self.training:
            return self._train_forward(x)
        from .engine import run_block

        return run_block(self, x)


class BaseConv(_B200Block):
    """Conv2d(bias=False, pad=(k-1)//2) -> BatchNorm2d -> act (network_blocks.py:27-52)."""

    def __init__(self, in_channels, out_channels, ksize, stride, groups=1, bias=False, act="silu"):
        super().__init__()
        self.conv = nn.Conv2d(in_channels, out_channels, kernel_size=ksize, stride=stride,
                              padding=(ksize - 1) // 2, groups=groups, bias=bias)
        self.bn = nn.BatchNorm2d(out_channels)
        self.act = get_activation(act, inplace=True)

    def _train_forward(self, x):
        from .train_conv import conv2d

        y = conv2d(x, self.conv)             # tcgen05 forward / dgrad / wgrad under 16-bit autocast, else torch
        bn = self.bn
        if (y.is_cuda and bn.training and bn.momentum is not None and bn.track_running_stats and bn.affine
                and bn.weight.dtype == torch.float32 and y.dim() == 4 and y.dtype in (torch.float32, torch.bfloat16, torch.float16)):
            # nn.BatchNorm2d.forward in train mode: batch statistics, running statistics updated with `momentum`
            # (num_batches_tracked counts the calls), then the activation -- one fused pass each way
            # (num_batches_tracked counts the calls: incremented by the kernel)
            return _FusedBnAct.apply(y, bn.weight, bn.bias, bn.running_mean, bn.running_var, bn.eps, bn.momentum,
                                     act_name(self.act), bn.num_batches_tracked)
        return self.act(bn(y))

    def fuseforward(self, x):
        return self.act(self.conv(x))

    def lower(self, b, x, out=None, res=None, ups=None):
        if self.conv.groups != 1:
            return b.dwconv(x, self, out=out)
        return b.conv(x, [b.part(self)], out=out, res=res, ups=ups, act=act_name(self.act),
                      ksize=self.conv.kernel_size[0], stride=self.conv.stride[0])


class DWConv(_B200Block):
    """Depthwise 3x3 BaseConv followed by a 1x1 BaseConv (network_blocks.py:55-74)."""

    def __init__(self, in_channels, out_channels, ksize, stride=1, act="silu"):
        super().__init__()
        self.dconv = BaseConv(in_channels, in_channels, ksize=ksize, stride=stride, groups=in_channels, act=act)
        self.pconv = BaseConv(in_channels, out_channels, ksize=1, stride=1, groups=1, act=act)

    def _train_forward(self, x):
        return self.pconv._train_forward(self.dconv._train_forward(x))

    def lower(self, b, x, out=None, res=None, ups=None):
        return self.pconv.lower(b, self.dconv.lower(b, x), out=out, res=res, ups=ups)


class Bottleneck(_B200Block):
    """1x1 -> 3x3 (+ x when shortcut and channels match) (network_blocks.py:77-99)."""

    def __init__(self, in_channels, out_channels, shortcut=True, expansion=0.5, depthwise=False, act="silu"):
        super().__init__()
        hidden_channels = int(out_channels * expansion)
        Conv = DWConv if depthwise else BaseConv
        self.conv1 = BaseConv(in_channels, hidden_channels, 1, stride=1, act=act)
        self.conv2 = Conv(hidden_channels, out_channels, 3, stride=1, act=act)
        self.use_add = shortcut and in_channels == out_channels

    def _train_forward(self, x):
        y = self.conv2._train_forward(self.conv1._train_forward(x))
        return y + x if self.use_add else y

    def lower(self, b, x, out=None):
        if b.bottleneck_fusable(x, self) and (out is None or out.t is not x.t or out.c_off != x.c_off):
            # one kernel: the hidden tensor never leaves the SM (yx_bottleneck_fwd); cannot run in place
            if out is None:
                out = b.new_feat(x.B, x.H, x.W, [self.conv2.conv.out_channels])
            return b.bottleneck(x, self, out)
        # the residual is added in the epilogue of conv2; writing in place over x is safe because
        # conv2 reads only conv1's output and each thread reads x[p] before it writes out[p]
        t = self.conv1.lower(b, x)
        return self.conv2.lower(b, t, out=out, res=x if self.use_add else None)


class ResLayer(_B200Block):
    "Residual layer with `in_channels` inputs (Darknet-53 only; network_blocks.py:102-117)."

    def __init__(self, in_channels: int):
        super().__init__()
        mid_channels = in_channels // 2
        self.layer1 = BaseConv(in_channels, mid_channels, ksize=1, stride=1, act="lrelu")
        self.layer2 = BaseConv(mid_channels, in_channels, ksize=3, stride=1, act="lrelu")

    def _train_forward(self, x):
        return x + self.layer2._train_forward(self.layer1._train_forward(x))

    def lower(self, b, x, out=None):
        return self.layer2.lower(b, self.layer1.lower(b, x), out=out, res=x)


class SPPBottleneck(_B200Block):
    """1x1 -> cat[x, maxpool5, maxpool9, maxpool13] -> 1x1 (network_blocks.py:120-142)."""

    def __init__(self, in_channels, out_channels, kernel_sizes=(5, 9, 13), activation="silu"):
        super().__init__()
        hidden_channels = in_channels // 2
        self.conv1 = BaseConv(in_channels, hidden_channels, 1, stride=1, act=activation)
        self.m = nn.ModuleList([nn.MaxPool2d(kernel_size=ks, stride=1, padding=ks // 2) for ks in kernel_sizes])
        conv2_channels = hidden_channels * (len(kernel_sizes) + 1)
        self.conv2 = BaseConv(conv2_channels, out_channels, 1, stride=1, act=activation)

    def _train_forward(self, x):
        x = self.conv1._train_forward(x)
        from . import ops

        if (x.is_cuda and tuple(m.kernel_size for m in self.m) == (5, 9, 13) and x.dtype in (torch.bfloat16, torch.float16)
                and ops._is_channels_last(x)):
            x = _SppCat.apply(x)
        else:
            x = torch.cat([x] + [m(x) for m in self.m], dim=1)
        return self.conv2._train_forward(x)

    def lower(self, b, x, out=None):
        ks = tuple(m.kernel_size for m in self.m)
        if ks != (5, 9, 13):
            raise NotImplementedError(f"SPP kernel sizes {ks}: the B200 kernel implements the 5/9/13 cascade")
        hidden = self.conv1.conv.out_channels
        cat = b.new_feat(x.B, x.H, x.W, [hidden] * 4)   # conv1 writes segment 0, the pool kernel 1..3
        self.conv1.lower(b, x, out=cat.seg(0))
        b.spp(cat, hidden)
        return self.conv2.lower(b, cat, out=out)


class CspLayer(_B200Block):
    """C3: conv3(cat(m(conv1(x)), conv2(x))) (network_blocks.py:145-183)."""

    def __init__(self, in_channels, out_channels, n=1, shortcut=True, expansion=0.5, depthwise=False, act="silu"):
        super().__init__()
        hidden_channels = int(out_channels * expansion)
        self.conv1 = BaseConv(in_channels, hidden_channels, 1, stride=1, act=act)
        self.conv2 = BaseConv(in_channels, hidden_channels, 1, stride=1, act=act)
        self.conv3 = BaseConv(2 * hidden_channels, out_channels, 1, stride=1, act=act)
        self.m = nn.Sequential(*[
            Bottleneck(hidden_channels, hidden_channels, shortcut, 1.0, depthwise, act=act) for _ in range(n)
        ])

    def _train_forward(self, x):
        from .streams import Branch

        br = Branch(x, 0)                    # conv2 (+ its BatchNorm) next to conv1 -> bottleneck chain, forward and backward
        with br:
            x_2 = self.conv2._train_forward(x)
        x_1 = self.conv1._train_forward(x)
        for blk in self.m:
            x_1 = blk._train_forward(x_1)
        br.join()
        return self.conv3._train_forward(torch.cat((x_1, x_2), dim=1))

    def lower(self, b, x, out=None):
        # conv1 and conv2 read the same tensor: one GEMM with stacked weights writes the concat
        # buffer [x_1 | x_2]; the bottleneck chain then updates the x_1 half in place, so the
        # torch.cat of the reference (network_blocks.py:182) never happens.
        hidden = self.conv1.conv.out_channels
        if len(self.m) > 0 and all(b.bottleneck_fusable(b.probe_feat(x, hidden), blk) for blk in self.m):
            # fused bottlenecks cannot run in place: the stacked GEMM writes x_1 to its own buffer and x_2 straight
            # into the concat buffer [y | x_2] (two destinations, yx_conv_desc.out2); the chain ping-pongs
            # x_1 -> tmp -> ... and its last link writes y, so conv3 reads one dense buffer (the torch.cat of
            # network_blocks.py:182 in the reference's channel order) and every access stays contiguous
            cat = b.new_feat(x.B, x.H, x.W, [hidden, hidden])
            cur = b.new_feat(x.B, x.H, x.W, [hidden])
            b.conv(x, [b.part(self.conv1), b.part(self.conv2)], out=cur, out2=cat.seg(1),
                   act=act_name(self.conv1.act), ksize=1, stride=1)
            spare = None
            for i, blk in enumerate(self.m):
                if i == len(self.m) - 1:
                    dst = cat.seg(0)
                else:
                    dst = spare if spare is not None else b.new_feat(x.B, x.H, x.W, [hidden])
                blk.lower(b, cur, out=dst)
                cur, spare = dst, cur
            return self.conv3.lower(b, cat, out=out)
        cat = b.conv(x, [b.part(self.conv1), b.part(self.conv2)], act=act_name(self.conv1.act), ksize=1, stride=1)
        x1 = cat.seg(0)
        for blk in self.m:
            blk.lower(b, x1, out=x1)
        return self.conv3.lower(b, cat, out=out)


class Focus(_B200Block):
    """Space-to-depth (TL, BL, TR, BR) then a conv (network_blocks.py:186-208)."""

    def __init__(self, in_channels, out_channels, ksize=1, stride=1, act="silu"):
        super().__init__()
        self.conv = BaseConv(in_channels * 4, out_channels, ksize, stride, act=act)

    def _train_forward(self, x):
        from . import ops
        from .train_conv import usable

        dt = usable(x, self.conv.conv) if x.dim() == 4 else None
        if (dt is not None and x.shape[1] == 3 and x.is_contiguous() and x.dtype in (torch.float32, torch.uint8)
                and x.shape[2] % 2 == 0 and x.shape[3] % 2 == 0 and not x.requires_grad
                and os.environ.get("YX_TRAIN_FOCUS", "1") != "0"):
            # the four strided slices + cat + cast + channel padding of the torch path (six launches over the largest tensor
            # of the step) as the inference space-to-depth kernel: image -> 16-bit NHWC with the 12 Focus channels padded to 16,
            # which is the layout the stem conv's tcgen05 kernels take (the conv pads its 12 input channels to 16 anyway)
            B, _, H, W = x.shape
            s2d = torch.empty((B, 16, H // 2, W // 2), dtype=dt, device=x.device, memory_format=torch.channels_last)
            ops.focus_s2d(x, ops._nhwc(s2d))
            return self.conv._train_forward(s2d)
        tl, tr = x[..., ::2, ::2], x[..., ::2, 1::2]
        bl, br = x[..., 1::2, ::2], x[..., 1::2, 1::2]
        return self.conv._train_forward(torch.cat((tl, bl, tr, br), dim=1))

    def lower_image(self, b, img, out=None):
        """img: NCHW fp32/uint8 image batch (raw 0..255)."""
        if img.shape[1] != 3:
            raise NotImplementedError("Focus on the B200 path expects a 3-channel image")
        conv = self.conv.conv
        fused = (b.dtype != torch.float32 and conv.kernel_size == (3, 3) and conv.stride == (1, 1) and conv.groups == 1
                 and conv.out_channels <= 128 and img.shape[2] % 2 == 0 and img.shape[3] % 2 == 0)
        if fused:
            return b.focus_conv(img, self.conv, out=out)      # one kernel: image -> stem activations
        return self.conv.lower(b, b.focus(img), out=out)      # fp32 verification path: s2d + SIMT conv
