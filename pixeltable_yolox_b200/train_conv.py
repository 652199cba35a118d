"""Dense convolution of the training step on the tensor cores, forward and backward.

Replaces what torch autograd dispatches to cuDNN for `BaseConv.conv` (yolox/models/network_blocks.py:27-52) and the
prediction convs (yolox/models/yolo_head.py:94-120) inside `Trainer.train_one_iter` (yolox/core/trainer.py:96-129):

  forward  y  = conv(x, W) (+ bias)     csrc/yx_conv_tc.cu, the inference implicit GEMM with unfolded weights, no activation
  dgrad    dx = conv(dy, rot180(W)^T)   the same kernel (stride 2: the four sub-pixel phases as one conv over dy with a
                                        depth-to-space store; odd input sizes: on the zero-stuffed dy, dilate2)
  wgrad    dW = sum_p dy[p] (x) x[p+t]  csrc/yx_wgrad_tc.cu (tcgen05, both operands MN-major straight from NHWC)

Activations stay 16-bit channels_last (NHWC) between layers, which is the layout every kernel of this package uses; the
fp32 master weights are packed to 16-bit operands once per step (WeightPacker: one launch for all layers; without it one
launch per layer for the forward and the dgrad operand). Numerics match torch.autocast: 16-bit operands, fp32 accumulation, fp32 weight gradients.

Depthwise 3x3 convs (groups == channels, the first half of DWConv in yolox_nano) run on SIMT kernels instead
(csrc/yx_dwconv_train.cu: forward and dgrad as one gather kernel, wgrad as a deterministic split reduction); they read the fp32
master weight directly, so they need no packed operands.
"""
from __future__ import annotations

import os
from typing import Optional

import torch

from . import ops
from ._lib import YX_ACT_NONE

_zero_bias = {}

# Direct gradient accumulation: for parameters that FusedSgdEma(direct_grads=True) has marked (`param._yx_direct_grad`: their
# .grad is a view of the optimizer's flat, zeroed gradient buffer) the wgrad reduction and the BatchNorm backward add their
# results straight into `param.grad` and return no gradient to autograd, so AccumulateGrad's one `grad += new` launch per
# parameter (242 per step) disappears. Opt-in per parameter, so other modules in the process are unaffected; not for modules
# wrapped in DistributedDataParallel, whose reduction hooks hang off AccumulateGrad. set_direct_grads(False) is a global off
# switch (scripts that fill .grad themselves).
_direct_grads = True


def set_direct_grads(on: bool) -> None:
    global _direct_grads
    _direct_grads = bool(on)


def direct_grads() -> bool:
    return _direct_grads


def direct_target(param: torch.Tensor) -> Optional[torch.Tensor]:
    """The tensor a backward kernel should accumulate this parameter's gradient into, or None (return it to autograd)."""
    if _direct_grads and getattr(param, "_yx_direct_grad", False) and param.grad is not None:
        return param.grad
    return None


# With direct gradient accumulation the weight-gradient launches have no consumer before the optimizer step, so they run on a
# side streams (_N_WGRAD_STREAMS per device, round robin) next to the backward's critical chain  BatchNorm backward -> dgrad -> BatchNorm backward ...:
# every kernel of an 8-image step is a fraction of a wave, so the two chains overlap (a CUDA-graph capture records the fork
# and the join as graph branches). The wgrad inputs (saved activation, output gradient) are kept referenced until
# `join_wgrad()` so that the caching allocator cannot hand their memory to the main stream while the side stream reads it.
_wgrad_side = {}


_N_WGRAD_STREAMS = 3


def _side(dev: torch.device):
    """(stream, pending list) for the next weight gradient: round robin over _N_WGRAD_STREAMS side streams (each with its own
    partial-sum workspace, ops.conv_wgrad keys it by stream), so consecutive layers' wgrad launches overlap each other too."""
    ent = _wgrad_side.get(dev)
    if ent is None:
        ent = _wgrad_side[dev] = [[torch.cuda.Stream(dev) for _ in range(_N_WGRAD_STREAMS)], [], 0]
    ent[2] = (ent[2] + 1) % len(ent[0])
    return ent[0][ent[2]], ent[1]


def join_wgrad(dev: Optional[torch.device] = None) -> None:
    """Make the current stream wait for the side-stream weight gradients (call before reading .grad: FusedSgdEma.step does)."""
    for d, (streams, pending, _) in _wgrad_side.items():
        if dev is None or d == dev:
            if pending:
                for stream in streams:
                    torch.cuda.current_stream(d).wait_stream(stream)
                pending.clear()
                ops.release_retired_workspaces(d)


class WeightPacker:
    """All conv weights of a model packed to their 16-bit forward / dgrad operands in ONE launch per step
    (yx_pack_train_weights_multi) instead of one launch per layer. `attach(model, dtype)` makes `YoloxModule.forward` call
    `pack()` at the start of every training forward; the packed buffers are used by the convs of THAT forward (and, through
    the tensors saved for backward, by its backward) and by nothing else."""

    CHUNK = 8192

    def __init__(self, model: torch.nn.Module, dtype: torch.dtype):
        import numpy as np

        self.dtype = dtype
        self.entries = {}
        rows, chunks = [], []
        dev = None
        for mod in model.modules():
            if not isinstance(mod, torch.nn.Conv2d) or mod.groups != 1 or mod.weight.dtype != torch.float32 or not mod.weight.is_cuda:
                continue
            k, s = mod.kernel_size, mod.stride
            if k[0] != k[1] or s[0] != s[1] or (k[0], s[0]) not in ((1, 1), (3, 1), (3, 2)):
                continue
            w = mod.weight
            dev = w.device
            o, i, taps = w.shape[0], w.shape[1], k[0] * k[0]
            o_pad, i_pad = _pad16(o), _pad16(i)
            wf = torch.empty((o_pad, taps, i_pad), dtype=dtype, device=dev)
            sub = s[0] == 2            # stride-2 dgrad as one sub-pixel conv: zeros of the buffer are written once, here
            wd = (torch.zeros((4 * i_pad, 9, o_pad), dtype=dtype, device=dev) if sub
                  else torch.empty((i_pad, taps, o_pad), dtype=dtype, device=dev))
            so, si, st = ops._weight_strides(w)
            t = len(rows)
            rows.append((w.data_ptr(), so, si, st, o, i, taps, o_pad, i_pad, wf.data_ptr(), wd.data_ptr(), 1 if sub else 0))
            chunks += [(t, e) for e in range(0, o_pad * taps * i_pad, self.CHUNK)]
            self.entries[id(w)] = (w, wf, wd, w.data_ptr())
        if not rows:
            raise ValueError("WeightPacker: the model has no dense CUDA convolution")
        self.device = dev
        self.table = torch.from_numpy(np.array(rows, dtype=np.int64)).to(dev)
        self.chunks = torch.from_numpy(np.array(chunks, dtype=np.int32)).to(dev)
        self.active = False

    def __deepcopy__(self, memo):
        return None                  # the table holds raw pointers of THIS model's weights: a copied model gets no packer

    def pack(self) -> None:
        from ._lib import check, dtype_code, lib, stream_ptr

        with ops.on_device(self.device):
            check(lib().yx_pack_train_weights_multi(self.table.data_ptr(), self.chunks.data_ptr(), self.chunks.shape[0], self.CHUNK,
                                                    dtype_code(self.dtype), stream_ptr(self.device)), "pack_train_weights_multi")
        self.active = True

    def lookup(self, weight: torch.Tensor, dtype: torch.dtype):
        if not self.active or dtype != self.dtype:
            return None
        ent = self.entries.get(id(weight))
        # a parameter that was reallocated since the table was built (.to(), load_state_dict(assign=True)) is not in it
        if ent is None or ent[0] is not weight or weight.data_ptr() != ent[3]:
            return None
        return ent[1], ent[2]


_packer: Optional[WeightPacker] = None


def attach_packer(model: torch.nn.Module, dtype: torch.dtype) -> WeightPacker:
    """Batched weight packing for `model`'s training forward (see WeightPacker). Returns the packer; detach with None."""
    p = WeightPacker(model, dtype)
    model.__dict__["_yx_train_packer"] = p
    return p


def _zeros(dev: torch.device, n: int) -> torch.Tensor:
    t = _zero_bias.get((dev, n))
    if t is None:
        t = _zero_bias[(dev, n)] = torch.zeros(n, dtype=torch.float32, device=dev)
    return t


def _pad16(c: int) -> int:
    return (c + 15) // 16 * 16


def _pad_channels(t: torch.Tensor, c_pad: int) -> torch.Tensor:
    """[B, C, H, W] -> dense channels_last [B, c_pad, H, W], extra channels zero."""
    if t.shape[1] == c_pad:
        return t.contiguous(memory_format=torch.channels_last)
    out = torch.empty((t.shape[0], c_pad, t.shape[2], t.shape[3]), dtype=t.dtype, device=t.device,
                      memory_format=torch.channels_last)
    out[:, :t.shape[1]] = t
    out[:, t.shape[1]:] = 0
    return out


def usable(x: torch.Tensor, conv: torch.nn.Conv2d) -> Optional[torch.dtype]:
    """The 16-bit compute dtype when this conv can run on the tcgen05 training path, else None (torch / cuDNN runs it):
    CUDA, dense (groups == 1) 1x1 stride 1 or 3x3 stride 1 / 2 with `same` padding, under 16-bit autocast or on 16-bit input."""
    if os.environ.get("YX_TRAIN_CONV", "1") == "0" or not x.is_cuda or x.dim() != 4:
        return None
    k, s = conv.kernel_size, conv.stride
    if conv.groups != 1 or k[0] != k[1] or s[0] != s[1] or conv.dilation != (1, 1) or conv.padding_mode != "zeros":
        return None
    if (k[0], s[0]) not in ((1, 1), (3, 1), (3, 2)) or conv.padding != ((k[0] - 1) // 2,) * 2:
        return None
    if conv.weight.dtype != torch.float32:
        return None
    if torch.is_autocast_enabled("cuda"):
        dt = torch.get_autocast_dtype("cuda")
    else:
        dt = x.dtype
    return dt if dt in (torch.bfloat16, torch.float16) else None


def usable_depthwise(x: torch.Tensor, conv: torch.nn.Conv2d) -> Optional[torch.dtype]:
    """The 16-bit compute dtype when this conv can run on the depthwise training kernels, else None (torch / cuDNN runs it):
    CUDA, groups == in == out channels (a multiple of 8), 3x3 stride 1 / 2, pad 1, no bias, fp32 weight, under 16-bit
    autocast or on 16-bit input."""
    if os.environ.get("YX_TRAIN_CONV", "1") == "0" or not x.is_cuda or x.dim() != 4:
        return None
    c = conv.in_channels
    if conv.groups != c or conv.out_channels != c or c % 8 != 0 or x.shape[1] != c or conv.bias is not None:
        return None
    if conv.kernel_size != (3, 3) or conv.stride not in ((1, 1), (2, 2)) or conv.padding != (1, 1):
        return None
    if conv.dilation != (1, 1) or conv.padding_mode != "zeros" or conv.weight.dtype != torch.float32:
        return None
    dt = torch.get_autocast_dtype("cuda") if torch.is_autocast_enabled("cuda") else x.dtype
    return dt if dt in (torch.bfloat16, torch.float16) else None


class _DwConv(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, weight, stride, dtype):
        xh = x.detach().to(dtype).contiguous(memory_format=torch.channels_last)
        y = ops.dwconv_train_fwd(xh, weight.detach(), stride)
        ctx.save_for_backward(xh, weight)
        ctx.geom = (stride, x.dtype)
        return y

    @staticmethod
    def backward(ctx, dy):
        xh, weight = ctx.saved_tensors
        stride, x_dtype = ctx.geom
        dyh = dy.to(xh.dtype).contiguous(memory_format=torch.channels_last)
        dx = dw = None
        if ctx.needs_input_grad[1]:
            target = direct_target(weight)
            if target is not None:
                stream, pending = _side(xh.device)
                stream.wait_event(torch.cuda.current_stream(xh.device).record_event())
                with torch.cuda.stream(stream):
                    ops.dwconv_wgrad(xh, dyh, weight, stride, accumulate_into=target)
                pending.append((xh, dyh))
            else:
                dw = ops.dwconv_wgrad(xh, dyh, weight, stride)
        if ctx.needs_input_grad[0]:
            dx = ops.dwconv_dgrad(dyh, weight.detach(), stride, xh.shape[2], xh.shape[3]).to(x_dtype)
        return dx, dw, None, None


class _ConvTc(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, weight, bias, stride, dtype):
        o, i, k, _ = weight.shape
        o_pad, i_pad = _pad16(o), _pad16(i)
        B, _, H, W = x.shape
        pad = (k - 1) // 2
        OH, OW = (H + 2 * pad - k) // stride + 1, (W + 2 * pad - k) // stride + 1
        xh = _pad_channels(x.detach().to(dtype), i_pad)
        # stride-2 dgrad: one sub-pixel conv over dy with a depth-to-space store when the input size is even, else the
        # rotated weights on the zero-stuffed dy
        sub = stride == 2 and H % 2 == 0 and W % 2 == 0
        pre = _packer.lookup(weight, dtype) if _packer is not None else None
        if pre is not None and (stride == 1 or sub):
            wf, wd = pre
        else:
            wf, wd = ops.pack_train_weights(weight.detach(), dtype, o_pad, i_pad, want_dgrad=ctx.needs_input_grad[0], subpixel=sub)
        if bias is None:
            b = _zeros(x.device, o_pad)
        elif o_pad == o:
            b = bias.detach().float().contiguous()
        else:
            b = torch.zeros(o_pad, dtype=torch.float32, device=x.device)
            b[:o] = bias.detach()
        y = torch.empty((B, o_pad, OH, OW), dtype=dtype, device=x.device, memory_format=torch.channels_last)
        ops.conv_bn_act(ops._nhwc(xh), wf, b, ops._nhwc(y), k, stride, YX_ACT_NONE)
        ctx.save_for_backward(xh, wd, weight)
        ctx.geom = (o, i, k, stride, o_pad, i_pad, H, W, x.dtype, bias is not None, sub)
        return y if o_pad == o else y[:, :o]

    @staticmethod
    def backward(ctx, dy):
        xh, wd, weight = ctx.saved_tensors
        o, i, k, stride, o_pad, i_pad, H, W, x_dtype, has_bias, sub = ctx.geom
        dyh = _pad_channels(dy.to(xh.dtype), o_pad)
        dx = dw = db = None
        if ctx.needs_input_grad[1]:
            target = direct_target(weight)
            if target is not None:
                stream, pending = _side(xh.device)
                stream.wait_event(torch.cuda.current_stream(xh.device).record_event())
                with torch.cuda.stream(stream):
                    ops.conv_wgrad(xh, dyh, weight, k, stride, accumulate_into=target)
                pending.append((xh, dyh))
            else:
                dw = ops.conv_wgrad(xh, dyh, weight, k, stride)
        if ctx.needs_input_grad[0]:
            dxp = torch.empty((xh.shape[0], i_pad, H, W), dtype=xh.dtype, device=xh.device, memory_format=torch.channels_last)
            if sub:
                ops.conv_bn_act(ops._nhwc(dyh), wd, _zeros(xh.device, 4 * i_pad), ops._nhwc(dxp), 3, 1, YX_ACT_NONE, shuffle2_c=i_pad)
            else:
                src = dyh if stride == 1 else ops.dilate2(dyh, H, W)
                ops.conv_bn_act(ops._nhwc(src), wd, _zeros(xh.device, i_pad), ops._nhwc(dxp), k, 1, YX_ACT_NONE)
            dx = (dxp if i_pad == i else dxp[:, :i]).to(x_dtype)
        if has_bias and ctx.needs_input_grad[2]:
            db = dy.float().sum((0, 2, 3))
        return dx, dw, db, None, None


class packed_weights:
    """Context of one training forward: `with packed_weights(model): ...` packs every conv weight in one launch when a
    WeightPacker is attached to the model and makes the convs inside the block use the packed operands."""

    def __init__(self, model: torch.nn.Module):
        self.packer = model.__dict__.get("_yx_train_packer")

    def __enter__(self):
        global _packer
        self.prev = _packer
        if self.packer is not None and torch.is_autocast_enabled("cuda") and torch.get_autocast_dtype("cuda") == self.packer.dtype:
            self.packer.pack()
            _packer = self.packer
        return self

    def __exit__(self, *exc):
        global _packer
        if self.packer is not None:
            self.packer.active = False
        _packer = self.prev
        return False


def conv2d(x: torch.Tensor, conv: torch.nn.Conv2d) -> torch.Tensor:
    """`conv(x)` in the training step: tcgen05 forward / dgrad / wgrad when `usable`, the depthwise kernels when
    `usable_depthwise`, else the module's own forward."""
    dt = usable(x, conv)
    if dt is not None:
        return _ConvTc.apply(x, conv.weight, conv.bias, conv.stride[0], dt)
    dt = usable_depthwise(x, conv)
    if dt is not None:
        return _DwConv.apply(x, conv.weight, conv.stride[0], dt)
    return conv(x)
