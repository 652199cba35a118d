"""Host-side lowering of the reference's eval forward onto the native plan runtime.

`Builder` turns a module tree (network_blocks / darknet / yolo_pafpn / yolo_head) into an ordered
list of launches over pre-allocated NHWC buffers: BN is folded and weights repacked once by a
CUDA kernel (yx_pack_weights), tensor maps are encoded once (yx_plan_add_conv), and a forward is a
single FFI call (yx_plan_run) that can replay one CUDA graph.

Data layout in HBM
  activations : NHWC, bf16/fp16 (tensor-core path) or fp32 (verification path); a logical tensor
                with c channels occupies pad16(c) channel slots (extra slots are exact zeros);
                concatenations (CSP, PAFPN, SPP, head towers) are *segments* of one buffer that
                the producers write directly, so no concat/upsample kernels exist.
  weights     : [out_c][taps][in_c] K-major in the activation dtype; bias fp32.
  head output : [B, A, 5+nc] fp32, written by the prediction-GEMM epilogue.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass, field
from typing import Dict, List, Optional, Sequence, Tuple

import torch
import torch.nn as nn

from . import _lib, ops
from ._lib import ACT_CODES, check, dtype_code, lib, stream_ptr
from .ops import View


def _on_device_of(get_device):
    """Run the wrapped function with the tensor's / engine's CUDA device current: the library launches on the current device
    and a module on cuda:1 must not launch on cuda:0 with cuda:1 pointers (advisor finding, round 1)."""
    import functools

    def deco(fn):
        @functools.wraps(fn)
        def wrapper(*args, **kwargs):
            dev = get_device(*args, **kwargs)
            if dev is not None and torch.device(dev).type == "cuda":
                with torch.cuda.device(dev):
                    return fn(*args, **kwargs)
            return fn(*args, **kwargs)
        return wrapper
    return deco


def pad16(c: int) -> int:
    return (c + 15) // 16 * 16


@dataclass
class Feat:
    """NHWC buffer slice made of channel segments; segment i has segs[i] real channels and
    occupies pad16(segs[i]) slots."""

    t: torch.Tensor          # [B, H, W, Ctot]
    c_off: int
    segs: List[int]

    @property
    def B(self): return self.t.shape[0]
    @property
    def H(self): return self.t.shape[1]
    @property
    def W(self): return self.t.shape[2]
    @property
    def c_slots(self): return sum(pad16(s) for s in self.segs)
    @property
    def c_real(self): return sum(self.segs)

    def seg_off(self, i: int) -> int:
        return sum(pad16(s) for s in self.segs[:i])

    def seg(self, i: int) -> "Feat":
        return Feat(self.t, self.c_off + self.seg_off(i), [self.segs[i]])

    def view(self) -> View:
        return View(self.t, self.c_off, self.c_slots)

    def to_nchw(self) -> torch.Tensor:
        """Logical NCHW tensor (drops the padding slots); for module-level forward only."""
        chunks = []
        for i, s in enumerate(self.segs):
            o = self.c_off + self.seg_off(i)
            chunks.append(self.t[..., o:o + s])
        x = chunks[0] if len(chunks) == 1 else torch.cat(chunks, dim=-1)
        return x.permute(0, 3, 1, 2).contiguous()


@dataclass
class Part:
    """One source conv of a (possibly merged) GEMM: rows [o_off, o_off+o) of the packed weight;
    its logical input channels map, in order, onto the listed input segments."""

    weight: torch.Tensor
    bn: Optional[nn.BatchNorm2d]
    bias: Optional[torch.Tensor]
    o_off: Optional[int] = None
    in_segs: Optional[List[int]] = None


class Builder:
    def __init__(self, device: torch.device, dtype: torch.dtype, use_plan: bool = True):
        if device.type != "cuda":
            raise RuntimeError(
                f"eval forward requested on {device}: the B200 path runs hand-written sm_100a CUDA only; "
                "there is no CPU fallback (put the module in train() mode for the autograd path)")
        self.dev = device
        self.dtype = dtype
        self.plan = lib().yx_plan_create() if use_plan else None
        self.keep: List[torch.Tensor] = []   # buffers and packed weights referenced by the plan
        self.weight_cache: Dict[tuple, Tuple[torch.Tensor, torch.Tensor]] = {}
        self.n_ops = 0
        self.flops = 0.0
        self.op_info: List[dict] = []    # per emitted op: name, algorithmic flops and bytes
        self.writer: Dict[int, int] = {}  # buffer data_ptr -> index of the last main-lane plan op that wrote it
        self._lane = 0

    def close(self):
        if self.plan is not None:
            lib().yx_plan_destroy(self.plan)
            self.plan = None

    def __deepcopy__(self, memo):
        raise TypeError("Builder owns a native plan (raw pointers into its buffers) and cannot be copied; build a new one")

    def __reduce__(self):
        raise TypeError("Builder owns a native plan (raw pointers into its buffers) and cannot be pickled")

    # ---------------------------------------------------------------- independent branches (graph lanes)
    def _wrote(self, feat: Optional["Feat"]) -> None:
        if feat is not None and self.plan is not None and self._lane == 0:
            self.writer[feat.t.data_ptr()] = lib().yx_plan_num_ops(self.plan) - 1

    def begin_lane(self, lane: int, after: Optional["Feat"]) -> None:
        """Ops emitted until end_lane() form an independent branch that only depends on the op that last wrote `after`."""
        if self.plan is None:
            return
        idx = self.writer.get(after.t.data_ptr(), -1) if after is not None else -1
        check(lib().yx_plan_begin_lane(self.plan, lane, idx), "plan_begin_lane")
        self._lane = lane

    def end_lane(self) -> None:
        if self.plan is not None:
            check(lib().yx_plan_end_lane(self.plan), "plan_end_lane")
        self._lane = 0

    def join_lanes(self) -> None:
        if self.plan is not None:
            check(lib().yx_plan_join_lanes(self.plan), "plan_join_lanes")
        self._lane = 0

    # ---------------------------------------------------------------- buffers
    def new_feat(self, B, H, W, segs: Sequence[int]) -> Feat:
        slots = sum(pad16(s) for s in segs)
        needs_zero = any(pad16(s) != s for s in segs)
        alloc = torch.zeros if needs_zero else torch.empty
        t = alloc((B, H, W, slots), dtype=self.dtype, device=self.dev)
        self.keep.append(t)
        return Feat(t, 0, list(segs))

    def from_nchw(self, x: torch.Tensor) -> Feat:
        B, Cc, H, W = x.shape
        f = self.new_feat(B, H, W, [Cc])
        if pad16(Cc) != Cc:
            f.t.zero_()
        f.t[..., :Cc] = x.permute(0, 2, 3, 1).to(self.dtype)
        return f

    # ---------------------------------------------------------------- weights
    def part(self, m, o_off=None, in_segs=None) -> Part:
        if isinstance(m, nn.Conv2d):
            return Part(m.weight, None, m.bias, o_off, in_segs)
        return Part(m.conv.weight, m.bn, m.conv.bias, o_off, in_segs)

    def _pack(self, parts: List[Part], x: Feat, ksize: int, o_total: Optional[int]):
        key = tuple((p.weight.data_ptr(), p.weight._version, p.o_off, tuple(p.in_segs or ())) for p in parts) + (
            tuple(x.segs), self.dtype, o_total)
        hit = self.weight_cache.get(key)
        if hit is not None:
            return hit
        # output rows: explicit offsets (head) or one padded segment per part
        out_segs = []
        if all(p.o_off is None for p in parts):
            off = 0
            for p in parts:
                p.o_off = off
                out_segs.append(p.weight.shape[0])
                off += pad16(p.weight.shape[0])
            O = off
        else:
            O = pad16(o_total)
            out_segs = [o_total]
        I = x.c_slots
        w = torch.zeros((O, ksize * ksize, I), dtype=self.dtype, device=self.dev)
        bias = torch.zeros((O,), dtype=torch.float32, device=self.dev)
        for p in parts:
            segs = p.in_segs if p.in_segs is not None else list(range(len(x.segs)))
            lo = 0
            bn = None
            eps = 0.0
            if p.bn is not None:
                bn = (p.bn.weight, p.bn.bias, p.bn.running_mean, p.bn.running_var)
                eps = p.bn.eps
            assert sum(x.segs[s] for s in segs) == p.weight.shape[1], (
                f"conv expects {p.weight.shape[1]} input channels, segments give {[x.segs[s] for s in segs]}")
            for s in segs:
                n = x.segs[s]
                ops.pack_weights(p.weight[:, lo:lo + n], bn, p.bias, eps, w, bias, o_off=p.o_off, i_off=x.seg_off(s))
                lo += n
        self.keep += [w, bias]
        self.weight_cache[key] = (w, bias, out_segs)
        return w, bias, out_segs

    # ---------------------------------------------------------------- ops
    def conv(self, x: Feat, parts: List[Part], out: Optional[Feat] = None, res: Optional[Feat] = None,
             ups: Optional[Feat] = None, act: Optional[str] = "silu", ksize: int = 1, stride: int = 1,
             o_total: Optional[int] = None, head: Optional[dict] = None, out2: Optional[Feat] = None) -> Optional[Feat]:
        """`out2`: second destination for the trailing output channels (those beyond out.c_slots)."""
        w, bias, out_segs = self._pack(parts, x, ksize, o_total)
        pad = (ksize - 1) // 2
        oh = (x.H + 2 * pad - ksize) // stride + 1
        ow = (x.W + 2 * pad - ksize) // stride + 1
        head_arg = None
        if head is not None:
            ho = head["out"]
            head_arg = dict(out_ptr=ho.data_ptr(), anchors=head["anchors"], anchor_off=head["anchor_off"],
                            nc=head["nc"], decode=head["decode"], stride=head["stride"])
            for k in ("cand_ptr", "keys_ptr", "counts_ptr", "conf_thre", "xyxy"):
                if head.get(k) is not None:
                    head_arg[k] = head[k]
            out_view = None
        else:
            if out is None:
                out = self.new_feat(x.B, oh, ow, out_segs)
            assert out.c_slots + (out2.c_slots if out2 is not None else 0) == w.shape[0], (out.segs, w.shape)
            out_view = out.view()
        d = ops.make_conv_desc(x.view(), w, bias, out_view, ksize, stride, ACT_CODES[act],
                               res.view() if res is not None else None,
                               ups.view() if ups is not None else None, head_arg,
                               out2.view() if out2 is not None else None, out.c_slots if out2 is not None else 0)
        self._emit_conv(d)
        self._wrote(out)
        self._wrote(out2)
        fl = 2.0 * x.B * oh * ow * sum(p.weight.shape[0] * p.weight.shape[1] for p in parts) * ksize * ksize
        esz = w.element_size()
        by = x.B * x.H * x.W * x.c_slots * esz + w.numel() * esz
        by += x.B * oh * ow * (5 + head["nc"]) * 4 if head is not None else x.B * oh * ow * w.shape[0] * esz * (5 if ups is not None else 1)
        if res is not None:
            by += x.B * oh * ow * w.shape[0] * esz
        self.flops += fl
        self.op_info.append(dict(name=f"conv{ksize}x{ksize}s{stride} {x.c_slots}->{w.shape[0]} @{oh}x{ow}", flops=fl, bytes=by,
                                 tc=self.dtype != torch.float32))
        return out

    def probe_feat(self, like: Feat, c: int) -> Feat:
        """A shape-only Feat (no storage of its own) for asking capability questions before allocating."""
        return Feat(like.t, like.c_off, [c])

    def bottleneck_fusable(self, x: Feat, m) -> bool:
        """True when Bottleneck `m` can run as the single fused kernel (yx_bottleneck_fwd)."""
        from .network_blocks import BaseConv

        if self.dtype == torch.float32:
            return False
        c1, c2 = m.conv1, m.conv2
        if not isinstance(c2, BaseConv) or c2.conv.groups != 1 or c2.conv.kernel_size != (3, 3) or c2.conv.stride != (1, 1):
            return False
        c = c1.conv.in_channels
        if not (c1.conv.out_channels == c and c2.conv.in_channels == c and c2.conv.out_channels == c):
            return False
        if type(c1.act) is not type(c2.act) or len(x.segs) != 1 or x.segs[0] != c:
            return False
        # no fused kernel for c = 128: streaming W2 through a 3-stage ring measured 65 us vs 55 us for the unfused pair
        return c in (16, 32, 64)

    def bottleneck(self, x: Feat, m, out: Feat) -> Feat:
        """Fused Bottleneck (1x1 -> 3x3 -> optional shortcut) as one launch; `out` must not alias `x`."""
        from ._lib import BneckDesc
        from .network_blocks import act_name

        w1, b1, _ = self._pack([self.part(m.conv1)], x, 1, None)
        hid = Feat(x.t, x.c_off, list(x.segs))               # same channel structure as the hidden tensor
        w2, b2, _ = self._pack([self.part(m.conv2)], hid, 3, None)
        c = x.segs[0]
        xv, ov = x.view(), out.view()
        d = BneckDesc()
        d.batch, d.h, d.w, d.c = x.B, x.H, x.W, c
        d.dtype = dtype_code(self.dtype)
        d.act = ACT_CODES[act_name(m.conv1.act)]
        d.use_add = 1 if m.use_add else 0
        d.x, d.x_ld = xv.ptr, xv.ld
        d.w1, d.bias1, d.w2, d.bias2 = w1.data_ptr(), b1.data_ptr(), w2.data_ptr(), b2.data_ptr()
        d.out, d.out_ld = ov.ptr, ov.ld
        if self.plan is not None:
            check(lib().yx_plan_add_bottleneck(self.plan, C.byref(d)), "plan_add_bottleneck")
        else:
            check(lib().yx_bottleneck_fwd(C.byref(d), stream_ptr(self.dev)), "bottleneck")
        self._wrote(out)
        self.n_ops += 1
        fl = 2.0 * x.B * x.H * x.W * c * c * 10
        esz = w1.element_size()
        self.flops += fl
        self.op_info.append(dict(name=f"bottleneck {c} @{x.H}x{x.W}", flops=fl,
                                 bytes=2 * x.B * x.H * x.W * c * esz + (w1.numel() + w2.numel()) * esz, tc=True))
        return out

    def _emit_conv(self, d):
        if self.plan is not None:
            check(lib().yx_plan_add_conv(self.plan, C.byref(d)), "plan_add_conv")
        else:
            check(lib().yx_conv_bn_act_fwd(C.byref(d), stream_ptr(self.dev)), "conv")
        self.n_ops += 1

    def dwconv(self, x: Feat, m, out: Optional[Feat] = None) -> Feat:
        """Depthwise 3x3 BaseConv (groups == channels)."""
        conv, bn = m.conv, m.bn
        c = conv.weight.shape[0]
        assert len(x.segs) == 1 and x.segs[0] == c and conv.kernel_size == (3, 3)
        key = (conv.weight.data_ptr(), conv.weight._version, "dw", self.dtype)
        hit = self.weight_cache.get(key)
        if hit is None:
            w = torch.zeros((9, pad16(c)), dtype=self.dtype, device=self.dev)
            bias = torch.zeros((pad16(c),), dtype=torch.float32, device=self.dev)
            ops.pack_weights(conv.weight, (bn.weight, bn.bias, bn.running_mean, bn.running_var), conv.bias, bn.eps,
                             w, bias, depthwise=True)
            self.keep += [w, bias]
            hit = (w, bias)
            self.weight_cache[key] = hit
        w, bias = hit
        stride = conv.stride[0]
        oh = (x.H + 2 - 3) // stride + 1
        ow = (x.W + 2 - 3) // stride + 1
        if out is None:
            out = self.new_feat(x.B, oh, ow, [c])
        from .network_blocks import act_name

        act = ACT_CODES[act_name(m.act)]
        xv, ov = x.view(), out.view()
        if self.plan is not None:
            check(lib().yx_plan_add_dwconv(self.plan, xv.ptr, xv.ld, w.data_ptr(), bias.data_ptr(), ov.ptr, ov.ld,
                                           x.B, x.H, x.W, xv.c, stride, act, dtype_code(self.dtype)), "plan_add_dwconv")
        else:
            ops.dwconv3x3(xv, w, bias, ov, stride, act)
        self._wrote(out)
        self.n_ops += 1
        self.flops += 2.0 * x.B * oh * ow * c * 9
        self.op_info.append(dict(name=f"dwconv3x3s{stride} {c} @{oh}x{ow}", flops=2.0 * x.B * oh * ow * c * 9,
                                 bytes=(x.B * x.H * x.W + x.B * oh * ow) * pad16(c) * w.element_size(), tc=False))
        return out

    def spp(self, cat: Feat, c: int) -> None:
        v = cat.view()
        if pad16(c) != c:
            raise NotImplementedError("SPP with a hidden width that is not a multiple of 16")
        if self.plan is not None:
            check(lib().yx_plan_add_spp(self.plan, v.ptr, v.ld, v.B, v.H, v.W, c, dtype_code(self.dtype)), "plan_add_spp")
        else:
            ops.spp_maxpool(v, c)
        self._wrote(cat)
        self.n_ops += 1
        self.op_info.append(dict(name=f"spp {c} @{v.H}x{v.W}", flops=0.0, bytes=v.B * v.H * v.W * 4 * c * cat.t.element_size(), tc=False))

    def focus(self, img: torch.Tensor) -> Feat:
        B, _, H, W = img.shape
        f = self.new_feat(B, H // 2, W // 2, [12])
        v = f.view()
        if self.plan is not None:
            check(lib().yx_plan_add_focus(self.plan, img.data_ptr(), dtype_code(img.dtype), v.ptr, v.ld,
                                          dtype_code(self.dtype), B, H, W), "plan_add_focus")
        else:
            ops.focus_s2d(img, v)
        self.n_ops += 1
        self.op_info.append(dict(name=f"focus {H}x{W}", flops=0.0,
                                 bytes=img.numel() * img.element_size() + f.t.numel() * f.t.element_size(), tc=False))
        return f

    def focus_conv(self, img: torch.Tensor, m, out: Optional[Feat] = None) -> Feat:
        """Fused Focus + stem BaseConv `m` (3x3, stride 1) on the tensor cores (16-bit paths)."""
        from .network_blocks import act_name

        conv, bn = m.conv, m.bn
        o = conv.weight.shape[0]
        B, _, H, W = img.shape
        key = (conv.weight.data_ptr(), conv.weight._version, "focus", self.dtype)
        hit = self.weight_cache.get(key)
        if hit is None:
            # per filter tap (r, s) of the 3x3 conv on the space-to-depth grid: k = 2*(2*c + py) + px holds Focus channel
            # 3*(2*px + py) + c (network_blocks.py:199-207), k = 12..15 zero; BN folded (model_utils.py:33-75).
            # One-time weight preparation in fp32 torch ops.
            wf = conv.weight.detach().float()
            scale = bn.weight.detach().float() / torch.sqrt(bn.running_var.detach().float() + bn.eps)
            shift = bn.bias.detach().float() - bn.running_mean.detach().float() * scale
            wf = wf * scale[:, None, None, None]
            packed = torch.zeros((pad16(o), 9, 16), dtype=torch.float32, device=wf.device)
            for c in range(3):
                for py in range(2):
                    for px in range(2):
                        packed[:o, :, 2 * (2 * c + py) + px] = wf[:, 3 * (2 * px + py) + c].reshape(o, 9)
            packed = packed.reshape(pad16(o), 144)
            bias = torch.zeros((pad16(o),), dtype=torch.float32, device=self.dev)
            bias[:o] = shift.to(self.dev)
            if self.dtype == torch.float16:
                packed = packed * 256.0      # the kernel feeds pixels as x/256 in fp16 (see yx_stem_tc.cu): keeps the
                                             # BN-folded weights out of fp16's subnormal range
            hit = (packed.to(self.dev).to(self.dtype).contiguous(), bias)
            self.keep += list(hit)
            self.weight_cache[key] = hit
        w, bias = hit
        if out is None:
            out = self.new_feat(B, H // 2, W // 2, [o])
        ov = out.view()
        args = (img.data_ptr(), dtype_code(img.dtype), w.data_ptr(), bias.data_ptr(), ov.ptr, ov.ld, B, H, W, ov.c,
                ACT_CODES[act_name(m.act)], dtype_code(self.dtype))
        if self.plan is not None:
            check(lib().yx_plan_add_focus_conv(self.plan, *args), "plan_add_focus_conv")
        else:
            check(lib().yx_focus_conv_bn_act_fwd(*args, stream_ptr(self.dev)), "focus_conv")
        self._wrote(out)
        self.n_ops += 1
        fl = 2.0 * B * (H // 2) * (W // 2) * o * 108
        self.flops += fl
        self.op_info.append(dict(name=f"focus+conv3x3 3->{o} @{H // 2}x{W // 2}", flops=fl,
                                 bytes=img.numel() * img.element_size() + B * (H // 2) * (W // 2) * ov.c * w.element_size(),
                                 tc=True))
        return out

    def postprocess(self, pred, nc, conf, nms, variant, inplace, dets, det_idx, det_count, max_det, ws):
        check(lib().yx_plan_add_postprocess(self.plan, pred.data_ptr(), pred.shape[0], pred.shape[1], nc, float(conf),
                                            float(nms), int(variant), 1 if inplace else 0, dets.data_ptr(),
                                            det_idx.data_ptr(), det_count.data_ptr(), max_det, ws.data_ptr(),
                                            ws.numel()), "plan_add_postprocess")
        self.keep += [pred, dets, det_idx, det_count, ws]
        self.op_info.append(dict(name="postprocess", flops=0.0, bytes=pred.numel() * 4, tc=False))

    def postprocess_begin(self, ws, batch, anchors):
        """Fused-filter postprocess, part 1: zero the per-image candidate counters before the head GEMMs run."""
        check(lib().yx_plan_add_postprocess_begin(self.plan, ws.data_ptr(), batch, anchors), "plan_add_postprocess_begin")
        self.keep.append(ws)
        self.op_info.append(dict(name="postprocess begin (memset)", flops=0.0, bytes=batch * 4, tc=False))

    def nms_prefiltered(self, batch, anchors, nms, variant, dets, det_idx, det_count, max_det, ws):
        """Fused-filter postprocess, part 2: sort + NMS over the candidates the head epilogues wrote."""
        check(lib().yx_plan_add_nms_prefiltered(self.plan, batch, anchors, float(nms), int(variant), dets.data_ptr(),
                                                det_idx.data_ptr(), det_count.data_ptr(), max_det, ws.data_ptr(),
                                                ws.numel()), "plan_add_nms_prefiltered")
        self.keep += [dets, det_idx, det_count, ws]
        self.op_info.append(dict(name="sort+nms (filter fused in the head)", flops=0.0, bytes=batch * anchors * 32, tc=False))

    def profile(self):
        """Per-op device times (ms) of one eager pass: list of dicts (op_info + ms + kind)."""
        n = lib().yx_plan_num_ops(self.plan)
        ms = (C.c_float * n)()
        kinds = (C.c_int32 * n)()
        check(lib().yx_plan_profile(self.plan, stream_ptr(self.dev), ms, kinds, n), "plan_profile")
        assert n == len(self.op_info), (n, len(self.op_info))
        return [dict(info, ms=float(ms[i]), kind=int(kinds[i])) for i, info in enumerate(self.op_info)]

    def run(self, use_graph: bool = False) -> None:
        check(lib().yx_plan_run(self.plan, stream_ptr(self.dev), 1 if use_graph else 0), "plan_run")

    @property
    def launches(self) -> int:
        return lib().yx_plan_num_launches(self.plan) if self.plan is not None else self.n_ops


# ---------------------------------------------------------------------------------------------
# module-level eval forward (NCHW in / NCHW out like the reference; eager launches)
# ---------------------------------------------------------------------------------------------
def _module_dtype(m: nn.Module, x: torch.Tensor) -> torch.dtype:
    for p in m.parameters():
        return p.dtype
    return x.dtype


def _check_dtype(dt: torch.dtype) -> None:
    if dt not in (torch.bfloat16, torch.float16, torch.float32):
        raise TypeError(f"unsupported module dtype {dt}")


@torch.no_grad()
@_on_device_of(lambda block, x: x.device)
def run_block(block: nn.Module, x: torch.Tensor):
    """Eval forward of a single block through eager C-ABI launches."""
    from .darknet import CspDarknet
    from .network_blocks import Focus
    from .yolo_pafpn import YoloPafpn

    dt = _module_dtype(block, x)
    _check_dtype(dt)
    b = Builder(x.device, dt, use_plan=False)
    if isinstance(block, Focus):
        return block.lower_image(b, x.contiguous()).to_nchw()
    if isinstance(block, CspDarknet):
        feats = block.lower_image(b, x.contiguous())
        return {k: v.to_nchw() for k, v in feats.items() if k in block.out_features}
    if isinstance(block, YoloPafpn):
        return tuple(f.to_nchw() for f in block.lower_image(b, x.contiguous()))
    return block.lower(b, b.from_nchw(x)).to_nchw()


@torch.no_grad()
@_on_device_of(lambda head, xin: xin[0].device)
def run_head(head: nn.Module, xin: Sequence[torch.Tensor]) -> torch.Tensor:
    dt = _module_dtype(head, xin[0])
    _check_dtype(dt)
    b = Builder(xin[0].device, dt, use_plan=False)
    feats = [b.from_nchw(x) for x in xin]
    A = sum(f.H * f.W for f in feats)
    out = torch.empty((xin[0].shape[0], A, 5 + head.num_classes), dtype=torch.float32, device=xin[0].device)
    head.lower(b, feats, out)
    return out if head.output_dtype is None else out.to(head.output_dtype)


# ---------------------------------------------------------------------------------------------
# whole-model engine
# ---------------------------------------------------------------------------------------------
class InferenceEngine:
    """One captured plan per (batch, H, W, input dtype, thresholds): YoloxModule.forward (eval) and,
    optionally, postprocess in the same CUDA graph. The batch is walked in micro-batches that
    share every intermediate buffer, so a micro-batch's activations stay resident in the 126 MB L2
    between producer and consumer layers."""

    @_on_device_of(lambda self, module, batch, height, width, in_dtype, device, *a, **k: device)
    def __init__(self, module: nn.Module, batch: int, height: int, width: int, in_dtype: torch.dtype,
                 device: torch.device, micro_batch: Optional[int] = None, use_graph: bool = True,
                 post: Optional[dict] = None):
        from .yolox import YoloxModule

        assert isinstance(module, YoloxModule)
        if height % 32 or width % 32:
            raise ValueError(f"input size must be a multiple of 32, got {height}x{width}")
        self.module = module
        self.dtype = _module_dtype(module, torch.empty(0))
        _check_dtype(self.dtype)
        self.use_graph = use_graph
        self.batch = batch
        self.mb = min(batch, micro_batch or batch)
        self.builder = Builder(device, self.dtype, use_plan=True)
        b = self.builder
        head = module.head
        strides = head.strides
        self.anchors = sum((height // s) * (width // s) for s in strides)
        self.nc = head.num_classes
        # persistent input staging buffer: the plan's pointers are fixed at build time
        self.input = torch.empty((batch, 3, height, width), dtype=in_dtype, device=device)
        self.pred = torch.empty((batch, self.anchors, 5 + self.nc), dtype=torch.float32, device=device)
        # postprocess in the same graph: on the 16-bit paths the score filter runs inside the decode epilogue of the
        # prediction GEMMs (yx_conv_desc.head_cand) and only sort + NMS remain as a kernel of their own
        self.post = None
        self._post_fused = None
        if post is not None:
            max_det = post.get("max_det") or self.anchors
            self.dets = torch.zeros((batch, max_det, 7), dtype=torch.float32, device=device)
            self.det_idx = torch.zeros((batch, max_det), dtype=torch.int64, device=device)
            self.det_count = torch.zeros((batch,), dtype=torch.int32, device=device)
            self._post_ws = torch.empty((lib().yx_postprocess_workspace_bytes(batch, self.anchors),), dtype=torch.uint8,
                                        device=device)
            self.post = dict(post, max_det=max_det)
            if self.dtype != torch.float32 and head.decode_in_inference:
                cand, keys, counts = ops.postprocess_ws_ptrs(self._post_ws, batch, self.anchors)
                self._post_fused = dict(cand=cand, keys=keys, counts=counts, conf_thre=post["conf_thre"])
                b.postprocess_begin(self._post_ws, batch, self.anchors)
        # intermediate buffers are allocated while lowering the first micro-batch (every Builder.new_feat call is recorded as
        # a slot: call index -> (shape, tensor)) and handed back, slot by slot, to the later micro-batches of the same size
        self._slots = None
        for b0 in range(0, batch, self.mb):
            b1 = min(batch, b0 + self.mb)
            self._lower_slice(self.input[b0:b1], self.pred[b0:b1], b0, record=self._slots is None and b1 - b0 == self.mb,
                              replay=self._slots is not None and b1 - b0 == self.mb)
            b.join_lanes()                       # slices share buffers: the next one starts after every branch is done
        if self.post is not None:
            if self._post_fused is not None:
                b.nms_prefiltered(batch, self.anchors, post["nms_thre"], post["nms_variant"], self.dets, self.det_idx,
                                  self.det_count, self.post["max_det"], self._post_ws)
            else:
                b.postprocess(self.pred, self.nc, post["conf_thre"], post["nms_thre"], post["nms_variant"], True,
                              self.dets, self.det_idx, self.det_count, self.post["max_det"], self._post_ws)
        self.flops_per_image = b.flops / batch

    # buffer reuse across micro-batches: new_feat hands back the tensors of the first lowering
    def _lower(self, img, pred_slice, b0=0):
        m = self.module
        feats = m.backbone.lower_image(self.builder, img)
        post = None
        if self._post_fused is not None:
            f = self._post_fused
            A = self.anchors
            # the in-place corner conversion of postprocess (boxes.py:32-37) happens in the same epilogue
            post = dict(cand_ptr=f["cand"] + b0 * A * 32, keys_ptr=f["keys"] + b0 * A * 8, counts_ptr=f["counts"] + b0 * 4,
                        conf_thre=f["conf_thre"], xyxy=True)
        m.head.lower(self.builder, list(feats), pred_slice, post=post)

    def _lower_slice(self, img, pred_slice, b0, record: bool, replay: bool):
        """Lower one micro-batch. record: remember every buffer new_feat allocates, in call order. replay: the lowering
        makes the same new_feat calls in the same order (same modules, same shapes), so call k gets slot k back; a
        shape mismatch or a different number of calls is an error, never a silent mix-up. A ragged tail allocates its own."""
        b = self.builder
        if not (record or replay):
            return self._lower(img, pred_slice, b0)
        orig_new_feat = b.new_feat
        slots = [] if record else self._slots
        cursor = [0]

        def slotted_new_feat(B, H, W, segs):
            shape = (B, H, W, sum(pad16(s) for s in segs))
            if record:
                f = orig_new_feat(B, H, W, segs)
                slots.append((shape, f.t))
                return f
            if cursor[0] >= len(slots):
                raise RuntimeError(f"buffer replay: micro-batch asks for buffer #{cursor[0]} but the first one allocated {len(slots)}")
            want, t = slots[cursor[0]]
            if want != shape:
                raise RuntimeError(f"buffer replay: slot {cursor[0]} was allocated as {want}, now requested as {shape}")
            cursor[0] += 1
            return Feat(t, 0, list(segs))

        b.new_feat = slotted_new_feat
        try:
            self._lower(img, pred_slice, b0)
        finally:
            b.new_feat = orig_new_feat
        if record:
            self._slots = slots
        elif cursor[0] != len(slots):
            raise RuntimeError(f"buffer replay: micro-batch used {cursor[0]} of {len(slots)} recorded buffers")

    @property
    def launches(self) -> int:
        return self.builder.launches

    @_on_device_of(lambda self, x: self.input.device)
    def forward(self, x: torch.Tensor) -> torch.Tensor:
        """x: [B,3,H,W] on any device (a host tensor is copied H2D here, a device tensor D2D into the persistent input
        buffer the plan's tensor maps point at; pass `engine.input` itself to run on what is already there). Returns
        the engine's own prediction buffer [B, A, 5+nc] fp32 (valid until the next call)."""
        if tuple(x.shape) != tuple(self.input.shape):
            raise ValueError(f"engine built for {tuple(self.input.shape)}, got {tuple(x.shape)}")
        if x.data_ptr() != self.input.data_ptr():        # a caller that fills `engine.input` itself skips the staging copy
            self.input.copy_(x, non_blocking=True)
        self.builder.run(self.use_graph)
        return self.pred

    def close(self):
        self.builder.close()

    def __deepcopy__(self, memo):
        raise TypeError("InferenceEngine is bound to one module's weights and buffers and cannot be copied "
                        "(YoloxModule drops its engine cache on deepcopy / pickle)")

    def __reduce__(self):
        raise TypeError("InferenceEngine cannot be pickled (YoloxModule drops its engine cache on deepcopy / pickle)")
