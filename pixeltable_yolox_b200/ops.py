"""Torch-tensor front end of the C-ABI ops (pointers in, pointers out; no compute in Python).

PyTorch is used for device memory and streams only. Every function here requires CUDA tensors
and raises otherwise: the hot path is hand-written sm_100a CUDA with no CPU fallback.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass
from typing import Optional, Sequence

import torch

from . import _lib
from ._lib import ConvDesc, check, dtype_code, lib, require_cuda, stream_ptr


def same_device(dev: torch.device, what: str, **tensors) -> None:
    """Every tensor whose raw pointer crosses the C-ABI must live on `dev`: a CPU tensor or a tensor of another GPU
    would be an illegal-address fault (sticky CUDA error) instead of the reference's clean device-mismatch error."""
    for name, t in tensors.items():
        if t is not None and t.device != dev:
            raise RuntimeError(f"{what}: `{name}` is on {t.device} but the call runs on {dev}; move it there first "
                               "(the B200 path has no CPU fallback and no implicit peer access)")


def on_device(dev: torch.device):
    """Make `dev` the current CUDA device for the FFI call (the library launches on the current device)."""
    return torch.cuda.device(dev)


@dataclass
class View:
    """A channel slice [c_off, c_off + c) of an NHWC buffer ``t`` of shape [B, H, W, Ctot]."""

    t: torch.Tensor
    c_off: int = 0
    c: Optional[int] = None

    def __post_init__(self):
        assert self.t.dim() == 4 and self.t.is_contiguous()
        if self.c is None:
            self.c = self.t.shape[3] - self.c_off
        assert 0 <= self.c_off and self.c_off + self.c <= self.t.shape[3]

    @property
    def ptr(self) -> int:
        return self.t.data_ptr() + self.c_off * self.t.element_size()

    @property
    def ld(self) -> int:
        return self.t.shape[3]

    @property
    def B(self) -> int:
        return self.t.shape[0]

    @property
    def H(self) -> int:
        return self.t.shape[1]

    @property
    def W(self) -> int:
        return self.t.shape[2]

    def sub(self, off: int, c: int) -> "View":
        return View(self.t, self.c_off + off, c)

    def batch_slice(self, b0: int, b1: int) -> "View":
        return View(self.t[b0:b1], self.c_off, self.c)

    def torch(self) -> torch.Tensor:
        return self.t[..., self.c_off:self.c_off + self.c]


def make_conv_desc(
    x: View, w: torch.Tensor, bias: torch.Tensor, out: Optional[View], ksize: int, stride: int, act: int,
    res: Optional[View] = None, ups: Optional[View] = None, head: Optional[dict] = None,
    out2: Optional[View] = None, out2_begin: int = 0, shuffle2_c: int = 0,
) -> ConvDesc:
    pad = (ksize - 1) // 2
    oh = (x.H + 2 * pad - ksize) // stride + 1
    ow = (x.W + 2 * pad - ksize) // stride + 1
    d = ConvDesc()
    d.batch, d.in_h, d.in_w, d.in_c = x.B, x.H, x.W, x.c
    d.out_h, d.out_w = oh, ow
    d.out_c = w.shape[0]
    d.ksize, d.stride = ksize, stride
    d.dtype = dtype_code(x.t.dtype)
    d.act = act
    d.in_, d.in_ld = x.ptr, x.ld
    assert w.dtype == x.t.dtype and w.is_contiguous() and w.shape[1] == ksize * ksize and w.shape[2] == x.c, (
        w.shape, x.c, ksize)
    assert bias.dtype == torch.float32 and bias.numel() == w.shape[0]
    d.w = w.data_ptr()
    d.bias = bias.data_ptr()
    if head is None:
        assert out is not None and out.t.dtype == x.t.dtype
        if shuffle2_c:                      # depth-to-space store: out is the 2x larger map with a quarter of the channels
            assert d.out_c == 4 * shuffle2_c and out.c == shuffle2_c and (out.B, out.H, out.W) == (x.B, 2 * oh, 2 * ow)
            assert res is None and ups is None and out2 is None
            d.shuffle2_c = shuffle2_c
        else:
            assert out.c == d.out_c or (out2 is not None and out.c == out2_begin), (out.c, d.out_c, out2_begin)
            assert (out.B, out.H, out.W) == (x.B, oh, ow), ((out.B, out.H, out.W), (x.B, oh, ow))
        d.epilogue = _lib.YX_EPI_STORE
        d.out, d.out_ld = out.ptr, out.ld
        if res is not None:
            assert (res.B, res.H, res.W, res.c) == (out.B, out.H, out.W, out.c)
            d.res, d.res_ld = res.ptr, res.ld
        if ups is not None:
            assert (ups.B, ups.H, ups.W, ups.c) == (out.B, 2 * out.H, 2 * out.W, out.c)
            d.ups, d.ups_ld = ups.ptr, ups.ld
        if out2 is not None:
            assert (out2.B, out2.H, out2.W) == (out.B, out.H, out.W) and out2.c == w.shape[0] - out2_begin
            d.out2, d.out2_ld, d.out2_begin = out2.ptr, out2.ld, out2_begin
    else:
        d.epilogue = _lib.YX_EPI_HEAD
        d.head_out = head["out_ptr"]
        d.head_anchors = head["anchors"]
        d.head_anchor_off = head["anchor_off"]
        d.head_nc = head["nc"]
        d.head_decode = head["decode"]
        d.head_stride = float(head["stride"])
        if head.get("cand_ptr"):
            # fused score filter (stage 1 of postprocess) in the decode epilogue
            d.head_cand, d.head_keys, d.head_counts = head["cand_ptr"], head["keys_ptr"], head["counts_ptr"]
            d.head_conf_thre = float(head["conf_thre"])
        d.head_xyxy = 1 if head.get("xyxy") else 0
    return d


def conv_bn_act(x: View, w, bias, out, ksize, stride, act, res=None, ups=None, head=None, simt=False,
                out2=None, out2_begin=0, shuffle2_c=0) -> None:
    require_cuda(x.t, "conv_bn_act")
    d = make_conv_desc(x, w, bias, out, ksize, stride, act, res, ups, head, out2, out2_begin, shuffle2_c)
    same_device(x.t.device, "conv_bn_act", w=w, bias=bias, out=None if out is None else out.t,
                res=None if res is None else res.t, ups=None if ups is None else ups.t, out2=None if out2 is None else out2.t)
    fn = lib().yx_conv_bn_act_fwd_simt if simt else lib().yx_conv_bn_act_fwd
    with on_device(x.t.device):
        check(fn(C.byref(d), stream_ptr(x.t.device)), "conv_bn_act")


def pack_weights(
    src: torch.Tensor, bn: Optional[Sequence[torch.Tensor]], conv_bias: Optional[torch.Tensor], eps: float,
    dst_w: torch.Tensor, dst_b: Optional[torch.Tensor], o_off: int = 0, i_off: int = 0, depthwise: bool = False,
) -> None:
    """BN-fold + repack one nn.Conv2d weight [o,i,kh,kw] into dst_w [O,kh*kw,I] at (o_off, i_off)."""
    require_cuda(dst_w, "pack_weights")
    dev = dst_w.device
    src = src.detach().to(device=dev, dtype=torch.float32).contiguous()
    o, i, kh, kw = src.shape
    ptrs = [0, 0, 0, 0]
    keep = [src]
    if bn is not None:
        for k, t in enumerate(bn):
            t = t.detach().to(device=dev, dtype=torch.float32).contiguous()
            keep.append(t)
            ptrs[k] = t.data_ptr()
    cb = 0
    if conv_bias is not None:
        conv_bias = conv_bias.detach().to(device=dev, dtype=torch.float32).contiguous()
        keep.append(conv_bias)
        cb = conv_bias.data_ptr()
    i_total = dst_w.shape[-1]
    if depthwise:
        assert dst_w.dim() == 2 and dst_w.shape[0] == kh * kw
    else:
        assert dst_w.dim() == 3 and dst_w.shape[1] == kh * kw and o_off + o <= dst_w.shape[0] and i_off + i <= i_total
    check(
        lib().yx_pack_weights(
            src.data_ptr(), ptrs[0], ptrs[1], ptrs[2], ptrs[3], cb, float(eps), o, i, kh, kw, dst_w.data_ptr(),
            dtype_code(dst_w.dtype), o_off, i_off, i_total, dst_b.data_ptr() if dst_b is not None else 0,
            1 if depthwise else 0, stream_ptr(dev)),
        "pack_weights")
    # the source temporaries must outlive the asynchronous kernel
    torch.cuda.current_stream(dev).synchronize()
    del keep


def dwconv3x3(x: View, w: torch.Tensor, bias: torch.Tensor, out: View, stride: int, act: int) -> None:
    require_cuda(x.t, "dwconv3x3")
    assert w.shape == (9, x.c) and out.c == x.c
    check(
        lib().yx_dwconv3x3_bn_act_fwd(x.ptr, x.ld, w.data_ptr(), bias.data_ptr(), out.ptr, out.ld, x.B, x.H, x.W, x.c,
                                      stride, act, dtype_code(x.t.dtype), stream_ptr(x.t.device)),
        "dwconv3x3")


def spp_maxpool(buf: View, c: int) -> None:
    require_cuda(buf.t, "spp_maxpool")
    assert buf.c >= 4 * c
    check(lib().yx_spp_maxpool(buf.ptr, buf.ld, buf.B, buf.H, buf.W, c, dtype_code(buf.t.dtype),
                               stream_ptr(buf.t.device)), "spp_maxpool")


def focus_s2d(img: torch.Tensor, out: View) -> None:
    require_cuda(img, "focus_s2d")
    assert img.dim() == 4 and img.shape[1] == 3 and img.is_contiguous()
    assert out.c_off == 0 and out.ld >= 16
    check(lib().yx_focus_s2d(img.data_ptr(), dtype_code(img.dtype), out.ptr, out.ld, dtype_code(out.t.dtype),
                             img.shape[0], img.shape[2], img.shape[3], stream_ptr(img.device)), "focus_s2d")


def head_decode_(pred: torch.Tensor, hw: Sequence[Sequence[int]], strides: Sequence[int]) -> torch.Tensor:
    require_cuda(pred, "head_decode")
    assert pred.dtype == torch.float32 and pred.is_contiguous() and pred.dim() == 3
    n = len(strides)
    hw_arr = (C.c_int32 * (2 * n))(*[int(v) for pair in hw for v in pair])
    st_arr = (C.c_int32 * n)(*[int(s) for s in strides])
    check(lib().yx_head_decode(pred.data_ptr(), pred.shape[0], pred.shape[1], pred.shape[2] - 5, hw_arr, st_arr, n,
                               stream_ptr(pred.device)), "head_decode")
    return pred


# ---------------------------------------------------------------------------------------------
# postprocess / NMS
# ---------------------------------------------------------------------------------------------
_ws_cache: dict = {}


_ws_retired = {}


def _workspace(dev: torch.device, nbytes: int, tag: str) -> torch.Tensor:
    key = (dev.index, tag)
    ws = _ws_cache.get(key)
    if ws is None or ws.numel() < nbytes:
        if ws is not None and tag.startswith("wgrad"):
            # weight-gradient launches may still be running on the side stream (train_conv): the outgrown buffer stays
            # allocated until the streams are joined, so the caching allocator cannot hand it to another stream
            _ws_retired.setdefault(dev.index, []).append(ws)
        ws = torch.empty(max(nbytes, 256), dtype=torch.uint8, device=dev)
        _ws_cache[key] = ws
    return ws


def release_retired_workspaces(dev: torch.device) -> None:
    _ws_retired.pop(dev.index, None)


def postprocess_device(pred: torch.Tensor, num_classes: int, conf_thre: float, nms_thre: float, nms_variant: int,
                       inplace_xyxy: bool = True, max_det: Optional[int] = None):
    """Returns (dets [B,max_det,7] fp32, det_idx [B,max_det] int64, det_count [B] int32) on device."""
    require_cuda(pred, "postprocess")
    assert pred.dtype == torch.float32 and pred.is_contiguous() and pred.dim() == 3
    B, A, nch = pred.shape
    assert nch == 5 + num_classes
    dev = pred.device
    if max_det is None:
        max_det = A
    dets = torch.empty((B, max_det, 7), dtype=torch.float32, device=dev)
    det_idx = torch.empty((B, max_det), dtype=torch.int64, device=dev)
    det_count = torch.empty((B,), dtype=torch.int32, device=dev)
    if B == 0:
        return dets, det_idx, det_count
    nbytes = lib().yx_postprocess_workspace_bytes(B, A)
    ws = _workspace(dev, nbytes, "post")
    with on_device(dev):
        check(lib().yx_postprocess(pred.data_ptr(), B, A, num_classes, float(conf_thre), float(nms_thre), int(nms_variant),
                                   1 if inplace_xyxy else 0, dets.data_ptr(), det_idx.data_ptr(), det_count.data_ptr(),
                                   max_det, ws.data_ptr(), ws.numel(), stream_ptr(dev)), "postprocess")
    return dets, det_idx, det_count


def postprocess_ws_ptrs(ws: torch.Tensor, batch: int, anchors: int):
    """(cand, keys, counts) device addresses inside a postprocess workspace (yx_postprocess_workspace_ptrs)."""
    cand, keys, counts = C.c_void_p(), C.c_void_p(), C.c_void_p()
    check(lib().yx_postprocess_workspace_ptrs(ws.data_ptr(), batch, anchors, C.byref(cand), C.byref(keys), C.byref(counts)),
          "postprocess_workspace_ptrs")
    return cand.value, keys.value, counts.value


def postprocess_begin(ws: torch.Tensor, batch: int, anchors: int) -> None:
    """Zero the per-image candidate counters of a postprocess workspace (before head GEMMs with a fused filter)."""
    check(lib().yx_postprocess_begin(ws.data_ptr(), batch, anchors, stream_ptr(ws.device)), "postprocess_begin")


def nms_prefiltered(ws: torch.Tensor, batch: int, anchors: int, nms_thre: float, nms_variant: int,
                    max_det: Optional[int] = None):
    """Stage 2 of postprocess over candidates written by the head epilogues; same outputs as postprocess_device."""
    dev = ws.device
    max_det = anchors if max_det is None else max_det
    dets = torch.empty((batch, max_det, 7), dtype=torch.float32, device=dev)
    det_idx = torch.empty((batch, max_det), dtype=torch.int64, device=dev)
    det_count = torch.empty((batch,), dtype=torch.int32, device=dev)
    check(lib().yx_nms_prefiltered(batch, anchors, float(nms_thre), int(nms_variant), dets.data_ptr(), det_idx.data_ptr(),
                                   det_count.data_ptr(), max_det, ws.data_ptr(), ws.numel(), stream_ptr(dev)), "nms_prefiltered")
    return dets, det_idx, det_count


def score_filter_compact(pred: torch.Tensor, num_classes: int, conf_thre: float):
    require_cuda(pred, "score_filter_compact")
    assert pred.dtype == torch.float32 and pred.is_contiguous()
    B, A, _ = pred.shape
    dev = pred.device
    cand = torch.zeros((B, A, 8), dtype=torch.float32, device=dev)
    idx = torch.zeros((B, A), dtype=torch.int32, device=dev)
    cnt = torch.zeros((B,), dtype=torch.int32, device=dev)
    ws = _workspace(dev, lib().yx_postprocess_workspace_bytes(B, A), "post")
    check(lib().yx_score_filter_compact(pred.data_ptr(), B, A, num_classes, float(conf_thre), cand.data_ptr(),
                                        idx.data_ptr(), cnt.data_ptr(), ws.data_ptr(), ws.numel(), stream_ptr(dev)),
          "score_filter_compact")
    return cand, idx, cnt


def batched_nms(boxes: torch.Tensor, scores: torch.Tensor, cls: torch.Tensor, counts: torch.Tensor, nms_thre: float,
                nms_variant: int):
    """boxes [B,n,4] fp32 xyxy, scores [B,n] fp32, cls [B,n] int32, counts [B] int32 -> keep [B,n], keep_count [B]."""
    require_cuda(boxes, "batched_nms")
    B, n, _ = boxes.shape
    dev = boxes.device
    same_device(dev, "batched_nms", scores=scores, cls=cls, counts=counts)
    boxes = boxes.contiguous().float(); scores = scores.contiguous().float()
    cls = cls.contiguous().to(torch.int32); counts = counts.contiguous().to(torch.int32)
    keep = torch.full((B, n), -1, dtype=torch.int32, device=dev)
    keep_count = torch.zeros((B,), dtype=torch.int32, device=dev)
    ws = _workspace(dev, lib().yx_postprocess_workspace_bytes(B, n), "post")
    with on_device(dev):
        check(lib().yx_batched_nms(boxes.data_ptr(), scores.data_ptr(), cls.data_ptr(), counts.data_ptr(), B, n,
                                   float(nms_thre), int(nms_variant), keep.data_ptr(), keep_count.data_ptr(),
                                   ws.data_ptr(), ws.numel(), stream_ptr(dev)), "batched_nms")
    return keep, keep_count


def bboxes_iou_device(a: torch.Tensor, b: torch.Tensor, xyxy: bool) -> torch.Tensor:
    require_cuda(a, "bboxes_iou")
    same_device(a.device, "bboxes_iou", bboxes_b=b)
    a = a.contiguous().float(); b = b.contiguous().float()
    out = torch.empty((a.shape[0], b.shape[0]), dtype=torch.float32, device=a.device)
    with on_device(a.device):
        check(lib().yx_bboxes_iou(a.data_ptr(), a.shape[0], b.data_ptr(), b.shape[0], 1 if xyxy else 0, out.data_ptr(),
                                  stream_ptr(a.device)), "bboxes_iou")
    return out


# ---------------------------------------------------------------------------------------------
# SimOTA
# ---------------------------------------------------------------------------------------------
_LEVELS_CACHE: dict = {}


def _stride_levels(st: torch.Tensor) -> int:
    """Number of distinct strides in the per-anchor stride vector (one device sync, cached per tensor)."""
    key = (st.data_ptr(), st.numel(), st._version, st.device)
    n = _LEVELS_CACHE.get(key)
    if n is None:
        if len(_LEVELS_CACHE) > 64:
            _LEVELS_CACHE.clear()
        n = _LEVELS_CACHE[key] = int(torch.unique(st).numel()) if st.numel() else 1
    return n


def simota_assign(pred: torch.Tensor, labels: torch.Tensor, x_shifts: torch.Tensor, y_shifts: torch.Tensor,
                  strides: torch.Tensor, num_classes: int, levels: Optional[int] = None):
    """Batched get_assignments. Returns dict of dense per-anchor tensors (see include/yx_b200.h)."""
    require_cuda(pred, "simota_assign")
    same_device(pred.device, "simota_assign", labels=labels, x_shifts=x_shifts, y_shifts=y_shifts, strides=strides)
    pred = pred.contiguous().float(); labels = labels.contiguous().float()
    B, A, nch = pred.shape
    assert nch == 5 + num_classes and labels.shape[0] == B and labels.shape[2] == 5
    max_gt = labels.shape[1]
    dev = pred.device
    xs = x_shifts.reshape(-1).contiguous().float(); ys = y_shifts.reshape(-1).contiguous().float()
    st = strides.reshape(-1).contiguous().float()
    assert xs.numel() == A and ys.numel() == A and st.numel() == A
    out = {
        "fg_mask": torch.empty((B, A), dtype=torch.uint8, device=dev),
        "matched_gt": torch.empty((B, A), dtype=torch.int32, device=dev),
        "matched_iou": torch.empty((B, A), dtype=torch.float32, device=dev),
        "matched_cls": torch.empty((B, A), dtype=torch.int32, device=dev),
        "num_fg": torch.empty((B,), dtype=torch.int32, device=dev),
        "num_gt": torch.empty((B,), dtype=torch.int32, device=dev),
        # 0 | YX_SIMOTA_CAPACITY (1) | YX_SIMOTA_BAD_CLASS (2), written by the kernel (no host sync here; callers that
        # already synchronise, e.g. YoloxHead.get_assignments, raise on it)
        "status": torch.zeros((B,), dtype=torch.int32, device=dev),
    }
    if B == 0 or max_gt == 0:
        # the reference accepts any padding length, including none: every anchor is background
        out["fg_mask"].zero_(); out["matched_gt"].fill_(-1); out["matched_iou"].zero_(); out["matched_cls"].fill_(-1)
        out["num_fg"].zero_(); out["num_gt"].zero_()
        return out
    if levels is None:
        levels = _stride_levels(st)
    ws = _workspace(dev, lib().yx_simota_workspace_bytes(B, A, max_gt, levels), "simota")
    with on_device(dev):
        check(lib().yx_simota_assign(pred.data_ptr(), labels.data_ptr(), xs.data_ptr(), ys.data_ptr(), st.data_ptr(), B, A,
                                     num_classes, max_gt, levels, out["fg_mask"].data_ptr(), out["matched_gt"].data_ptr(),
                                     out["matched_iou"].data_ptr(), out["matched_cls"].data_ptr(), out["num_fg"].data_ptr(),
                                     out["num_gt"].data_ptr(), out["status"].data_ptr(), ws.data_ptr(), ws.numel(), stream_ptr(dev)), "simota_assign")
    return out


def head_losses(pred: torch.Tensor, labels: torch.Tensor, asg: dict, origin: Optional[torch.Tensor] = None,
                x_shifts: Optional[torch.Tensor] = None, y_shifts: Optional[torch.Tensor] = None,
                strides: Optional[torch.Tensor] = None, giou: bool = False, reg_weight: float = 5.0):
    """Loss sums and gradients of YoloxHead.get_losses in one kernel (yx_head_losses).
    pred [B,A,5+nc] fp32 (training-branch outputs), labels [B,G,5], asg = simota_assign(...) outputs.
    Returns (sums [4] fp64: iou/obj/cls/l1, un-normalised; grad [B,A,5+nc]; grad_origin [B,A,4] or None)."""
    require_cuda(pred, "head_losses")
    assert pred.dtype == torch.float32 and pred.is_contiguous() and pred.dim() == 3
    B, A, nch = pred.shape
    dev = pred.device
    same_device(dev, "head_losses", labels=labels, origin=origin, x_shifts=x_shifts, y_shifts=y_shifts, strides=strides,
                **{f"asg[{k}]": v for k, v in asg.items() if k in ("fg_mask", "matched_gt", "matched_iou", "matched_cls")})
    labels = labels.contiguous().float()
    sums = torch.empty((4,), dtype=torch.float64, device=dev)
    grad = torch.empty_like(pred)
    g_or = None
    o_ptr = xs_ptr = ys_ptr = st_ptr = go_ptr = None
    if origin is not None:
        origin = origin.contiguous().float()
        xs = x_shifts.reshape(-1).contiguous().float(); ys = y_shifts.reshape(-1).contiguous().float()
        st = strides.reshape(-1).contiguous().float()
        assert origin.shape == (B, A, 4) and xs.numel() == A and ys.numel() == A and st.numel() == A
        g_or = torch.empty_like(origin)
        o_ptr, xs_ptr, ys_ptr, st_ptr, go_ptr = origin.data_ptr(), xs.data_ptr(), ys.data_ptr(), st.data_ptr(), g_or.data_ptr()
    with on_device(dev):
        check(lib().yx_head_losses(pred.data_ptr(), labels.data_ptr(), labels.shape[1], asg["fg_mask"].data_ptr(),
                                   asg["matched_gt"].data_ptr(), asg["matched_iou"].data_ptr(), asg["matched_cls"].data_ptr(),
                                   o_ptr, xs_ptr, ys_ptr, st_ptr, B, A, nch - 5, 1 if giou else 0, float(reg_weight),
                                   sums.data_ptr(), grad.data_ptr(), go_ptr, stream_ptr(dev)), "head_losses")
    return sums, grad, g_or


def simota_matching_device(cost: torch.Tensor, ious: torch.Tensor):
    """simota_matching on a [G, n] cost / IoU pair. Returns (match_gt [n] int32, match_iou [n], num_fg [1])."""
    require_cuda(cost, "simota_matching")
    same_device(cost.device, "simota_matching", ious=ious)
    cost = cost.contiguous().float(); ious = ious.contiguous().float()
    G, n = cost.shape
    dev = cost.device
    mg = torch.empty((n,), dtype=torch.int32, device=dev)
    mi = torch.empty((n,), dtype=torch.float32, device=dev)
    nf = torch.zeros((1,), dtype=torch.int32, device=dev)
    check(lib().yx_simota_matching(cost.data_ptr(), ious.data_ptr(), G, n, n, mg.data_ptr(), mi.data_ptr(),
                                   nf.data_ptr(), stream_ptr(dev)), "simota_matching")
    return mg, mi, nf


def bottleneck_fwd(x: View, w1: torch.Tensor, b1: torch.Tensor, w2: torch.Tensor, b2: torch.Tensor, out: View,
                   act: int, use_add: bool) -> None:
    """Fused Bottleneck (network_blocks.py:77-99): out = [x +] act(conv3x3(act(conv1x1(x)))); w1 [c,1,c], w2 [c,9,c]."""
    from ._lib import BneckDesc

    require_cuda(x.t, "bottleneck_fwd")
    d = BneckDesc()
    d.batch, d.h, d.w, d.c = x.B, x.H, x.W, x.c
    d.dtype = dtype_code(x.t.dtype)
    d.act = act
    d.use_add = 1 if use_add else 0
    d.x, d.x_ld = x.ptr, x.ld
    d.w1, d.bias1, d.w2, d.bias2 = w1.data_ptr(), b1.data_ptr(), w2.data_ptr(), b2.data_ptr()
    d.out, d.out_ld = out.ptr, out.ld
    check(lib().yx_bottleneck_fwd(C.byref(d), stream_ptr(x.t.device)), "bottleneck_fwd")


# ---------------------------------------------------------------------------------------------
# training branch rows, optimizer + EMA, preprocessing, evaluator rows
# ---------------------------------------------------------------------------------------------
def head_train_decode(reg: torch.Tensor, obj: torch.Tensor, cls: torch.Tensor, stride: float, out: torch.Tensor,
                      anchor_off: int, origin: Optional[torch.Tensor] = None) -> None:
    """One level of the training branch (yolo_head.py:161-201, 213-231): NCHW conv outputs -> decoded fp32 rows
    [anchor_off, anchor_off + h*w) of `out` [B, A, 5+nc] (and the raw regression rows of `origin` [B, A, 4])."""
    require_cuda(reg, "head_train_decode")
    dev = reg.device
    same_device(dev, "head_train_decode", obj=obj, cls=cls, out=out, origin=origin)
    B, _, h, w = reg.shape
    nc = cls.shape[1]
    assert reg.shape[1] == 4 and obj.shape[1] == 1 and reg.dtype == obj.dtype == cls.dtype
    assert reg.is_contiguous() and obj.is_contiguous() and cls.is_contiguous() and out.is_contiguous() and out.dtype == torch.float32
    assert out.shape[0] == B and out.shape[2] == 5 + nc and (origin is None or (origin.is_contiguous() and origin.dtype == torch.float32))
    with on_device(dev):
        check(lib().yx_head_train_decode(reg.data_ptr(), obj.data_ptr(), cls.data_ptr(), dtype_code(reg.dtype), B, nc, h, w,
                                         float(stride), out.shape[1], int(anchor_off), out.data_ptr(),
                                         0 if origin is None else origin.data_ptr(), stream_ptr(dev)), "head_train_decode")


def head_train_decode_bwd(grad_out: torch.Tensor, out: torch.Tensor, grad_origin: Optional[torch.Tensor], stride: float,
                          anchor_off: int, g_reg: torch.Tensor, g_obj: torch.Tensor, g_cls: torch.Tensor) -> None:
    dev = grad_out.device
    same_device(dev, "head_train_decode_bwd", out=out, grad_origin=grad_origin, g_reg=g_reg, g_obj=g_obj, g_cls=g_cls)
    B, _, h, w = g_reg.shape
    assert grad_out.is_contiguous() and out.is_contiguous() and grad_out.dtype == out.dtype == torch.float32
    with on_device(dev):
        check(lib().yx_head_train_decode_bwd(grad_out.data_ptr(), out.data_ptr(), 0 if grad_origin is None else grad_origin.data_ptr(),
                                             dtype_code(g_reg.dtype), B, g_cls.shape[1], h, w, float(stride), out.shape[1],
                                             int(anchor_off), g_reg.data_ptr(), g_obj.data_ptr(), g_cls.data_ptr(),
                                             stream_ptr(dev)), "head_train_decode_bwd")


def sgd_ema_step(table: torch.Tensor, chunks: torch.Tensor, chunk_elems: int, lr: float, momentum: float, nesterov: bool,
                 first_step: bool, ema_decay: float, hyper: Optional[torch.Tensor] = None) -> None:
    """One launch over every tensor of `table` (see include/yx_b200.h: yx_sgd_ema_step). `hyper`: device fp32[3]
    {lr, ema_decay, 1 - ema_decay} read by the kernel instead of the arguments (CUDA-graph replay)."""
    import numpy as np

    dev = table.device
    same_device(dev, "sgd_ema_step", chunks=chunks)
    with on_device(dev):
        check(lib().yx_sgd_ema_step(table.data_ptr(), chunks.data_ptr(), chunks.shape[0], int(chunk_elems), float(lr), float(momentum),
                                    1 if nesterov else 0, 1 if first_step else 0, float(np.float32(ema_decay)),
                                    float(np.float32(1.0 - ema_decay)), 0 if hyper is None else hyper.data_ptr(), stream_ptr(dev)),
              "sgd_ema_step")


def letterbox_u8(images, size, device: torch.device, dtype: torch.dtype = torch.uint8) -> torch.Tensor:
    """`preproc` (data_augment.py:140-156) for a list of decoded HWC (or HW) uint8 numpy images, on the device: the raw bytes
    are packed into one pinned buffer, uploaded with one copy and resized / padded / transposed by one launch. Returns
    [B, C, H, W] uint8 or float32 (0..255)."""
    import numpy as np

    if device.type != "cuda":
        raise RuntimeError("letterbox_u8 needs a CUDA device (the B200 path has no CPU fallback; use processor.letterbox on the host)")
    H, W = int(size[0]), int(size[1])
    imgs = [np.ascontiguousarray(im if im.ndim == 3 else im[..., None]) for im in images]
    ch = imgs[0].shape[2]
    assert all(im.dtype == np.uint8 and im.shape[2] == ch for im in imgs), "letterbox_u8: uint8 images with the same channel count"
    offs, total = [], 0
    for im in imgs:
        offs.append(total)
        total += (im.size + 255) & ~255
    host = torch.empty(total + 24 * len(imgs), dtype=torch.uint8).pin_memory()
    hv = host.numpy()
    for im, o in zip(imgs, offs):
        hv[o:o + im.size] = im.reshape(-1)
    raw = host.to(device, non_blocking=True)
    base = raw.data_ptr()
    table = np.zeros((len(imgs), 3), dtype=np.int64)            # yx_letterbox_image: ptr | (h, w) packed | pitch
    for i, (im, o) in enumerate(zip(imgs, offs)):
        table[i, 0] = base + o
        table[i, 1] = int(im.shape[0]) | (int(im.shape[1]) << 32)
        table[i, 2] = im.shape[1] * ch
    tdev = torch.from_numpy(table).to(device)
    out = torch.empty((len(imgs), ch, H, W), dtype=dtype, device=device)
    with on_device(device):
        check(lib().yx_letterbox_u8(tdev.data_ptr(), len(imgs), ch, H, W, out.data_ptr(), dtype_code(dtype), stream_ptr(device)),
              "letterbox_u8")
    out._yx_keepalive = (raw, tdev)      # the launch is asynchronous: keep the sources alive with the result
    return out


def coco_rows(dets: torch.Tensor, det_count: torch.Tensor, scale: torch.Tensor, image_ids: torch.Tensor,
              class_ids: Optional[torch.Tensor] = None):
    """Device half of convert_to_coco_format (coco_evaluator.py:205-251). Returns (bbox_xywh [N,4], score [N], category [N],
    image_id [N]) as HOST tensors after one device->host copy."""
    require_cuda(dets, "coco_rows")
    dev = dets.device
    B, max_det, _ = dets.shape
    dets = dets.contiguous().float()
    det_count = det_count.contiguous().to(torch.int32)
    scale = scale.to(dev).contiguous().float()
    image_ids = image_ids.to(dev).contiguous().to(torch.int64)
    cid = None if class_ids is None else class_ids.to(dev).contiguous().to(torch.int32)
    n = B * max_det
    bbox = torch.empty((n, 4), dtype=torch.float32, device=dev)
    score = torch.empty((n,), dtype=torch.float32, device=dev)
    cat = torch.empty((n,), dtype=torch.int32, device=dev)
    iid = torch.empty((n,), dtype=torch.int64, device=dev)
    total = torch.zeros((1,), dtype=torch.int32, device=dev)
    with on_device(dev):
        check(lib().yx_coco_rows(dets.data_ptr(), det_count.data_ptr(), B, max_det, scale.data_ptr(), image_ids.data_ptr(),
                                 0 if cid is None else cid.data_ptr(), 0 if cid is None else cid.numel(), bbox.data_ptr(),
                                 score.data_ptr(), cat.data_ptr(), iid.data_ptr(), total.data_ptr(), stream_ptr(dev)), "coco_rows")
    k = int(total.item())
    return bbox[:k].cpu(), score[:k].cpu(), cat[:k].cpu(), iid[:k].cpu()


def _is_channels_last(x: torch.Tensor) -> bool:
    """Dense NHWC memory (torch.channels_last) that is not also plain NCHW-contiguous, with a channel count the 16-byte
    channel vectors of the channels-last kernels can take."""
    return (x.dim() == 4 and not x.is_contiguous() and x.is_contiguous(memory_format=torch.channels_last) and x.shape[1] % 8 == 0)


def bn_act_train_fwd(x: torch.Tensor, gamma: torch.Tensor, beta: torch.Tensor, running_mean: Optional[torch.Tensor],
                     running_var: Optional[torch.Tensor], eps: float, momentum: float, act: int,
                     num_batches_tracked: Optional[torch.Tensor] = None):
    """Training-mode BatchNorm2d + activation on a conv output x [N, C, H, W] (contiguous NCHW). Returns
    (y, save_mean, save_invstd); running statistics are updated in place like F.batch_norm."""
    require_cuda(x, "bn_act_train_fwd")
    dev = x.device
    same_device(dev, "bn_act_train_fwd", gamma=gamma, beta=beta, running_mean=running_mean, running_var=running_var,
                num_batches_tracked=num_batches_tracked)
    assert num_batches_tracked is None or (num_batches_tracked.dtype == torch.int64 and num_batches_tracked.numel() == 1)
    cl = _is_channels_last(x)
    assert x.dim() == 4 and (cl or x.is_contiguous()) and gamma.dtype == beta.dtype == torch.float32
    N, Cc, H, W = x.shape
    y = torch.empty_like(x)                  # preserves the memory format
    mean = torch.empty((Cc,), dtype=torch.float32, device=dev)
    invstd = torch.empty((Cc,), dtype=torch.float32, device=dev)
    nbytes = lib().yx_bn_act_workspace_bytes(N, Cc, H * W)
    ws = _workspace(dev, nbytes, f"bn:{stream_ptr(dev)}")          # per stream: branches of the step run concurrently
    with on_device(dev):
        check(lib().yx_bn_act_train_fwd(x.data_ptr(), dtype_code(x.dtype), 1 if cl else 0, N, Cc, H * W, gamma.data_ptr(), beta.data_ptr(),
                                        float(eps), float(momentum), 0 if running_mean is None else running_mean.data_ptr(),
                                        0 if running_var is None else running_var.data_ptr(),
                                        0 if num_batches_tracked is None else num_batches_tracked.data_ptr(), int(act), y.data_ptr(),
                                        mean.data_ptr(), invstd.data_ptr(), ws.data_ptr(), ws.numel(), stream_ptr(dev)),
              "bn_act_train_fwd")
    return y, mean, invstd


def bn_act_train_bwd(x: torch.Tensor, dy: torch.Tensor, gamma: torch.Tensor, beta: torch.Tensor, mean: torch.Tensor,
                     invstd: torch.Tensor, act: int, acc_dgamma: Optional[torch.Tensor] = None,
                     acc_dbeta: Optional[torch.Tensor] = None):
    """Backward of bn_act_train_fwd: (dx in x's dtype, dgamma, dbeta fp32). acc_dgamma / acc_dbeta: contiguous fp32 [C]
    tensors (the parameters' .grad) that dgamma / dbeta are also added to, in the same launch."""
    dev = x.device
    same_device(dev, "bn_act_train_bwd", dy=dy, gamma=gamma, beta=beta, mean=mean, invstd=invstd, acc_dgamma=acc_dgamma,
                acc_dbeta=acc_dbeta)
    for t in (acc_dgamma, acc_dbeta):
        assert t is None or (t.dtype == torch.float32 and t.is_contiguous() and t.numel() == x.shape[1])
    cl = _is_channels_last(x)
    N, Cc, H, W = x.shape
    dy_ld = 0
    if cl and dy.stride() != x.stride():
        dy_ld = dy.stride(3)               # a channel slice of a wider channels_last tensor (the backward of torch.cat)
        assert dy.stride() == (H * W * dy_ld, 1, W * dy_ld, dy_ld) and dy_ld % 8 == 0 and dy.data_ptr() % 16 == 0, "dy layout"
    else:
        assert dy.stride() == x.stride(), "dy must have x's memory format"
    assert dy.dtype == x.dtype and dy.shape == x.shape
    dx = torch.empty_like(x)
    dgamma = torch.empty((Cc,), dtype=torch.float32, device=dev)
    dbeta = torch.empty((Cc,), dtype=torch.float32, device=dev)
    ws = _workspace(dev, lib().yx_bn_act_workspace_bytes(N, Cc, H * W), f"bn:{stream_ptr(dev)}")
    with on_device(dev):
        check(lib().yx_bn_act_train_bwd(x.data_ptr(), dy.data_ptr(), dtype_code(x.dtype), 1 if cl else 0, N, Cc, H * W, gamma.data_ptr(),
                                        beta.data_ptr(), mean.data_ptr(), invstd.data_ptr(), int(act), dx.data_ptr(),
                                        dgamma.data_ptr(), dbeta.data_ptr(), 0 if acc_dgamma is None else acc_dgamma.data_ptr(),
                                        0 if acc_dbeta is None else acc_dbeta.data_ptr(), dy_ld, ws.data_ptr(), ws.numel(),
                                        stream_ptr(dev)),
              "bn_act_train_bwd")
    return dx, dgamma, dbeta


# ------------------------------------------------------------------------------------------ training conv stack
def _nhwc(t: torch.Tensor) -> View:
    """[B, C, H, W] tensor in dense channels_last memory -> the NHWC View the conv kernels take."""
    assert t.dim() == 4 and t.is_contiguous(memory_format=torch.channels_last), "expected dense channels_last memory"
    return View(t.permute(0, 2, 3, 1))


def _weight_strides(w: torch.Tensor):
    """(stride_o, stride_i, stride_tap) of an nn.Conv2d weight [o, i, kh, kw], tap = kw_count * kh + kw; holds for
    NCHW-contiguous and channels_last weights alike."""
    o, i, kh, kw = w.shape
    so, si, sh, sw = w.stride()
    if kh * kw > 1:
        assert sh == kw * sw, "conv weight: the filter taps are not linearly strided"
    return so, si, sw


def pack_train_weights(weight: torch.Tensor, dtype: torch.dtype, o_pad: int, i_pad: int, want_dgrad: bool, subpixel: bool = False):
    """fp32 conv weight -> (w_fwd [o_pad, taps, i_pad], w_dgrad [i_pad, taps, o_pad] or None) in `dtype`, one launch.
    subpixel (3x3 stride-2 convs): w_dgrad is [4 * i_pad, 9, o_pad], the transposed conv as one stride-1 conv over dy whose
    output is stored depth-to-space (conv_bn_act(..., shuffle2_c=i_pad))."""
    require_cuda(weight, "pack_train_weights")
    dev = weight.device
    assert weight.dtype == torch.float32 and weight.dim() == 4
    o, i, kh, kw = weight.shape
    taps = kh * kw
    wf = torch.empty((o_pad, taps, i_pad), dtype=dtype, device=dev)
    wd = None
    if want_dgrad:
        wd = (torch.zeros((4 * i_pad, 9, o_pad), dtype=dtype, device=dev) if subpixel
              else torch.empty((i_pad, taps, o_pad), dtype=dtype, device=dev))
    so, si, st = _weight_strides(weight)
    with on_device(dev):
        check(lib().yx_pack_train_weights(weight.data_ptr(), so, si, st, o, i, taps, o_pad, i_pad, wf.data_ptr(),
                                          0 if wd is None else wd.data_ptr(), 1 if subpixel else 0, dtype_code(dtype),
                                          stream_ptr(dev)),
              "pack_train_weights")
    return wf, wd


def conv_wgrad(x: torch.Tensor, dy: torch.Tensor, weight_like: torch.Tensor, ksize: int, stride: int,
               accumulate_into: Optional[torch.Tensor] = None) -> torch.Tensor:
    """dW of y = conv(x, W): x [B, Ci_pad, H, W], dy [B, Co_pad, OH, OW], both 16-bit dense channels_last with channel
    counts padded to multiples of 16; returns fp32 dW with weight_like's shape [o, i, k, k] and strides.
    accumulate_into: an fp32 tensor of the weight's shape (its .grad): dW is ADDED to it in place and returned."""
    require_cuda(x, "conv_wgrad")
    dev = x.device
    same_device(dev, "conv_wgrad", dy=dy, weight=weight_like)
    xv, dv = _nhwc(x), _nhwc(dy)
    assert x.dtype == dy.dtype and x.dtype in (torch.bfloat16, torch.float16)
    o, i = weight_like.shape[0], weight_like.shape[1]
    assert i <= xv.c and o <= dv.c and xv.B == dv.B
    if accumulate_into is not None:
        dw = accumulate_into
        assert dw.dtype == torch.float32 and dw.shape == weight_like.shape and dw.device == dev
    else:
        dw = torch.empty_strided(weight_like.shape, weight_like.stride(), dtype=torch.float32, device=dev)
    so, si, st = _weight_strides(dw)
    args = (xv.B, xv.H, xv.W, xv.c, dv.H, dv.W, dv.c, ksize, stride)
    nbytes = lib().yx_conv_wgrad_workspace_bytes(*args)
    if nbytes < 0:
        check(-1, "conv_wgrad (workspace query)")
    ws = _workspace(dev, nbytes, f"wgrad:{stream_ptr(dev)}")        # per stream: wgrad launches of several layers run concurrently
    with on_device(dev):
        check(lib().yx_conv_wgrad(xv.ptr, xv.ld, dv.ptr, dv.ld, dtype_code(x.dtype), *args, i, o, dw.data_ptr(), so, si, st,
                                  0 if accumulate_into is None else 1, ws.data_ptr(), ws.numel(), stream_ptr(dev)), "conv_wgrad")
    return dw


def _dw_weight_strides(w: torch.Tensor):
    """(stride_c, stride_tap) of a depthwise conv weight (or its gradient) [c, 1, 3, 3]."""
    assert w.dim() == 4 and w.shape[1:] == (1, 3, 3) and w.dtype == torch.float32, (w.shape, w.dtype)
    sc, _, st = _weight_strides(w)
    return sc, st


def dwconv_train_fwd(x: torch.Tensor, weight: torch.Tensor, stride: int) -> torch.Tensor:
    """Depthwise 3x3 conv (pad 1, no bias) of the training step: x [B, c, H, W] 16-bit dense channels_last, weight the fp32
    parameter [c, 1, 3, 3] (any strides; rounded to x's dtype as the kernel reads it) -> y [B, c, OH, OW] channels_last."""
    require_cuda(x, "dwconv_train_fwd")
    dev = x.device
    same_device(dev, "dwconv_train_fwd", weight=weight)
    xv = _nhwc(x)
    sc, st = _dw_weight_strides(weight)
    assert weight.shape[0] == xv.c and x.dtype in (torch.bfloat16, torch.float16)
    oh, ow = (xv.H - 1) // stride + 1, (xv.W - 1) // stride + 1
    y = torch.empty((xv.B, xv.c, oh, ow), dtype=x.dtype, device=dev, memory_format=torch.channels_last)
    yv = _nhwc(y)
    with on_device(dev):
        check(lib().yx_dwconv3x3_train_fwd(xv.ptr, xv.ld, weight.data_ptr(), sc, st, yv.ptr, yv.ld, xv.B, xv.H, xv.W, xv.c, stride,
                                           dtype_code(x.dtype), stream_ptr(dev)), "dwconv3x3_train_fwd")
    return y


def dwconv_dgrad(dy: torch.Tensor, weight: torch.Tensor, stride: int, in_h: int, in_w: int) -> torch.Tensor:
    """Input gradient of dwconv_train_fwd: dy [B, c, OH, OW] 16-bit dense channels_last -> dx [B, c, in_h, in_w] (same)."""
    require_cuda(dy, "dwconv_dgrad")
    dev = dy.device
    same_device(dev, "dwconv_dgrad", weight=weight)
    dv = _nhwc(dy)
    sc, st = _dw_weight_strides(weight)
    assert weight.shape[0] == dv.c and dy.dtype in (torch.bfloat16, torch.float16)
    assert (dv.H, dv.W) == ((in_h - 1) // stride + 1, (in_w - 1) // stride + 1), ((dv.H, dv.W), (in_h, in_w), stride)
    dx = torch.empty((dv.B, dv.c, in_h, in_w), dtype=dy.dtype, device=dev, memory_format=torch.channels_last)
    xv = _nhwc(dx)
    with on_device(dev):
        check(lib().yx_dwconv3x3_dgrad(dv.ptr, dv.ld, weight.data_ptr(), sc, st, xv.ptr, xv.ld, xv.B, in_h, in_w, xv.c, stride,
                                       dtype_code(dy.dtype), stream_ptr(dev)), "dwconv3x3_dgrad")
    return dx


def dwconv_wgrad(x: torch.Tensor, dy: torch.Tensor, weight_like: torch.Tensor, stride: int,
                 accumulate_into: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Weight gradient of dwconv_train_fwd: x [B, c, H, W] and dy [B, c, OH, OW], both 16-bit dense channels_last -> fp32 dW
    with weight_like's shape [c, 1, 3, 3] and strides; deterministic. accumulate_into: an fp32 tensor of the weight's shape
    (its .grad): dW is ADDED to it in place and returned."""
    require_cuda(x, "dwconv_wgrad")
    dev = x.device
    same_device(dev, "dwconv_wgrad", dy=dy, weight=weight_like)
    xv, dv = _nhwc(x), _nhwc(dy)
    assert x.dtype == dy.dtype and x.dtype in (torch.bfloat16, torch.float16)
    assert xv.B == dv.B and xv.c == dv.c == weight_like.shape[0]
    assert (dv.H, dv.W) == ((xv.H - 1) // stride + 1, (xv.W - 1) // stride + 1)
    if accumulate_into is not None:
        dw = accumulate_into
        assert dw.dtype == torch.float32 and dw.shape == weight_like.shape and dw.device == dev
    else:
        dw = torch.empty_strided(weight_like.shape, weight_like.stride(), dtype=torch.float32, device=dev)
    sc, st = _dw_weight_strides(dw)
    nbytes = lib().yx_dwconv3x3_wgrad_workspace_bytes(xv.B, xv.H, xv.W, xv.c, stride)
    if nbytes < 0:
        check(-1, "dwconv3x3_wgrad (workspace query)")
    ws = _workspace(dev, nbytes, f"wgrad:{stream_ptr(dev)}")        # per stream, shared with conv_wgrad (same-stream launches serialise)
    with on_device(dev):
        check(lib().yx_dwconv3x3_wgrad(xv.ptr, xv.ld, dv.ptr, dv.ld, dtype_code(x.dtype), xv.B, xv.H, xv.W, xv.c, stride,
                                       dw.data_ptr(), sc, st, 0 if accumulate_into is None else 1, ws.data_ptr(), ws.numel(),
                                       stream_ptr(dev)), "dwconv3x3_wgrad")
    return dw


def dilate2(dy: torch.Tensor, zh: int, zw: int) -> torch.Tensor:
    """Zero-stuffed copy of dy [B, C, OH, OW] (channels_last): z [B, C, zh, zw] with z[..., 2*oy, 2*ox] = dy[..., oy, ox]."""
    require_cuda(dy, "dilate2")
    dv = _nhwc(dy)
    z = torch.empty((dv.B, dv.c, zh, zw), dtype=dy.dtype, device=dy.device, memory_format=torch.channels_last)
    with on_device(dy.device):
        check(lib().yx_dilate2(dv.ptr, z.data_ptr(), dv.B, dv.H, dv.W, zh, zw, dv.c, stream_ptr(dy.device)), "dilate2")
    return z


def spp_maxpool_bwd(cat: torch.Tensor, dout: torch.Tensor) -> torch.Tensor:
    """Backward of cat[x, m5, m9, m13]: cat [B, 4c, H, W] (the forward's output, channels [0, c) = x) and its gradient, both
    dense channels_last 16-bit -> dx [B, c, H, W] (channels_last, same dtype)."""
    require_cuda(cat, "spp_maxpool_bwd")
    same_device(cat.device, "spp_maxpool_bwd", dout=dout)
    cv, dv = _nhwc(cat), _nhwc(dout)
    assert cat.shape == dout.shape and cat.dtype == dout.dtype and cv.c % 4 == 0
    c = cv.c // 4
    dx32 = dout[:, :c].to(torch.float32, memory_format=torch.channels_last)
    with on_device(cat.device):
        check(lib().yx_spp_maxpool_bwd(cv.ptr, cv.ld, dv.ptr, dv.ld, dx32.data_ptr(), cv.B, cv.H, cv.W, c, dtype_code(cat.dtype),
                                       stream_ptr(cat.device)), "spp_maxpool_bwd")
    return dx32.to(cat.dtype)


def allreduce_sgd_ema_step(table: torch.Tensor, chunks: torch.Tensor, chunk_elems: int, momentum: float, nesterov: bool,
                           first_step: bool, hyper: torch.Tensor, peer_grad_ptrs, peer_flag_ptrs, flat_elems: int, rank: int,
                           world: int, state: torch.Tensor) -> None:
    """Gradient all-reduce over NVLink peer memory fused with the SGD + EMA update (csrc/yx_allreduce_sgd.cu). peer_*_ptrs:
    sequences of `world` integer addresses (this rank's mapping of every rank's symmetric buffer)."""
    require_cuda(table, "allreduce_sgd_ema_step")
    dev = table.device
    same_device(dev, "allreduce_sgd_ema_step", chunks=chunks, hyper=hyper, state=state)
    assert len(peer_grad_ptrs) == world and len(peer_flag_ptrs) == world and state.dtype == torch.int32 and state.numel() >= 4
    pg = (C.c_int64 * world)(*[int(v) for v in peer_grad_ptrs])
    pf = (C.c_int64 * world)(*[int(v) for v in peer_flag_ptrs])
    with on_device(dev):
        check(lib().yx_allreduce_sgd_ema_step(table.data_ptr(), chunks.data_ptr(), chunks.shape[0], int(chunk_elems), float(momentum),
                                              1 if nesterov else 0, 1 if first_step else 0, hyper.data_ptr(), pg, pf, int(flat_elems),
                                              int(rank), int(world), state.data_ptr(), stream_ptr(dev)), "allreduce_sgd_ema_step")
