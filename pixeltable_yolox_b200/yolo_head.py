"""Decoupled YOLOX head with the reference's interface (yolox/models/yolo_head.py:17-574).

eval  : lowered onto the B200 plan; the three prediction convs of a level are one implicit GEMM
        with block-diagonal weights whose epilogue applies sigmoid/decode and writes the final
        fp32 [B, A, 5+nc] tensor directly (yolo_head.py:185-187, 203-211, 233-251).
train : the network runs through PyTorch autograd; the SimOTA assignment of the whole batch is a
        single launch of the sm_100a kernel (no per-image Python loop, no host sync), and the
        losses are assembled from its dense per-anchor outputs (yolo_head.py:253-411).
"""
from __future__ import annotations

import math

import torch
import torch.nn as nn
import torch.nn.functional as F

from . import ops
from .losses import IouLoss
from .network_blocks import BaseConv, DWConv, _B200Block, act_name


class _FusedHeadLoss(torch.autograd.Function):
    """total = reg_weight * iou_sum + obj_sum + cls_sum (+ l1_sum), un-normalised, with the gradient produced by the same
    kernel launch that produced the value (ops.head_losses). `sums` (iou, obj, cls, l1) is returned for reporting."""

    @staticmethod
    def forward(ctx, pred, origin, labels, asg, x_shifts, y_shifts, strides, giou, reg_weight):
        sums, grad, g_or = ops.head_losses(pred, labels, asg, origin, x_shifts, y_shifts, strides, giou, reg_weight)
        ctx.save_for_backward(grad, g_or if g_or is not None else grad.new_empty(0))
        ctx.has_origin = origin is not None
        sums = sums.to(torch.float32)
        total = reg_weight * sums[0] + sums[1] + sums[2] + sums[3]
        ctx.mark_non_differentiable(sums)
        return total, sums

    @staticmethod
    def backward(ctx, g_total, _g_sums):
        grad, g_or = ctx.saved_tensors
        return (grad * g_total, g_or * g_total if ctx.has_origin else None, None, None, None, None, None, None, None)


class _TrainRows(torch.autograd.Function):
    """One level of the training branch (yolo_head.py:161-201 + get_output_and_grid :213-231) as one kernel each way:
    (reg, obj, cls) NCHW conv outputs -> decoded fp32 rows [B, h*w, 5+nc] (+ the raw regression rows for the L1 term)."""

    @staticmethod
    def forward(ctx, reg, obj, cls, stride, want_origin):
        B, _, h, w = reg.shape
        reg, obj, cls = reg.contiguous(), obj.contiguous(), cls.contiguous()
        out = torch.empty((B, h * w, 5 + cls.shape[1]), dtype=torch.float32, device=reg.device)
        origin = torch.empty((B, h * w, 4), dtype=torch.float32, device=reg.device) if want_origin else None
        ops.head_train_decode(reg, obj, cls, stride, out, 0, origin)
        ctx.save_for_backward(out)
        ctx.meta = (float(stride), tuple(reg.shape), tuple(obj.shape), tuple(cls.shape), reg.dtype, want_origin)
        if not want_origin:
            origin = out.new_empty(0)
            ctx.mark_non_differentiable(origin)
        return out, origin

    @staticmethod
    def backward(ctx, g_out, g_origin):
        (out,) = ctx.saved_tensors
        stride, s_reg, s_obj, s_cls, dt, want_origin = ctx.meta
        dev = out.device
        g_reg, g_obj, g_cls = (torch.empty(sh, dtype=dt, device=dev) for sh in (s_reg, s_obj, s_cls))
        g_out = torch.zeros_like(out) if g_out is None else g_out.contiguous().float()
        g_or = g_origin.contiguous().float() if (want_origin and g_origin is not None) else None
        ops.head_train_decode_bwd(g_out, out, g_or, stride, 0, g_reg, g_obj, g_cls)
        return g_reg, g_obj, g_cls, None, None


class YoloxHead(_B200Block):
    def __init__(self, num_classes, width=1.0, strides=[8, 16, 32], in_channels=[256, 512, 1024], act="silu",
                 depthwise=False):
        super().__init__()
        self.num_classes = num_classes
        self.decode_in_inference = True  # for deploy, set to False
        self.cls_convs = nn.ModuleList()
        self.reg_convs = nn.ModuleList()
        self.cls_preds = nn.ModuleList()
        self.reg_preds = nn.ModuleList()
        self.obj_preds = nn.ModuleList()
        self.stems = nn.ModuleList()
        Conv = DWConv if depthwise else BaseConv
        hid = int(256 * width)
        for cin in in_channels:
            self.stems.append(BaseConv(int(cin * width), hid, ksize=1, stride=1, act=act))
            self.cls_convs.append(nn.Sequential(Conv(hid, hid, 3, 1, act=act), Conv(hid, hid, 3, 1, act=act)))
            self.reg_convs.append(nn.Sequential(Conv(hid, hid, 3, 1, act=act), Conv(hid, hid, 3, 1, act=act)))
            self.cls_preds.append(nn.Conv2d(hid, self.num_classes, 1, 1, 0))
            self.reg_preds.append(nn.Conv2d(hid, 4, 1, 1, 0))
            self.obj_preds.append(nn.Conv2d(hid, 1, 1, 1, 0))
        self.use_l1 = False
        self.l1_loss = nn.L1Loss(reduction="none")
        self.bcewithlog_loss = nn.BCEWithLogitsLoss(reduction="none")
        self.iou_loss = IouLoss(reduction="none")
        self.strides = strides
        self.grids = [torch.zeros(1)] * len(in_channels)
        self.hw = None
        # "auto" follows torchvision.ops.batched_nms on CUDA; see boxes.postprocess
        self.output_dtype = None

    def initialize_biases(self, prior_prob):
        # yolo_head.py:129-138
        v = -math.log((1 - prior_prob) / prior_prob)
        for conv in list(self.cls_preds) + list(self.obj_preds):
            conv.bias = nn.Parameter(torch.full_like(conv.bias.data, v), requires_grad=True)

    # ------------------------------------------------------------------ eval lowering
    def decode_flags(self) -> int:
        return 3 if self.decode_in_inference else 2

    def lower(self, b, feats, head_out, decode=None, post=None):
        """feats: 3 Feats (strides 8/16/32); head_out: fp32 tensor [B, A, 5+nc]. `post` (cand_ptr, keys_ptr, counts_ptr,
        conf_thre, xyxy): run the score filter of postprocess (boxes.py:38-50) inside the decode epilogue."""
        decode = self.decode_flags() if decode is None else decode
        hw = []
        off = 0
        total = sum(f.H * f.W for f in feats)
        assert head_out.shape[1] == total and head_out.shape[2] == 5 + self.num_classes
        for k, x in enumerate(feats):
            # the levels are independent chains (yolo_head.py:140-160): all but the last one (whose input is the final
            # neck op anyway) run as side lanes of the graph, forked right after the op that produced their input, so
            # the 80x80 chain overlaps the bottom-up half of the neck and the small 40x40 / 20x20 kernels
            side = k < len(feats) - 1
            if side:
                b.begin_lane(k + 1, x)
            stem = self.stems[k].lower(b, x)
            hid = stem.c_real
            c0, c1 = self.cls_convs[k][0], self.cls_convs[k][1]
            r0, r1 = self.reg_convs[k][0], self.reg_convs[k][1]
            if isinstance(c0, BaseConv):
                # first tower convs share their input -> one 3x3 GEMM with N = 2*hid
                t0 = b.conv(stem, [b.part(c0), b.part(r0)], act=act_name(c0.act), ksize=3, stride=1)
                t1 = b.new_feat(stem.B, stem.H, stem.W, [hid, hid])
                c1.lower(b, t0.seg(0), out=t1.seg(0))
                r1.lower(b, t0.seg(1), out=t1.seg(1))
            else:
                t1 = b.new_feat(stem.B, stem.H, stem.W, [hid, hid])
                c1.lower(b, c0.lower(b, stem), out=t1.seg(0))
                r1.lower(b, r0.lower(b, stem), out=t1.seg(1))
            # [reg(4) | obj(1) | cls(nc)] rows; reg/obj read the reg tower (segment 1), cls segment 0
            parts = [
                b.part(self.reg_preds[k], o_off=0, in_segs=[1]),
                b.part(self.obj_preds[k], o_off=4, in_segs=[1]),
                b.part(self.cls_preds[k], o_off=5, in_segs=[0]),
            ]
            b.conv(t1, parts, act=None, ksize=1, stride=1, o_total=5 + self.num_classes,
                   head=dict(out=head_out, anchors=total, anchor_off=off, nc=self.num_classes, decode=decode,
                             stride=self.strides[k], **(post or {})))
            if side:
                b.end_lane()
            hw.append((x.H, x.W))
            off += x.H * x.W
        b.join_lanes()
        self.hw = [torch.Size(v) for v in hw]
        return head_out

    def _torch_raw_outputs(self, xin, rows=None):
        """Prediction-conv outputs per level through torch ops (used by the training branch and by
        synthetic.randomize_and_calibrate; never by the eval hot path). rows(k, reg, obj, cls): optional per-level
        continuation that runs inside the level's branch; its result replaces the (reg, obj, cls) tuple."""
        from .train_conv import conv2d

        from .streams import Branch

        # the levels are independent chains and so are the two towers of a level (yolo_head.py:140-160): level k on side
        # stream 1 + k, its reg tower on side stream 4 + k; every kernel here is a fraction of a wave at training batch sizes
        outs, levels = [None] * len(xin), []
        for k, x in enumerate(xin):
            lvl = Branch(x, 1 + k)
            with lvl:
                x = self.stems[k]._train_forward(x)
                tower = Branch(x, 4 + k)
                with tower:
                    reg_feat = x
                    for blk in self.reg_convs[k]:
                        reg_feat = blk._train_forward(reg_feat)
                    reg_out, obj_out = conv2d(reg_feat, self.reg_preds[k]), conv2d(reg_feat, self.obj_preds[k])
                cls_feat = x
                for blk in self.cls_convs[k]:
                    cls_feat = blk._train_forward(cls_feat)
                cls_out = conv2d(cls_feat, self.cls_preds[k])
                tower.join()
                outs[k] = (reg_out, obj_out, cls_out) if rows is None else rows(k, reg_out, obj_out, cls_out)
            levels.append(lvl)
        for lvl in levels:
            lvl.join()
        return outs

    # ------------------------------------------------------------------ forward
    def forward(self, xin, labels=None, imgs=None):
        if not self.training:
            from .engine import run_head

            return run_head(self, xin)
        outputs, origin_preds, x_shifts, y_shifts, expanded_strides = [], [], [], [], []

        def rows(k, reg_output, obj_output, cls_output):
            # cat + view + permute + decode (get_output_and_grid) and the origin_preds gather in one transposing kernel
            # (csrc/yx_train.cu), fp32 rows out, still inside the level's branch
            return _TrainRows.apply(reg_output, obj_output, cls_output, self.strides[k], self.use_l1) + (reg_output.shape,)

        for k, (output, origin, shape) in enumerate(self._torch_raw_outputs(xin, rows)):
            # only the (cached) grid is still built with torch
            grid = self._level_grid(k, shape[-2], shape[-1], xin[0].type())
            x_shifts.append(grid[:, :, 0])
            y_shifts.append(grid[:, :, 1])
            expanded_strides.append(self._level_strides(k, grid.shape[1], xin[0]))
            if self.use_l1:
                origin_preds.append(origin)
            outputs.append(output)
        return self.get_losses(imgs, x_shifts, y_shifts, expanded_strides, labels, torch.cat(outputs, 1),
                               origin_preds, dtype=xin[0].dtype)

    def _level_strides(self, k, n, like):
        """[1, n] tensor filled with the level's stride (yolo_head.py:175-179), built once per level / size / dtype: the
        reference builds it on the host every step (an H2D copy per level, which also breaks CUDA-graph capture)."""
        cache = self.__dict__.setdefault("_stride_cache", {})
        key = (k, n, like.dtype, like.device)
        t = cache.get(key)
        if t is None:
            t = cache[key] = torch.full((1, n), float(self.strides[k]), dtype=like.dtype, device=like.device)
        return t

    def _level_grid(self, k, hsize, wsize, dtype):
        grid = self.grids[k]
        if grid.shape[2:4] != (hsize, wsize) or grid.type() != dtype:
            yv, xv = torch.meshgrid([torch.arange(hsize), torch.arange(wsize)], indexing="ij")
            grid = torch.stack((xv, yv), 2).view(1, 1, hsize, wsize, 2).type(dtype)
            self.grids[k] = grid
        return grid.view(1, -1, 2)

    def get_output_and_grid(self, output, k, stride, dtype):
        # yolo_head.py:213-231
        grid = self.grids[k]
        batch_size = output.shape[0]
        n_ch = 5 + self.num_classes
        hsize, wsize = output.shape[-2:]
        if grid.shape[2:4] != output.shape[2:4]:
            yv, xv = torch.meshgrid([torch.arange(hsize), torch.arange(wsize)], indexing="ij")
            grid = torch.stack((xv, yv), 2).view(1, 1, hsize, wsize, 2).type(dtype)
            self.grids[k] = grid
        output = output.view(batch_size, 1, n_ch, hsize, wsize).permute(0, 1, 3, 4, 2).reshape(batch_size, hsize * wsize, -1)
        grid = grid.view(1, -1, 2)
        xy = (output[..., :2] + grid) * stride
        wh = torch.exp(output[..., 2:4]) * stride
        return torch.cat([xy, wh, output[..., 4:]], dim=-1), grid

    def decode_outputs(self, outputs, dtype=None):
        """yolo_head.py:233-251 as one in-place kernel (grids are never materialised)."""
        ops.require_cuda(outputs, "decode_outputs")
        out = outputs.float().contiguous()
        if out.data_ptr() == outputs.data_ptr():
            out = out.clone()
        ops.head_decode_(out, [tuple(hw) for hw in self.hw], self.strides)
        return out if outputs.dtype == torch.float32 else out.to(outputs.dtype)

    # ------------------------------------------------------------------ training: losses
    def get_losses(self, imgs, x_shifts, y_shifts, expanded_strides, labels, outputs, origin_preds, dtype):
        """yolo_head.py:253-418 without the per-image Python loop: one SimOTA launch for the whole batch
        (yx_simota_assign), then one launch that evaluates the IoU / objectness / class / L1 terms AND their gradients
        w.r.t. the prediction tensor (yx_head_losses) -- no boolean-mask gathers, no one-hot tensor, no host sync.
        Returns the reference's 6-tuple; only the total loss carries a gradient (the components are reported values)."""
        x_shifts = torch.cat(x_shifts, 1)
        y_shifts = torch.cat(y_shifts, 1)
        expanded_strides = torch.cat(expanded_strides, 1)
        origin = torch.cat(origin_preds, 1) if self.use_l1 else None
        ops.require_cuda(outputs, "get_losses")
        pred = outputs.float().contiguous()
        with torch.no_grad():
            asg = ops.simota_assign(pred.detach(), labels, x_shifts, y_shifts, expanded_strides, self.num_classes,
                                    levels=len(set(self.strides)))
        num_fg = asg["num_fg"].sum().clamp(min=1).to(torch.float32)
        num_gts = asg["num_gt"].sum().clamp(min=1).to(torch.float32)
        reg_weight = 5.0
        total, sums = _FusedHeadLoss.apply(pred, None if origin is None else origin.float().contiguous(), labels, asg,
                                           x_shifts, y_shifts, expanded_strides, self.iou_loss.loss_type == "giou", reg_weight)
        loss = (total / num_fg).to(outputs.dtype)
        parts = (sums / num_fg).to(outputs.dtype)
        loss_l1 = parts[3] if self.use_l1 else 0.0
        return (loss, reg_weight * parts[0], parts[1], parts[2], loss_l1, num_fg / num_gts)

    def get_l1_target(self, l1_target, gt, stride, x_shifts, y_shifts, eps=1e-8):
        l1_target[:, 0] = gt[:, 0] / stride - x_shifts
        l1_target[:, 1] = gt[:, 1] / stride - y_shifts
        l1_target[:, 2] = torch.log(gt[:, 2] / stride + eps)
        l1_target[:, 3] = torch.log(gt[:, 3] / stride + eps)
        return l1_target

    # ------------------------------------------------------------------ reference-shaped SimOTA API
    @torch.no_grad()
    def get_assignments(self, batch_idx, num_gt, gt_bboxes_per_image, gt_classes, bboxes_preds_per_image,
                        expanded_strides, x_shifts, y_shifts, cls_preds, obj_preds, mode="gpu"):
        """Same arguments and return tuple as yolo_head.py:420-509, computed by one kernel launch.
        ``mode="cpu"`` (the reference's OOM escape hatch) is rejected: the kernel never
        materialises the [G, A', nc] tensor that made it necessary."""
        if mode != "gpu":
            raise RuntimeError("get_assignments(mode='cpu') is not available: the B200 path has no CPU fallback")
        A = bboxes_preds_per_image.shape[0]
        pred = torch.cat([bboxes_preds_per_image.float(), obj_preds[batch_idx].float().reshape(A, 1),
                          cls_preds[batch_idx].float()], dim=1).unsqueeze(0)
        labels = torch.cat([gt_classes.float().reshape(-1, 1), gt_bboxes_per_image.float()], dim=1)[:num_gt]
        pad = max(num_gt, 1)
        lab = torch.zeros((1, pad, 5), dtype=torch.float32, device=pred.device)
        lab[0, :num_gt] = labels
        asg = ops.simota_assign(pred, lab, x_shifts, y_shifts, expanded_strides, self.num_classes)
        status = int(asg["status"][0].item())          # this reference-shaped entry point synchronises anyway (num_fg below)
        if status == 2:
            raise RuntimeError("get_assignments: class values must be smaller than num_classes and non-negative")
        if status == 1:
            raise RuntimeError("get_assignments: more in-centre anchors than 9 per stride level and GT "
                               "(the anchor grid is not one unit-spaced grid per level)")
        fg_mask = asg["fg_mask"][0].bool()
        matched_gt_inds = asg["matched_gt"][0][fg_mask].long()
        gt_matched_classes = gt_classes[matched_gt_inds]
        pred_ious = asg["matched_iou"][0][fg_mask]
        return gt_matched_classes, fg_mask, pred_ious, matched_gt_inds, int(asg["num_fg"][0].item())

    def simota_matching(self, cost, pair_wise_ious, gt_classes, num_gt, fg_mask):
        """yolo_head.py:542-574 (mutates fg_mask in place like the reference)."""
        mg, mi, nf = ops.simota_matching_device(cost[:num_gt], pair_wise_ious[:num_gt])
        fg_inboxes = mg >= 0
        num_fg = int(nf.item())
        fg_mask[fg_mask.clone()] = fg_inboxes
        matched_gt_inds = mg[fg_inboxes].long()
        gt_matched_classes = gt_classes[matched_gt_inds]
        return num_fg, gt_matched_classes, mi[fg_inboxes], matched_gt_inds
