"""Per-layer times of the training BatchNorm + activation kernels (yolox_s, 8 images, bf16), channels_last vs NCHW, forward and
backward, with the bytes each pass must move. usage: python tools/gpu_prof_trainbn.py"""
import sys
from collections import OrderedDict
from pathlib import Path

import torch

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
import pixeltable_yolox_b200 as yx  # noqa: E402
from pixeltable_yolox_b200 import ops  # noqa: E402
from pixeltable_yolox_b200._lib import YX_ACT_SILU  # noqa: E402

B = 8
dev = torch.device("cuda", 0)
model = yx.YoloxConfig.get_named_config("yolox_s").get_model()
shapes = OrderedDict()
H = {}


def walk():
    # BN shapes = outputs of the convs inside BaseConv: run the train forward with the convs on torch, whose hooks fire
    from pixeltable_yolox_b200.network_blocks import BaseConv

    def hook(m, inp, out):
        key = tuple(out.shape[1:])
        shapes[key] = shapes.get(key, 0) + 1
    hs = [m.conv.register_forward_hook(hook) for m in model.modules() if isinstance(m, BaseConv)]
    import os
    os.environ["YX_TRAIN_CONV"] = "0"
    model.to(dev).train()
    with torch.no_grad():
        lab = torch.zeros(1, 120, 5, device=dev); lab[:, 0] = torch.tensor([1.0, 320, 320, 100, 100], device=dev)
        model(torch.rand(1, 3, 640, 640, device=dev) * 255, lab)
    for h in hs:
        h.remove()


walk()


def timeit(fn, reps=10):
    for _ in range(2):
        fn()
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for _ in range(reps):
            fn()
    g.replay(); torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(); g.replay(); e1.record(); torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps * 1e3


tot = [0.0] * 4
print("    C    HxW   n |  MB  | nhwc fwd   bwd | nchw fwd   bwd   (us)  | nhwc GB/s fwd  bwd")
for (c, h, w), cnt in shapes.items():
    res = []
    for fmt in (torch.channels_last, torch.contiguous_format):
        x = torch.randn(B, c, h, w, device=dev).bfloat16().contiguous(memory_format=fmt)
        dy = torch.randn(B, c, h, w, device=dev).bfloat16().contiguous(memory_format=fmt)
        g, b = torch.ones(c, device=dev), torch.zeros(c, device=dev)
        rm, rv = torch.zeros(c, device=dev), torch.ones(c, device=dev)
        y, mean, invstd = ops.bn_act_train_fwd(x, g, b, rm, rv, 1e-3, 0.03, YX_ACT_SILU)
        res.append(timeit(lambda: ops.bn_act_train_fwd(x, g, b, rm, rv, 1e-3, 0.03, YX_ACT_SILU)))
        res.append(timeit(lambda: ops.bn_act_train_bwd(x, dy, g, b, mean, invstd, YX_ACT_SILU)))
    mb = B * c * h * w * 2 / 1e6
    for i in range(4):
        tot[i] += res[i] * cnt
    print(f"{c:5d} {h:3d}x{w:<3d} {cnt:3d} | {mb:5.1f} | {res[0]:7.1f} {res[1]:6.1f} | {res[2]:7.1f} {res[3]:6.1f} | {3 * mb / res[0] * 1e3:8.0f} {5 * mb / res[1] * 1e3:6.0f}")
print(f"sum over the network (us): nhwc fwd {tot[0]:.0f} bwd {tot[1]:.0f} | nchw fwd {tot[2]:.0f} bwd {tot[3]:.0f}")
