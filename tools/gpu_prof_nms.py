"""Device time of the sort + NMS kernel (yx_nms_prefiltered after one filter pass) and of the score filter on
B = 64 images: sparse scenes (~20 candidates, the bench's regime: single-warp path), dense scenes at three thresholds
(config 5) and the degenerate every-anchor-kept scene (conf 0.01 on random weights). CUDA-graph replay, no Python time."""
import sys
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
from pixeltable_yolox_b200 import ops, synthetic as syn  # noqa: E402
from pixeltable_yolox_b200.boxes import NMS_VARIANTS  # noqa: E402

dev = torch.device("cuda", 0)
B, A = 64, 8400


def graph_us(fn, n=20):
    fn(); torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        fn()
    for _ in range(3):
        g.replay()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        g.replay()
    e1.record(); torch.cuda.synchronize()
    return e0.elapsed_time(e1) * 1e3 / n


def case(name, pred_np, thr):
    pred = torch.from_numpy(pred_np).to(dev)
    ws = ops._workspace(dev, ops.lib().yx_postprocess_workspace_bytes(B, A), "post")
    _, _, cnt = ops.postprocess_device(pred.clone(), 80, thr, 0.65, NMS_VARIANTS["auto"])
    work = pred.clone()
    t_all = graph_us(lambda: ops.postprocess_device(work, 80, thr, 0.65, NMS_VARIANTS["auto"], inplace_xyxy=False))
    t_nms = graph_us(lambda: ops.nms_prefiltered(ws, B, A, 0.65, NMS_VARIANTS["auto"]))
    sc = pred[..., 4] * pred[..., 5:].max(-1).values
    print(f"{name:34s} thr {thr:5.3f}: candidates/img {float((sc >= thr).sum()) / B:7.1f} kept/img {float(cnt.sum()) / B:7.1f} | "
          f"filter+sort+nms {t_all:8.1f} us, sort+nms {t_nms:8.1f} us, filter {t_all - t_nms:6.1f} us")


case("sparse (12 objects)", syn.sparse_scene(B, A, seed=5), 0.5)
dense = syn.dense_scene(B, anchors=A, seed=13)
for thr in (0.001, 0.25, 0.5):
    case("dense clusters", dense, thr)
grid = np.zeros((B, A, 85), dtype=np.float32)
gx, gy = np.meshgrid(np.arange(100), np.arange(84))
grid[:, :, 0] = (gx.reshape(-1) * 6.0 + 3.0)[None]; grid[:, :, 1] = (gy.reshape(-1) * 6.0 + 3.0)[None]
grid[:, :, 2:4] = 5.0
rng = np.random.default_rng(10)
grid[:, :, 4] = rng.uniform(0.5, 1.0, (B, A))
np.put_along_axis(grid[:, :, 5:], rng.integers(0, 80, (B, A))[..., None], 0.9, axis=2)
case("every anchor kept (disjoint)", grid, 0.01)
