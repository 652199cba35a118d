"""sort_nms_kernel: one CTA per image (YX_NMS_CLUSTER=1) against the thread-block-cluster kernel (host's choice of 2 / 4 / 8
CTAs per image) on the dense scenes of config 5, with equality of the kept rows checked on every case.
usage: python tools/gpu_nms_cluster.py [out.json]"""
import json
import os
import sys
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
from pixeltable_yolox_b200 import ops, synthetic as syn  # noqa: E402
from pixeltable_yolox_b200.boxes import NMS_VARIANTS  # noqa: E402

dev = torch.device("cuda", 0)
A = 8400


def timed(pred, thr, reps=20):
    """median device time (us) of filter + sort_nms, and of the filter alone (nms threshold path identical)"""
    work = [pred.clone() for _ in range(reps + 3)]
    for w in work[:3]:
        out = ops.postprocess_device(w, 80, thr, 0.65, NMS_VARIANTS["auto"])
    torch.cuda.synchronize()
    ts = []
    for w in work[3:]:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        out = ops.postprocess_device(w, 80, thr, 0.65, NMS_VARIANTS["auto"])
        e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1) * 1e3)
    return float(np.median(ts)), out


def all_kept(batch, classes):
    grid = np.zeros((batch, A, 85), dtype=np.float32)
    gx, gy = np.meshgrid(np.arange(100), np.arange(84))
    grid[:, :, 0] = (gx.reshape(-1) * 6.0 + 3.0)[None]; grid[:, :, 1] = (gy.reshape(-1) * 6.0 + 3.0)[None]
    grid[:, :, 2:4] = 9.0                                                  # neighbours overlap a little (IoU 0.2): divisions run
    rng = np.random.default_rng(10)
    grid[:, :, 4] = rng.uniform(0.5, 1.0, (batch, A))
    np.put_along_axis(grid[:, :, 5:], rng.integers(0, classes, (batch, A))[..., None], 0.9, axis=2)
    return grid


rows = []
for batch in (64, 16, 4, 1):
    dense = torch.from_numpy(syn.dense_scene(batch, anchors=A, seed=13)).to(dev)
    kept3 = torch.from_numpy(all_kept(batch, 3)).to(dev)
    for name, pred, thr in (("dense", dense, 0.001), ("dense", dense, 0.25), ("dense", dense, 0.5), ("all_kept_3_classes", kept3, 0.01)):
        os.environ["YX_NMS_CLUSTER"] = "1"
        t1, o1 = timed(pred, thr)
        del os.environ["YX_NMS_CLUSTER"]
        tc, oc = timed(pred, thr)
        same = bool(torch.equal(o1[2], oc[2]))
        cnt = o1[2].cpu().tolist()
        for b in range(batch):
            same = same and bool(torch.equal(o1[0][b, :cnt[b]], oc[0][b, :cnt[b]])) and bool(torch.equal(o1[1][b, :cnt[b]], oc[1][b, :cnt[b]]))
        row = dict(scene=name, batch=batch, conf_thre=thr, kept_per_image=float(np.mean(cnt)), postprocess_us_one_cta=round(t1, 1),
                   postprocess_us_cluster=round(tc, 1), speedup=round(t1 / tc, 2), rows_equal=same)
        print(json.dumps(row), flush=True)
        rows.append(row)
if len(sys.argv) > 1:
    Path(sys.argv[1]).write_text(json.dumps(rows, indent=1))
assert all(r["rows_equal"] for r in rows), "cluster kernel keeps different rows"
