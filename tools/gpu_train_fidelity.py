"""Gradient / loss fidelity of the 16-bit training forward + backward against the fp32 run, over several seeds: our kernels
(fast and precise SiLU in the BatchNorm passes) and torch's 16-bit path. usage: python tools/gpu_train_fidelity.py [seeds]"""
import os
import sys
from pathlib import Path

import torch

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
import pixeltable_yolox_b200 as yx  # noqa: E402
from pixeltable_yolox_b200 import synthetic as syn  # noqa: E402

seeds = int(sys.argv[1]) if len(sys.argv) > 1 else 6
named = sys.argv[2] if len(sys.argv) > 2 else None
dev = torch.device("cuda", 0)


def cos(a, b):
    return float(torch.dot(a, b) / (a.norm() * b.norm()))


rows = []
for seed in range(seeds):
    torch.manual_seed(seed)
    m = (yx.YoloxConfig.get_named_config(named) if named else yx.YoloxConfig("fid", depth=0.33, width=0.25)).get_model().to(dev).train()
    x = torch.from_numpy(syn.images(2, 128, 128, seed=seed + 3)).to(dev)
    sd = {k: v.clone() for k, v in m.state_dict().items()}
    res = {}
    for name, flag, amp in (("fp32", "0", False), ("ours", "1", True), ("torch16", "0", True)):
        os.environ["YX_TRAIN_CONV"] = flag
        m.load_state_dict(sd)
        m.zero_grad(set_to_none=True)
        with torch.autocast("cuda", dtype=torch.bfloat16, enabled=amp):
            outs = m.head._torch_raw_outputs(m.backbone(x))
        loss = sum(t.float().square().mean() for lvl in outs for t in lvl)
        loss.backward()
        res[name] = (float(loss.detach()), torch.cat([p.grad.flatten() for p in m.parameters() if p.grad is not None]).clone(),
                     torch.cat([t.detach().float().flatten() for lvl in outs for t in lvl]))
    l32, g32, o32 = res["fp32"]
    print(f"   max |pred - fp32|: ours {float((res['ours'][2] - o32).abs().max()):.4f} torch16 {float((res['torch16'][2] - o32).abs().max()):.4f}; "
          f"rms: ours {float((res['ours'][2] - o32).square().mean().sqrt()):.5f} torch16 {float((res['torch16'][2] - o32).square().mean().sqrt()):.5f}")
    rows.append((cos(res["ours"][1], g32), cos(res["torch16"][1], g32), abs(res["ours"][0] - l32) / l32, abs(res["torch16"][0] - l32) / l32))
    print(f"seed {seed}: gradient cosine vs fp32 ours {rows[-1][0]:.4f} torch16 {rows[-1][1]:.4f} | loss rel err ours {rows[-1][2]:.2e} torch16 {rows[-1][3]:.2e}", flush=True)
n = len(rows)
print(f"mean over {n} seeds: cosine ours {sum(r[0] for r in rows) / n:.4f} torch16 {sum(r[1] for r in rows) / n:.4f} | "
      f"loss rel err ours {sum(r[2] for r in rows) / n:.2e} torch16 {sum(r[3] for r in rows) / n:.2e}")
