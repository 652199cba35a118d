"""The 30 depthwise convs of a yolox_nano training step at 416x416: our forward / dgrad / wgrad (csrc/yx_dwconv_train.cu) against
what torch runs for them under 16-bit autocast (weight cast + cuDNN conv, its input and weight gradients, the cast of dW back to
fp32), per layer: many calls captured in one CUDA graph, CUDA events around its replays after a warm-up. Inputs are L2-warm,
as they are in the training step, where the producing layer has just written them.

usage: python tools/gpu_prof_dwconv_train.py [--batch 8 64] [--iters 50] [--dtype bf16] [--json PATH]
       python tools/gpu_prof_dwconv_train.py --launches [--torch-depthwise]
         kernel launches of one eager bf16 yolox_nano training step (8 images, channels_last, direct gradients), counted with
         torch.profiler; --torch-depthwise routes the depthwise convs to torch as before these kernels existed
"""
import argparse
import copy
import json
import subprocess
import sys
from collections import Counter
from pathlib import Path

import torch
import torch.nn.functional as F

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
from pixeltable_yolox_b200 import ops  # noqa: E402

HBM_BYTES_PER_S = 7.7e12          # HGX B200 data sheet, one GPU

# (c, H, W, stride) of the depthwise convs of yolox_nano at 416x416, in forward order
NANO_416 = ([(16, 208, 208, 2), (16, 104, 104, 1), (32, 104, 104, 2)] + [(32, 52, 52, 1)] * 3 + [(64, 52, 52, 2)]
            + [(64, 26, 26, 1)] * 3 + [(128, 26, 26, 2), (128, 13, 13, 1), (64, 26, 26, 1), (32, 52, 52, 1), (64, 52, 52, 2),
                                       (64, 26, 26, 1), (128, 26, 26, 2), (128, 13, 13, 1)]
            + [(64, 52, 52, 1)] * 4 + [(64, 26, 26, 1)] * 4 + [(64, 13, 13, 1)] * 4)


def card():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:  # noqa: BLE001
        q = f"unknown ({e!r})"
    return name, q


def time_us(fn, iters, replays=5):
    """GPU time per call: `iters` calls captured in one CUDA graph (so the host's launch rate does not set the time), replayed
    after a warm-up, CUDA events around `replays` replays."""
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(3):
            fn()
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for _ in range(iters):
            fn()
    g.replay()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(replays):
        g.replay()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / (iters * replays) * 1e3


def layer_rows(batch, dtype, iters):
    dev = torch.device("cuda", 0)
    rows, cache = [], {}
    for li, (c, H, W, s) in enumerate(NANO_416):
        key = (c, H, W, s)
        if key not in cache:
            OH, OW = (H - 1) // s + 1, (W - 1) // s + 1
            x = torch.randn(batch, c, H, W, device=dev).to(dtype).contiguous(memory_format=torch.channels_last)
            dy = torch.randn(batch, c, OH, OW, device=dev).to(dtype).contiguous(memory_format=torch.channels_last)
            w = torch.randn(c, 1, 3, 3, device=dev) * 0.3
            dw_ws = ops.dwconv_wgrad(x, dy, w, s)           # sizes the workspace outside the timed loop
            mask_d, mask_w = [True, False, False], [False, True, False]

            def t_fwd():
                F.conv2d(x, w.to(dtype), None, s, 1, 1, c)

            def t_dgrad():
                torch.ops.aten.convolution_backward(dy, x, w.to(dtype), None, [s, s], [1, 1], [1, 1], False, [0, 0], c, mask_d)

            def t_wgrad():
                torch.ops.aten.convolution_backward(dy, x, w.to(dtype), None, [s, s], [1, 1], [1, 1], False, [0, 0], c,
                                                    mask_w)[1].float()

            ours = dict(fwd=time_us(lambda: ops.dwconv_train_fwd(x, w, s), iters),
                        dgrad=time_us(lambda: ops.dwconv_dgrad(dy, w, s, H, W), iters),
                        wgrad=time_us(lambda: ops.dwconv_wgrad(x, dy, w, s, accumulate_into=dw_ws), iters))
            theirs = dict(fwd=time_us(t_fwd, iters), dgrad=time_us(t_dgrad, iters), wgrad=time_us(t_wgrad, iters))
            e = x.element_size()
            nx, ny = x.numel() * e, dy.numel() * e
            nbytes = dict(fwd=nx + ny, dgrad=ny + nx, wgrad=nx + ny + 9 * c * 4)
            cache[key] = (ours, theirs, nbytes)
        ours, theirs, nbytes = cache[key]
        rows.append(dict(layer=li, c=c, hw=f"{H}x{W}", stride=s, batch=batch, ours_us=ours, torch_us=theirs, bytes=nbytes))
    return rows


def print_table(rows):
    print("| layer | c | in | s | B | fwd us ours / torch | dgrad us ours / torch | wgrad us ours / torch | ours GB/s fwd / dgrad / wgrad (share of 7.7 TB/s) |")
    print("|---:|---:|---|---:|---:|---|---|---|---|")
    tot_o, tot_t = Counter(), Counter()
    for r in rows:
        o, t, b = r["ours_us"], r["torch_us"], r["bytes"]
        gbs = {k: b[k] / (o[k] * 1e-6) / 1e9 for k in o}
        share = " / ".join(f"{gbs[k]:.0f} ({gbs[k] * 1e9 / HBM_BYTES_PER_S:.0%})" for k in ("fwd", "dgrad", "wgrad"))
        print(f"| {r['layer']} | {r['c']} | {r['hw']} | {r['stride']} | {r['batch']} | {o['fwd']:.1f} / {t['fwd']:.1f} | "
              f"{o['dgrad']:.1f} / {t['dgrad']:.1f} | {o['wgrad']:.1f} / {t['wgrad']:.1f} | {share} |")
        tot_o.update(o)
        tot_t.update(t)
    print(f"| sum | | | | | {tot_o['fwd']:.0f} / {tot_t['fwd']:.0f} | {tot_o['dgrad']:.0f} / {tot_t['dgrad']:.0f} | "
          f"{tot_o['wgrad']:.0f} / {tot_t['wgrad']:.0f} | |")


def count_launches(torch_depthwise):
    import pixeltable_yolox_b200 as yx
    from pixeltable_yolox_b200 import synthetic as syn
    from pixeltable_yolox_b200 import train_conv
    from pixeltable_yolox_b200.optim import FusedSgdEma

    if torch_depthwise:
        train_conv.usable_depthwise = lambda x, conv: None
    dev = torch.device("cuda", 0)
    torch.manual_seed(0)
    m = copy.deepcopy(yx.YoloxConfig.get_named_config("yolox_nano").get_model()).float().to(dev).train()
    m = m.to(memory_format=torch.channels_last)
    train_conv.attach_packer(m, torch.bfloat16)
    x = torch.from_numpy(syn.images(8, 416, 416, seed=3)).to(dev).contiguous(memory_format=torch.channels_last)
    lab = torch.from_numpy(syn.labels(8, max_gt=16, seed=5, size=416.0)).to(dev)
    opt = FusedSgdEma(m, lr=1e-3, ema=True, direct_grads=True)

    def step():
        with torch.autocast("cuda", dtype=torch.bfloat16):
            out = m(x, lab)
        opt.zero_grad()
        out["total_loss"].backward()
        opt.step()

    for _ in range(3):
        step()
    torch.cuda.synchronize()
    from torch.profiler import ProfilerActivity, profile

    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        step()
        torch.cuda.synchronize()
    kernels = [e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA and "memcpy" not in e.name.lower()
               and "memset" not in e.name.lower()]
    by = Counter(e.name for e in kernels)
    ours = sum(n for k, n in by.items() if "dw_gather_kernel" in k or "dw_wgrad" in k)
    torch_conv = sum(n for k, n in by.items() if any(s in k.lower() for s in ("depthwise", "cudnn", "conv2d")))
    print(json.dumps(dict(torch_depthwise=torch_depthwise, kernels_per_step=len(kernels), ours_depthwise_kernels=ours,
                          torch_conv_kernels=torch_conv, top=by.most_common(15))))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, nargs="+", default=[8, 64])
    ap.add_argument("--iters", type=int, default=50)
    ap.add_argument("--dtype", default="bf16", choices=["bf16", "fp16"])
    ap.add_argument("--json", default=None)
    ap.add_argument("--launches", action="store_true")
    ap.add_argument("--torch-depthwise", action="store_true")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: these are GPU timings")
    name, limit = card()
    print(f"# {name}, power limit / max SM clock: {limit}")
    if args.launches:
        count_launches(args.torch_depthwise)
        return
    dtype = torch.bfloat16 if args.dtype == "bf16" else torch.float16
    out = []
    for b in args.batch:
        rows = layer_rows(b, dtype, args.iters)
        print(f"\n## batch {b}, {args.dtype}, us per call (CUDA events around replays of a graph of {args.iters} calls, L2-warm)\n")
        print_table(rows)
        out += rows
    if args.json:
        Path(args.json).parent.mkdir(parents=True, exist_ok=True)
        Path(args.json).write_text(json.dumps(dict(card=name, power_limit=limit, rows=out), indent=1))


if __name__ == "__main__":
    main()
