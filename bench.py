"""bench.py — YOLOX-s 640^2 images/s (fwd + decode + NMS) on N B200s (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
        --master-port P bench.py --gpus N --steps K --warmup W

A "step" is one pass of the hot path (YoloxModule.forward eval + postprocess, i.e. focus -> convs ->
head decode -> score filter -> NMS, one CUDA graph) over one batch of 64 synthetic 640x640 images
per GPU (weak scaling: the batch is sharded by image, no data-path collective).
  value     : whole-job images/s with the inputs already resident in HBM (CUDA events, max over ranks)
  e2e       : the same metric through the public API with HOST (pinned) uint8 images: H2D of the batch
              and D2H of the detections inside the timed region, double-buffered over two streams
              (e2e_fp32_input: the same with the fp32 host tensor the reference's processor produces)
  roofline  : the dominant kernel (tcgen05 implicit-GEMM conv): algorithmic conv FLOPs / its device
              time, measured live with CUDA events around every launch of an eager pass
  cpu_baseline : the CPU restatement of the reference path (oracle/, torch CPU ops + numpy/C NMS) on the host cores,
              on a bounded sample of the same workload (rank 0, N = 1 only)
  --impl reference : the UNMODIFIED reference (baseline/_ref, installed by baseline/install_ref.py) on the host cores:
              YoloxModule.forward + yolox.utils.postprocess, fp32, all threads (falls back to the oracle port if
              baseline/_ref is missing)
  extra     : conf 0.01 leg (the evaluator's threshold), dense NMS stress (config 5), per-family HBM rooflines, the
              same-box torch GPU reference (unmodified reference module in bf16 on cuDNN + torchvision NMS)
  --train   : config 4, one training step (fwd-train + SimOTA + losses + backward + gradient all-reduce + SGD)
  --global-batch G : strong scaling, G images per step split over the ranks (config 3: --model yolox_l --dtype fp16
              --global-batch 512)
  --dump-outputs DIR : after the timed steps, what the last one returned to its caller as DIR/<name>.npy (see
              dump_outputs), so that two builds can be compared output for output on the same seeded inputs
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))
sys.dont_write_bytecode = True          # the benchmark writes nothing into the tree it runs from (it may be read-only)

GFLOP_PER_IMAGE = {"yolox_s": 26.686, "yolox_m": 73.530, "yolox_l": 155.293, "yolox_x": 281.410,
                   "yolox_tiny": 6.413, "yolox_nano": 1.045}   # BASELINE.md section 2 (conv 2*MAC)


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--model", default="yolox_s")
    ap.add_argument("--batch", type=int, default=64, help="images per GPU per step")
    ap.add_argument("--size", type=int, default=640)
    ap.add_argument("--dtype", default="bf16", choices=["bf16", "fp16", "fp32"])
    ap.add_argument("--micro-batch", type=int, default=64)
    ap.add_argument("--conf", type=float, default=0.5)
    ap.add_argument("--nms", type=float, default=0.65)
    ap.add_argument("--max-det", type=int, default=1000)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-images", type=int, default=16)
    ap.add_argument("--profile-ops", action="store_true", help="print the per-op table of the eager pass")
    ap.add_argument("--global-batch", type=int, default=0, help="strong scaling: images per step over ALL ranks")
    ap.add_argument("--train", action="store_true", help="config 4: training step (8 images per rank by default)")
    ap.add_argument("--train-batch", type=int, default=8, help="--train: images per rank")
    ap.add_argument("--train-format", default="channels_last", choices=["channels_last", "contiguous"],
                    help="--train: memory format of the module and its input in our arm (cuDNN's 16-bit kernels are NHWC; "
                         "our BatchNorm + activation kernels take both)")
    ap.add_argument("--no-extras", action="store_true", help="skip the extra legs (conf 0.01, config 5, torch GPU reference)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the outputs of the last timed inference step to DIR/<name>.npy (rank 0's images)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.train or args.impl != "ours"):
        ap.error("--dump-outputs writes the outputs of the inference step of --impl ours")
    return args


def peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        d = json.loads(p.read_text())
        return dict(hbm=d["hbm_gbs"], tf_burst=d["bf16_tflops"], tf_sustained=d["bf16_tflops_sustained"], source="measured")
    return dict(hbm=6650.0, tf_burst=1590.0, tf_sustained=1400.0, source="fallback")


class ClockSampler:
    """nvidia-smi clocks + throttle reasons during the timed region (B200_PROFILING.md)."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index = index
        self.rows = []
        self.stamps = []          # host arrival time of each row
        self.window = None        # (t0, t1) of the timed region; rows outside it are dropped when enough fall inside
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "25"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            parts = [p.strip() for p in line.split(",")]
            if len(parts) >= 7:
                self.rows.append(parts)
                self.stamps.append(time.perf_counter())

    def mark(self, t0: float, t1: float):
        self.window = (t0, t1)

    def wait_first(self, timeout: float = 1.0):
        """Block until nvidia-smi has produced its first row (it needs ~100-300 ms to start)."""
        t_end = time.perf_counter() + timeout
        while self.proc is not None and not self.rows and time.perf_counter() < t_end:
            time.sleep(0.01)

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        if self.window is not None:
            inside = [r for r, t in zip(self.rows, self.stamps) if self.window[0] <= t <= self.window[1] + 0.03]
            if inside:
                self.rows = inside
        sm = sorted(float(r[0]) for r in self.rows if r[0].replace(".", "").isdigit())
        mx = [float(r[1]) for r in self.rows if r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({n for r in self.rows for n, v in zip(names, r[3:7]) if v.lower().startswith("active")})
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx[0] if mx else None, "reasons": reasons,
                "samples": len(self.rows)}


def bind_to_gpu_numa_node(local: int):
    """Multi-rank runs: keep this rank's threads (and therefore its pinned host buffers, first touch) on the NUMA node the
    GPU hangs off, so that eight ranks' H2D streams do not cross the socket interconnect. Best effort: returns the node
    or None (single rank, sysfs not visible, or the container's cpuset has no CPU of that node)."""
    try:
        import torch

        pr = torch.cuda.get_device_properties(local)
        bus = f"{pr.pci_domain_id:04x}:{pr.pci_bus_id:02x}:{pr.pci_device_id:02x}.0"
        node = int(Path(f"/sys/bus/pci/devices/{bus}/numa_node").read_text())
        if node < 0:
            return None
        cpus = set()
        for part in Path(f"/sys/devices/system/node/node{node}/cpulist").read_text().strip().split(","):
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        avail = os.sched_getaffinity(0) & cpus
        if not avail:
            return None
        os.sched_setaffinity(0, avail)
        return node
    except Exception:
        return None


def build_model(args, device):
    import torch

    import pixeltable_yolox_b200 as yx
    from pixeltable_yolox_b200 import synthetic as syn

    cfg = yx.YoloxConfig.get_named_config(args.model)
    cfg.model = None
    torch.manual_seed(0)
    model = cfg.get_model().to(device)
    calib = syn.images(4, args.size, args.size, seed=1234)
    syn.randomize_and_calibrate(model, calib, seed=0)       # non-degenerate random-init weights (SURVEY 8c)
    return cfg, model


def cpu_reference_rate(args, sd, images_np, seconds_cap=25.0):
    """The reference path restated on CPU (oracle/): torch CPU fp32 forward + numpy/C postprocess."""
    import numpy as np
    import torch

    from oracle import postprocess_oracle as po
    from oracle import yolox_oracle as yo

    threads = os.cpu_count() or 1
    torch.set_num_threads(threads)
    x = torch.from_numpy(images_np)
    done, t_used = 0, 0.0
    chunk = 4
    yo.forward(sd, x[:1])   # warm-up (thread pool, allocator)
    while done < x.shape[0] and t_used < seconds_cap:
        t0 = time.perf_counter()
        out = yo.forward(sd, x[done:done + chunk]).numpy()
        po.postprocess(np.ascontiguousarray(out), 80, args.conf, args.nms, variant="auto_cpu")
        t_used += time.perf_counter() - t0
        done += min(chunk, x.shape[0] - done)
    return done / t_used, threads, done


def workload_name(args) -> str:
    """The same string in both arms (ours / --impl reference): the BASELINE.json configuration being measured."""
    if args.train:
        return (f"{args.model} {args.size}x{args.size} training step, {args.train_batch} images/GPU (fwd-train + SimOTA + losses + "
                "backward + gradient all-reduce + SGD), config[3] of BASELINE.json")
    if args.global_batch:
        return (f"{args.model} {args.size}x{args.size} global batch-{args.global_batch} {args.dtype} inference (fwd+decode+NMS) "
                "sharded by image over the ranks, config[2] of BASELINE.json")
    return (f"{args.model} {args.size}x{args.size} batch-{args.batch}/GPU {args.dtype} inference (fwd+decode+NMS), "
            "config[1] of BASELINE.json")


def reference_modules():
    """The unmodified reference from baseline/_ref (baseline/install_ref.py), or None. pycocotools is the one import this
    image cannot satisfy (yolox/data/datasets/coco.py:7, dataset / evaluator only): stubbed, never called on the path."""
    import types

    ref = ROOT / "baseline" / "_ref"
    if not (ref / "yolox").is_dir():
        return None
    if str(ref) not in sys.path:
        sys.path.insert(0, str(ref))
    for name, attrs in {"pycocotools": [], "pycocotools.coco": ["COCO"], "pycocotools.cocoeval": ["COCOeval"],
                        "pycocotools.mask": []}.items():
        if name not in sys.modules:
            mod = types.ModuleType(name)
            for a in attrs:
                setattr(mod, a, type(a, (), {}))
            sys.modules[name] = mod
    try:
        from yolox.config import YoloxConfig
        from yolox.utils import postprocess
    except Exception as e:                      # noqa: BLE001 - report, never crash the bench
        print(f"# reference import failed: {e!r}", file=sys.stderr)
        return None
    return dict(YoloxConfig=YoloxConfig, postprocess=postprocess)


def reference_model(ref, name: str, sd, device, dtype=None):
    """A fresh instance of the reference's own module for a named config, carrying OUR arm's weights."""
    cfg = ref["YoloxConfig"].get_named_config(name)
    cfg.model = None                             # get_model() caches the module on the singleton config (config.py:168-172)
    m = cfg.get_model()
    m.load_state_dict(sd)
    m = m.to(device)
    if dtype is not None:
        m = m.to(dtype)
    return m.eval()


def run_reference(args):
    """--impl reference: the reference's own CPU implementation of the path on the host cores."""
    import numpy as np
    import torch

    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from pixeltable_yolox_b200 import synthetic as syn

    threads = os.cpu_count() or 1
    torch.set_num_threads(threads)
    if args.train:
        return run_reference_train(args, threads)
    _, model = build_model(args, torch.device("cpu"))
    sd = {k: v.detach().clone() for k, v in model.state_dict().items()}
    ref = reference_modules()
    B = args.batch if not args.global_batch else args.global_batch
    if ref is not None:
        kind = "reference"
        how = "unmodified reference (baseline/_ref): YoloxModule.forward + yolox.utils.postprocess, CPU fp32"
        rmodel = reference_model(ref, args.model, sd, torch.device("cpu"))

        def step(x):
            with torch.no_grad():
                out = rmodel(x)
            ref["postprocess"](out, rmodel.head.num_classes, args.conf, args.nms, class_agnostic=False)
    else:
        from oracle import postprocess_oracle as po
        from oracle import yolox_oracle as yo

        kind = "port"
        how = "oracle/ torch-CPU fp32 forward + numpy/C NMS (baseline/_ref missing)"

        def step(x):
            out = yo.forward(sd, x).numpy()
            po.postprocess(np.ascontiguousarray(out), 80, args.conf, args.nms, variant="auto_cpu")

    probe = torch.from_numpy(syn.images(4, args.size, args.size, seed=7))
    step(probe)                                   # thread pool / allocator warm-up
    t0 = time.perf_counter()
    step(probe)
    rate = 4 / (time.perf_counter() - t0)
    warm = min(args.warmup, 3)
    # bounded sample: at most 16 images per step (the CPU path is at its best rate in small batches: at 64 the activations
    # fall out of the host caches) and the whole run (warm-up + steps) within ~150 s of CPU work
    per_step = int(max(2, min(B, 16, rate * 150.0 / (args.steps + warm))))
    x = torch.from_numpy(syn.images(per_step, args.size, args.size, seed=7))
    for _ in range(warm):
        step(x)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step(x)
    dt = time.perf_counter() - t0
    value = per_step * args.steps / dt
    sample = (f"{args.steps} steps x {per_step} images" + ("" if per_step == B else f" (bounded sample of the {B}-image step)") +
              f", {how}")
    line = {
        "metric": "images_per_second", "impl": "reference", "value": value, "unit": "images/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": warm, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True,
        "scaling": "strong" if args.global_batch else "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_name(args), "per_gpu_batch": args.batch, "conf_thre": args.conf, "nms_thre": args.nms,
                   "reference_arm": f"host CPU fp32, {per_step} images per step"},
        "cpu_baseline": {"value": value, "unit": "images/s", "cores": threads, "kind": kind, "sample": sample},
        "e2e": {"value": value, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


def timed_us(fn, n: int = 10, warm: int = 3) -> float:
    """Mean device time of fn() in microseconds (CUDA events on the current stream, synchronised on both sides)."""
    import torch

    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) * 1e3 / n


def parity_check(model, engine, args) -> dict:
    """Outside the timed region: the detections of the LAST timed step (fused graph: score filter in the head epilogues +
    sort/NMS kernel) must equal YoloxModule.forward + postprocess (the reference-shaped two-call API) on the same input,
    row for row and bit for bit."""
    import torch

    import pixeltable_yolox_b200 as yx

    pred = model(engine.input)                                       # separate engine without postprocess: cxcywh rows
    want = yx.postprocess(pred, model.head.num_classes, args.conf, args.nms, nms_variant="auto")
    cnt = engine.det_count.cpu().tolist()
    ok, rows = True, 0
    for b, w in enumerate(want):
        n = min(cnt[b], args.max_det)
        if w is None:
            ok = ok and cnt[b] == 0
            continue
        ok = ok and cnt[b] == w.shape[0] and torch.equal(engine.dets[b, :n], w[:n])
        rows += n
    key = next(k for k, e in model._engines.items() if e.post is None and k[0] == tuple(engine.input.shape))
    model._engines.pop(key).close()
    return {"parity_checked": bool(ok), "parity_rows": rows,
            "parity_how": "last timed step's detections == YoloxModule.forward + postprocess on the same batch (torch.equal per image)"}


DUMP_BYTES = 64 << 20                   # --dump-outputs: at most this much in all
PRED_SAMPLE_ROWS = 65536                # head-output rows kept in the dump (seeded sample; 22 MB at 85 columns)


def dump_outputs(out_dir: str, engine, max_det: int) -> dict:
    """--dump-outputs: what the timed step hands its caller (YoloxModule.detect returns dets / det_idx / det_count, the
    engine's forward the head output), copied after the timed region and written as float32 / float64 .npy files:
      dets [B, K, 7] f32, det_idx [B, K] f64, det_count [B] f64: K is the largest kept count of the batch (at most max_det);
          the rows past an image's own count are zero in dets and -1 in det_idx (the buffers leave them undefined)
      pred_rows [N, 5 + nc] f32: the rows pred_rows_index [N] f64 (row numbers of the flattened [B * A] head output) of a
          fixed, seeded sample of the head output, which is too large to store whole (183 MB for yolox_s at batch 64)."""
    import numpy as np
    import torch

    count = engine.det_count.cpu()
    kept = count.clamp(max=max_det).long()
    k = int(kept.max().item()) if kept.numel() else 0
    live = torch.arange(k)[None, :] < kept[:, None]
    dets = torch.where(live[..., None], engine.dets[:, :k].cpu(), torch.zeros(()))
    idx = torch.where(live, engine.det_idx[:, :k].cpu(), torch.full((), -1, dtype=torch.int64))
    pred = engine.pred.reshape(-1, engine.pred.shape[-1])
    left = DUMP_BYTES - 4 * dets.numel() - 8 * idx.numel() - 8 * count.numel()
    n = max(0, min(pred.shape[0], PRED_SAMPLE_ROWS, left // (4 * pred.shape[1] + 8)))
    rows = np.sort(np.random.default_rng(0).choice(pred.shape[0], size=n, replace=False))
    out = {"dets": dets.float().numpy(), "det_idx": idx.double().numpy(), "det_count": count.double().numpy(),
           "pred_rows": pred[torch.from_numpy(rows).to(pred.device)].float().cpu().numpy(),
           "pred_rows_index": rows.astype(np.float64)}
    os.makedirs(out_dir, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)
    return {name: list(a.shape) for name, a in out.items()}


def extra_conf_leg(args, model, dev_in, conf: float, steps: int) -> dict:
    """The same step at another score threshold (0.01 = the evaluator's test_conf, yolox/config.py:115)."""
    import torch

    from pixeltable_yolox_b200.boxes import NMS_VARIANTS

    post = dict(conf_thre=conf, nms_thre=args.nms, nms_variant=NMS_VARIANTS["auto"], max_det=args.max_det)
    eng = [model.engine_for(dev_in[0], post, slot=10 + i) for i in range(2)]
    for i in range(2):
        eng[i].input.copy_(dev_in[i])
    for i in range(4):
        eng[i % 2].forward(eng[i % 2].input)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(steps):
        eng[i % 2].forward(eng[i % 2].input)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    last = eng[(steps - 1) % 2]
    scores = last.pred[..., 4] * last.pred[..., 5:].max(-1).values
    out = {"conf_thre": conf, "value": args.batch / (ms / 1e3), "unit": "images/s (one GPU, inputs resident)", "ms_per_step": ms,
           "steps": steps, "candidates_per_image_mean": float((scores >= conf).float().sum(1).mean().item()),
           "kept_per_image_mean": float(last.det_count.float().mean().item())}
    for k in [k for k, e in model._engines.items() if e in eng]:
        model._engines.pop(k).close()
    return out


def extra_config5(args, dev, pk, ref) -> dict:
    """BASELINE.json config 5: dense-scene NMS stress on a synthetic decoded head tensor [64, 8400, 85] (SURVEY 8d),
    thr 0.001 / 0.25 / 0.5, nms 0.65: filter_kernel and sort_nms_kernel device times, GB/s against the bytes they must
    move, and the reference's postprocess (torchvision CUDA batched_nms, per-image Python loop) on the same tensor."""
    import torch

    from pixeltable_yolox_b200 import ops
    from pixeltable_yolox_b200 import synthetic as syn
    from pixeltable_yolox_b200.boxes import NMS_VARIANTS

    B, A, nc = 64, 8400, 80
    pred = torch.from_numpy(syn.dense_scene(B, anchors=A, seed=13)).to(dev)
    ws = ops._workspace(dev, ops.lib().yx_postprocess_workspace_bytes(B, A), "post")
    rows = []
    for thr in (0.001, 0.25, 0.5):
        _, _, cnt = ops.postprocess_device(pred.clone(), nc, thr, 0.65, NMS_VARIANTS["auto"], inplace_xyxy=True)
        work = pred.clone()
        t_total = timed_us(lambda: ops.postprocess_device(work, nc, thr, 0.65, NMS_VARIANTS["auto"], inplace_xyxy=False))
        t_nms = timed_us(lambda: ops.nms_prefiltered(ws, B, A, 0.65, NMS_VARIANTS["auto"]))     # candidates of the last filter pass
        t_filter = max(t_total - t_nms, 1e-3)
        scores = pred[..., 4] * pred[..., 5:].max(-1).values
        n_cand = int((scores >= thr).sum().item())
        kept = int(cnt.sum().item())
        filter_bytes = B * A * ((5 + nc) * 4 + 32) + n_cand * 8           # rows read, candidate rows + keys written
        nms_bytes = n_cand * (32 + 8) + kept * (28 + 8)                   # candidate rows + keys read, detections written
        row = {"conf_thre": thr, "candidates_per_image": n_cand / B, "kept_per_image": kept / B,
               "postprocess_us": t_total, "filter_us": t_filter, "sort_nms_us": t_nms, "us_per_image": t_total / B,
               "filter_GBps": filter_bytes / t_filter / 1e3, "filter_frac_of_hbm_peak": filter_bytes / t_filter / 1e3 / pk["hbm"],
               "sort_nms_GBps_minimal_bytes": nms_bytes / t_nms / 1e3,
               "sort_nms_frac_of_hbm_peak": nms_bytes / t_nms / 1e3 / pk["hbm"]}
        if ref is not None:
            try:
                def ref_post():
                    ref["postprocess"](pred.clone(), nc, thr, 0.65, class_agnostic=False)
                ref_post(); torch.cuda.synchronize()
                t0 = time.perf_counter()
                for _ in range(3):
                    ref_post()
                torch.cuda.synchronize()
                row["reference_postprocess_us_same_gpu"] = (time.perf_counter() - t0) / 3 * 1e6
            except Exception as e:                    # noqa: BLE001
                row["reference_postprocess_us_same_gpu"] = f"failed: {e!r}"
        rows.append(row)
    return {"workload": "synthetic dense scenes [64, 8400, 85] fp32 (synthetic.dense_scene seed 13), nms 0.65, config[4] of BASELINE.json",
            "hbm_peak_GBps": pk["hbm"], "rows": rows,
            "note": "sort_nms is latency-bound (one thread-block cluster of 2 CTAs per image at batch 64, 4 / 8 at smaller batches; "
                    "merge sort, suppression mask and kept list stay in (distributed) shared memory): its GB/s is quoted against "
                    "the minimal bytes (candidates in, detections out)"}


def extra_hbm_families(prof, pk) -> dict:
    """Per-family achieved GB/s of the HBM-bound launches of the step (algorithmic bytes / device time of the eager
    per-op pass), against the measured copy bandwidth."""
    fam = {}
    for q in prof:
        name = q["name"]
        if name.startswith("conv1x1") and "->96 " in name:
            key = "head prediction GEMM (decode + score filter epilogue)"
        elif name.startswith("conv1x1"):
            key = "conv1x1 @" + name.split("@")[1]
        elif name.startswith(("spp", "dwconv", "focus", "bottleneck", "sort+nms", "conv3x3s2")):
            key = name.split(" ")[0] + (" @" + name.split("@")[1] if "@" in name else "")
        else:
            continue
        f = fam.setdefault(key, dict(launches=0, us=0.0, bytes=0.0))
        f["launches"] += 1; f["us"] += q["ms"] * 1e3; f["bytes"] += q["bytes"]
    out = {}
    for k, f in fam.items():
        gbps = f["bytes"] / max(f["us"], 1e-9) / 1e3
        out[k] = {"launches": f["launches"], "us": round(f["us"], 1), "GBps": round(gbps, 1), "frac_of_hbm_peak": round(gbps / pk["hbm"], 3)}
    return out


def extra_torch_gpu(args, sd_cpu, dev_in, ref, dtype) -> dict:
    """The reference on the same box: its unmodified YoloxModule in the bench dtype on cuDNN (torch eager, cudnn.benchmark,
    both memory formats tried) + its own postprocess (torchvision CUDA batched_nms) on the same resident inputs."""
    import torch

    if ref is None:
        return {"unavailable": "baseline/_ref missing (python baseline/install_ref.py)"}
    dev = dev_in[0].device
    torch.backends.cudnn.benchmark = True
    best = None
    for fmt_name, fmt in (("contiguous", torch.contiguous_format), ("channels_last", torch.channels_last)):
        try:
            m = reference_model(ref, args.model, sd_cpu, dev, dtype).to(memory_format=fmt)
            xs = [d.to(dtype).contiguous(memory_format=fmt) for d in dev_in]

            def step(i):
                with torch.no_grad():
                    out = m(xs[i % 2])
                return ref["postprocess"](out.float(), m.head.num_classes, args.conf, args.nms, class_agnostic=False)

            for i in range(3):
                step(i)
            torch.cuda.synchronize()
            n = 10
            t0 = time.perf_counter()
            for i in range(n):
                step(i)
            torch.cuda.synchronize()
            rate = n * xs[0].shape[0] / (time.perf_counter() - t0)
            if best is None or rate > best["value"]:
                best = {"value": rate, "unit": "images/s (one GPU, inputs resident)", "memory_format": fmt_name, "steps": n}
            del m, xs
            torch.cuda.empty_cache()
        except Exception as e:                        # noqa: BLE001
            print(f"# torch_gpu leg ({fmt_name}) failed: {e!r}", file=sys.stderr)
    if best is None:
        return {"unavailable": "the reference module failed on this GPU (see stderr)"}
    best["what"] = (f"unmodified reference YoloxModule ({args.dtype}, cuDNN, torch eager) + yolox.utils.postprocess "
                    "(torchvision.ops.batched_nms on CUDA), same weights and inputs; informational")
    return best


def extra_user_api(args, model, host_u8) -> dict:
    """The reference-shaped user call, `Yolox.__call__(list of PIL images, threshold)` (yolox/models/yolox.py:41-52): PIL ->
    numpy, letterbox ON THE DEVICE from the raw image bytes (YoloxProcessor.device), fused detect graph, one D2H copy, Python
    `Detections` dictionaries. Wall clock, everything included; informational (the per-image Python work dominates)."""
    import torch
    from PIL import Image

    import pixeltable_yolox_b200 as yx

    dev = next(model.parameters()).device
    proc = yx.YoloxProcessor(args.model)
    proc.device, proc.dtype = dev, torch.uint8
    wrapper = yx.Yolox(model, proc)
    imgs = [Image.fromarray(host_u8[i].permute(1, 2, 0).contiguous().numpy()) for i in range(host_u8.shape[0])]
    res = wrapper(imgs, threshold=args.conf)
    torch.cuda.synchronize()
    n = 5
    t0 = time.perf_counter()
    for _ in range(n):
        res = wrapper(imgs, threshold=args.conf)
    torch.cuda.synchronize()
    dt = (time.perf_counter() - t0) / n
    return {"value": len(imgs) / dt, "unit": "images/s (one GPU, wall clock)", "ms_per_call": 1e3 * dt, "images_per_call": len(imgs),
            "detections_last_call": sum(len(r["labels"]) for r in res),
            "what": "Yolox.__call__(list of 640x640 PIL images): PIL -> numpy -> one H2D of the raw bytes -> device letterbox -> "
                    "fused detect graph -> one D2H -> Python Detections; informational"}


def run_ours(args):
    import numpy as np
    import torch
    import torch.distributed as dist

    from pixeltable_yolox_b200 import synthetic as syn
    from pixeltable_yolox_b200.boxes import NMS_VARIANTS
    from pixeltable_yolox_b200.sharding import shard_range

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the B200 path has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    numa = bind_to_gpu_numa_node(local) if world > 1 and os.environ.get("YX_NUMA_BIND", "1") != "0" else None
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    if args.train:
        return run_train(args, world, rank, dev)

    dtype = {"bf16": torch.bfloat16, "fp16": torch.float16, "fp32": torch.float32}[args.dtype]
    cfg, model = build_model(args, dev)
    sd_cpu = {k: v.detach().float().cpu().clone() for k, v in model.state_dict().items()} if rank == 0 else None
    model = model.to(dtype).eval()
    model.micro_batch = args.micro_batch
    S = args.size
    if args.global_batch:                      # strong scaling: this rank's contiguous slice of the global batch
        lo, hi = shard_range(args.global_batch, rank, world)
        B = hi - lo
        total_images = args.global_batch
    else:
        B = args.batch
        total_images = B * world
    # two distinct synthetic batches per rank, alternated, each > 126 MB L2 (315 MB fp32 at batch 64)
    host = [torch.from_numpy(syn.images(B, S, S, seed=7 + 100 * rank + i)).pin_memory() for i in range(2)]
    dev_in = [h.to(dev) for h in host]
    post = dict(conf_thre=args.conf, nms_thre=args.nms, nms_variant=NMS_VARIANTS["auto"], max_det=args.max_det)
    eng = [model.engine_for(dev_in[0], post, slot=i) for i in range(2)]
    launches_per_step = eng[0].launches

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---------------- value: inputs resident in HBM ----------------
    # Two engines (own plan, own activation buffers) alternate, each with its batch already in its input buffer: no
    # staging copy inside the timed region, and every step reads an input batch the previous step did not touch.
    for i in range(2):
        eng[i].input.copy_(dev_in[i])
    clocks = ClockSampler(local)
    clocks.start()                # before the warm-up: nvidia-smi needs ~100-300 ms before its first row
    clocks.wait_first()
    for i in range(args.warmup):
        eng[i % 2].forward(eng[i % 2].input)
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    w0 = time.perf_counter()
    e0.record()
    for i in range(args.steps):
        eng[i % 2].forward(eng[i % 2].input)
    e1.record()
    torch.cuda.synchronize()
    w1 = time.perf_counter()
    ms = e0.elapsed_time(e1)
    clocks.mark(w0, w1)           # keep the rows sampled while the timed steps ran
    clk = clocks.stop()
    per_rank_ms, per_rank_clk = [ms / args.steps], [clk]
    if world > 1:
        t = torch.tensor([ms], device=dev)
        allt = [torch.zeros_like(t) for _ in range(world)]
        dist.all_gather(allt, t)
        per_rank_ms = [float(v.item()) / args.steps for v in allt]
        ms = max(float(v.item()) for v in allt)
        per_rank_clk = [None] * world
        dist.all_gather_object(per_rank_clk, clk)
    barrier()
    value = total_images * args.steps / (ms / 1e3)
    last = eng[(args.steps - 1) % 2]
    if args.dump_outputs and rank == 0:
        shapes = dump_outputs(args.dump_outputs, last, args.max_det)
        print(f"# outputs of the last timed step written to {args.dump_outputs}: {shapes}", file=sys.stderr)
    kept = int(last.det_count.clamp(max=args.max_det).sum().item())
    kept_true_mean = float(last.det_count.float().mean().item())
    scores = last.pred[..., 4] * last.pred[..., 5:].max(-1).values
    cand_mean = float((scores >= args.conf).float().sum(1).mean().item())
    parity = parity_check(model, last, args) if rank == 0 else None

    # ---------------- e2e: host buffers in, detections out, every step ----------------
    # Headline: uint8 pixels (what decoders / YoloxProcessor(dtype=torch.uint8) produce; exactly the values the
    # reference's float 0..255 tensor holds) are uploaded and converted by the stem kernel. The fp32 host tensor
    # of the reference's own processor is timed too (e2e_fp32_input): 4x the PCIe bytes for the same pixels.
    streams = [torch.cuda.Stream(dev), torch.cuda.Stream(dev)]
    out_host = [torch.empty((B, args.max_det, 7), dtype=torch.float32).pin_memory() for _ in range(2)]
    cnt_host = [torch.empty((B,), dtype=torch.int32).pin_memory() for _ in range(2)]

    def run_e2e(hosts, engines):
        def e2e_step(i):
            s = i % 2
            with torch.cuda.stream(streams[s]):
                engines[s].forward(hosts[s])                  # H2D copy + graph on this stream
                out_host[s].copy_(engines[s].dets, non_blocking=True)
                cnt_host[s].copy_(engines[s].det_count, non_blocking=True)

        for i in range(max(2, args.warmup)):
            e2e_step(i)
        barrier()
        t0 = time.perf_counter()
        for i in range(args.steps):
            e2e_step(i)
            if i >= 1:
                streams[(i - 1) % 2].synchronize()            # consume step i-1's detections while step i runs
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        if world > 1:
            t = torch.tensor([dt], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dt = float(t.item())
        return total_images * args.steps / dt

    host_u8 = [h.to(torch.uint8).pin_memory() for h in host]
    eng_u8 = [model.engine_for(host_u8[0], post, slot=i) for i in range(2)]
    e2e_value = run_e2e(host_u8, eng_u8)
    kept_u8 = int(eng_u8[(args.steps - 1) % 2].det_count.clamp(max=args.max_det).sum().item())
    e2e_fp32 = run_e2e(host, eng)
    h2d = host_u8[0].numel() * host_u8[0].element_size()
    h2d_fp32 = host[0].numel() * host[0].element_size()
    d2h = out_host[0].numel() * 4 + cnt_host[0].numel() * 4

    # ---------------- roofline of the dominant kernel (rank 0, eager pass with per-op events) ----------------
    line = None
    if rank == 0:
        pk = peaks()
        prof = eng[0].builder.profile()
        prof = eng[0].builder.profile()
        tc = [p for p in prof if p["kind"] == 0]
        tc_ms = sum(p["ms"] for p in tc)
        tc_flops = sum(p["flops"] for p in tc)
        all_ms = sum(p["ms"] for p in prof)
        achieved = tc_flops / (tc_ms / 1e3) / 1e12 if tc_ms > 0 else 0.0
        if args.profile_ops:
            for p in prof:
                print(f"# {p['name']:44s} {p['ms']*1e3:9.1f} us  {p['flops']/max(p['ms'],1e-9)/1e9:8.1f} TFLOP/s  "
                      f"{p['bytes']/max(p['ms'],1e-9)/1e6:8.1f} GB/s", file=sys.stderr)
        traffic, traffic_src = None, None
        tfiles = sorted(f for f in (ROOT / "profiles").glob("*_traffic.json") if "train" not in f.name)   # the inference step's own list
        if tfiles:                                   # DRAM bytes per launch of the same kernel from the committed ncu pass
            tj = json.loads(tfiles[-1].read_text())
            traffic, traffic_src = tj.get("dram_bytes_per_launch"), f"profiles/{tfiles[-1].name}"
        roof = {"bound": "tensor", "kernel": "conv_tc_kernel (tcgen05 implicit GEMM)", "achieved": achieved,
                "peak": pk["tf_sustained"], "unit": "TFLOP/s", "frac": achieved / pk["tf_sustained"], "traffic": traffic,
                "traffic_unit": "DRAM bytes per launch (dram__bytes_read.sum + dram__bytes_write.sum, ncu)",
                "traffic_source": traffic_src,
                "algorithmic_flops_per_launch": tc_flops / max(len(tc), 1),
                "peak_source": pk["source"] + " bf16 sustained (kernel timed inside a long step)",
                "launches": len(tc), "avg_launch_us": 1e3 * tc_ms / max(len(tc), 1), "share_of_step": tc_ms / all_ms,
                "whole_step_frac_of_peak": GFLOP_PER_IMAGE.get(args.model, 0) * 1e9 * (value / world) / (pk["tf_sustained"] * 1e12)}
        extra = {"hbm_bound_families": extra_hbm_families(prof, pk)}
        cpu = None
        if world == 1 and not args.no_extras:
            ref = reference_modules()
            try:
                extra["thr001"] = extra_conf_leg(args, model, dev_in, 0.01, min(args.steps, 20))
            except Exception as e:                    # noqa: BLE001 - an extra leg never takes the headline down
                extra["thr001"] = {"failed": repr(e)}
            try:
                extra["config5"] = extra_config5(args, dev, pk, ref)
            except Exception as e:                    # noqa: BLE001
                extra["config5"] = {"failed": repr(e)}
            try:
                extra["torch_gpu"] = extra_torch_gpu(args, sd_cpu, dev_in, ref, dtype)
            except Exception as e:                    # noqa: BLE001
                extra["torch_gpu"] = {"failed": repr(e)}
            try:
                extra["user_api"] = extra_user_api(args, model, host_u8[0])
            except Exception as e:                    # noqa: BLE001
                extra["user_api"] = {"failed": repr(e)}
        if world == 1 and not args.no_cpu_baseline:   # N = 1 only: seven other ranks would spin in a barrier meanwhile
            imgs = host[0][:args.cpu_images].numpy()
            rate, threads, n = cpu_reference_rate(args, sd_cpu, imgs)
            cpu = {"value": rate, "unit": "images/s", "cores": threads, "kind": "port",
                   "sample": f"{n} of the step's images, oracle/ torch-CPU fp32 forward + numpy/C NMS"}
        vs = None
        in_mb = dev_in[0].numel() * dev_in[0].element_size() / 1e6
        line = {
            "metric": "images_per_second", "value": value, "unit": "images/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True,
            "scaling": "strong" if args.global_batch else "weak",
            "vs_baseline": vs, "dtype": args.dtype, "data": "synthetic",
            "config": {"workload": workload_name(args),
                       "per_gpu_batch": B, "global_batch": total_images, "micro_batch": args.micro_batch,
                       "conf_thre": args.conf, "nms_thre": args.nms, "nms_variant": "auto (torchvision CUDA rule)",
                       "weights": "random init, BN calibrated (synthetic.randomize_and_calibrate)",
                       "l2": f"two alternating engines, each with its own {in_mb:.0f} MB input batch resident in its input buffer (> 126 MB L2)",
                       "detections_kept_last_step": kept, "kept_per_image_mean": kept_true_mean,
                       "candidates_per_image_mean": cand_mean},
            "e2e": {"value": e2e_value, "unit": "images/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "input": "pinned host uint8 [B,3,H,W] pixels, converted on device by the stem kernel; "
                             "double-buffered over 2 streams", "detections_kept_last_step": kept_u8,
                    "numa_node_rank0": numa},
            "e2e_fp32_input": {"value": e2e_fp32, "unit": "images/s", "h2d_bytes_per_step": h2d_fp32,
                               "d2h_bytes_per_step": d2h,
                               "input": "pinned host fp32 [B,3,H,W] (the reference processor's dtype), same pixels"},
            "gpu_launches": launches_per_step * args.steps,
            "launches_per_step": launches_per_step,
            "roofline": roof, "cpu_baseline": cpu, "clocks": clk,
            "per_rank": {"ms_per_step": per_rank_ms, "clocks": per_rank_clk},
            "extra": extra,
        }
        line.update(parity)
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


# ------------------------------------------------------------------------------------------------------------------
# config 4: training step
# ------------------------------------------------------------------------------------------------------------------
def train_batch(args, rank: int, B: int):
    """Images as config 2; labels [B, 120, 5] per SURVEY 8d config 4: G ~ randint(0, 50) per image with one G = 0 and one
    G = 120 image on rank 0, cls ~ randint(80), centres inside the image, w,h ~ U(8, 208), zero padded."""
    import torch

    from pixeltable_yolox_b200 import synthetic as syn

    import numpy as np

    rng = np.random.default_rng(3 + rank)
    counts = [int(rng.integers(0, 50)) for _ in range(B)]
    if rank == 0 and B >= 2:
        counts[0], counts[1] = 0, 120
    x = torch.from_numpy(syn.images(B, args.size, args.size, seed=7 + 100 * rank))
    lab = torch.from_numpy(syn.labels(B, max_gt=120, seed=3 + rank, size=float(args.size), counts=counts))
    return x, lab, counts


def sgd_for(model):
    """The reference's optimizer (yolox/config.py:307-333): SGD momentum 0.9 nesterov; BN weights and biases without
    weight decay, conv / linear weights with 5e-4."""
    import torch
    import torch.nn as nn

    pg0, pg1, pg2 = [], [], []
    for _, v in model.named_modules():
        if hasattr(v, "bias") and isinstance(v.bias, nn.Parameter):
            pg2.append(v.bias)
        if isinstance(v, nn.BatchNorm2d) or "bn" in type(v).__name__.lower():
            pg0.append(v.weight)
        elif hasattr(v, "weight") and isinstance(v.weight, nn.Parameter):
            pg1.append(v.weight)
    opt = torch.optim.SGD(pg0, lr=1e-3, momentum=0.9, nesterov=True)
    opt.add_param_group({"params": pg1, "weight_decay": 5e-4})
    opt.add_param_group({"params": pg2})
    return opt


class TorchSgdWithEma:
    """The reference's own optimizer + EMA pair for the same-box reference arm: torch.optim.SGD (config.py:307-333) and the
    reference's ModelEMA.update (yolox/utils/ema.py:46-58), called like Trainer.train_one_iter does (trainer.py:119-124)."""

    def __init__(self, model, ema_cls):
        self.opt = sgd_for(model)
        self.model = model
        self.ema = ema_cls(model, 0.9998) if ema_cls is not None else None

    def zero_grad(self, set_to_none=True):
        self.opt.zero_grad(set_to_none=set_to_none)

    def step(self):
        self.opt.step()
        if self.ema is not None:
            self.ema.update(self.model)


def time_train_steps(model, opt, x, lab, steps, warm, amp_dtype, world, dev, host=None):
    """ms per step (device events, max over ranks) and the phase split of the last step. `host`: (pinned images, pinned
    labels) -> every step uploads them and reads the loss back (the e2e leg)."""
    import torch
    import torch.distributed as dist

    def one(i, ev=None):
        if host is not None:
            x.copy_(host[0], non_blocking=True); lab.copy_(host[1], non_blocking=True)
        if ev: ev[0].record()
        with torch.autocast("cuda", dtype=amp_dtype, enabled=amp_dtype is not None):
            out = model(x, lab)
        loss = out["total_loss"]
        if ev: ev[1].record()
        opt.zero_grad()
        loss.backward()
        if ev: ev[2].record()
        opt.step()
        if ev: ev[3].record()
        return float(loss.item()) if host is not None else loss

    for i in range(warm):
        one(i)
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
    e0.record()
    for i in range(steps):
        loss = one(i, ev if i == steps - 1 else None)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    if world > 1:
        t = torch.tensor([ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    phases = {"forward_incl_assignment_and_losses_ms": ev[0].elapsed_time(ev[1]), "backward_incl_allreduce_ms": ev[1].elapsed_time(ev[2]),
              "optimizer_ms": ev[2].elapsed_time(ev[3])}
    return ms / steps, phases, float(loss) if not isinstance(loss, float) else loss


def time_train_graph(model, opt, x, lab, steps, amp_dtype, world, dev, host=None):
    """The whole training step -- forward, SimOTA assignment, losses, backward (+ DDP all-reduce), SGD + EMA -- captured ONCE
    as a CUDA graph and replayed: possible because nothing in our step synchronises with the host (the reference's
    get_assignments reads device scalars per image and per GT, yolo_head.py:269-351,549-564, and cannot be captured).
    The learning rate and the EMA ramp reach the captured optimizer launch through a 12-byte device buffer."""
    import torch
    import torch.distributed as dist

    if world > 1:
        # a copy of the module WITHOUT the DDP wrapper: DDP's gradient hooks live on the parameters themselves and launch on
        # streams of their own during backward, which a stream capture rejects (cudaErrorStreamCaptureImplicit)
        import copy

        from pixeltable_yolox_b200.optim import FusedSgdEma

        raw = copy.deepcopy(model.module).train()
        if amp_dtype is not None and os.environ.get("YX_TRAIN_CONV", "1") != "0":
            from pixeltable_yolox_b200 import train_conv

            train_conv.attach_packer(raw, amp_dtype)
        kw = dict(lr=opt.lr, momentum=opt.momentum, weight_decay=5e-4, nesterov=opt.nesterov, ema=True, ema_decay=opt.ema_decay,
                  direct_grads=True)
        # the flat gradient buffer as symmetric memory (every rank maps every peer's buffer over NVLink): all-reduce + SGD +
        # EMA run as ONE kernel of ours over those mappings and the whole step is one graph; without symmetric memory the
        # step is two graphs around an eager ncclAllReduce. Every rank must take the same branch.
        fused_collective = os.environ.get("YX_FUSED_ALLREDUCE", "1") != "0"
        try:
            opt = FusedSgdEma(raw, peer_group=dist.group.WORLD if fused_collective else None, **kw)
        except Exception as e:                      # noqa: BLE001
            print(f"# symmetric memory unavailable ({e!r}): NCCL all-reduce between two graphs", file=sys.stderr)
            fused_collective = False
            opt = FusedSgdEma(raw, **kw)
        ok = torch.tensor([1 if fused_collective else 0], device=dev)
        dist.all_reduce(ok, op=dist.ReduceOp.MIN)
        if fused_collective and int(ok.item()) == 0:                     # some rank fell back: all do
            fused_collective = False
            opt = FusedSgdEma(raw, **kw)
    else:
        raw = model
        fused_collective = False
    time_train_graph.fused_collective = fused_collective

    def eager():
        with torch.autocast("cuda", dtype=amp_dtype, enabled=amp_dtype is not None):
            out = raw(x, lab)
        opt.zero_grad()
        out["total_loss"].backward()
        if world > 1:
            opt.join()
            dist.all_reduce(opt.flat_grad)
            opt.flat_grad.div_(world)
        opt.step()

    side = torch.cuda.Stream(dev)
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(3):
            eager()
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    # With several ranks the step is TWO graphs around one eager ncclAllReduce of the flattened gradients:
    # graph 1 = forward + assignment + losses + backward + flatten, graph 2 = average + scatter + SGD/EMA
    params = [q for q in raw.parameters() if q.requires_grad]
    g, g2, flat = torch.cuda.CUDAGraph(), None, None
    with torch.cuda.graph(g, capture_error_mode="thread_local"):
        with torch.autocast("cuda", dtype=amp_dtype, enabled=amp_dtype is not None):
            out = raw(x, lab)
        loss = out["total_loss"]
        opt.zero_grad()
        loss.backward()
        opt.join()                                 # side-stream weight gradients rejoin the captured stream
        if fused_collective:
            opt.step_allreduce_captured()          # reduce-scatter over peer memory -> all-gather fused with SGD + EMA
        elif world > 1:
            flat = opt.flat_grad                   # every .grad is a view into it: the all-reduce needs no flatten / scatter
        else:
            opt.step_captured()
    if world > 1 and not fused_collective:
        g2 = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g2, capture_error_mode="thread_local"):
            flat.div_(world)
            opt.step_captured()

    def replay():
        opt.set_hyper()
        g.replay()
        if world > 1 and not fused_collective:
            dist.all_reduce(flat)
            g2.replay()

    def timed(fn):
        for _ in range(3):
            fn()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms / steps

    ms_resident = timed(replay)
    loss_resident = float(loss.item())
    ms_host, loss_host = None, None
    if host is not None:
        last = [0.0]

        def from_host():                 # every step: H2D of the pinned images + labels, replay, loss read back
            x.copy_(host[0], non_blocking=True); lab.copy_(host[1], non_blocking=True)
            replay()
            last[0] = float(loss.item())

        ms_host = timed(from_host)
        loss_host = last[0]
    return ms_resident, loss_resident, ms_host, loss_host


def run_train(args, world, rank, dev):
    import torch
    import torch.distributed as dist

    from pixeltable_yolox_b200 import ops

    B = args.train_batch
    amp_dtype = {"bf16": torch.bfloat16, "fp16": torch.float16, "fp32": None}[args.dtype]
    cfg, model = build_model(args, dev)
    sd_cpu = {k: v.detach().float().cpu().clone() for k, v in model.state_dict().items()}
    model.train()
    if args.train_format == "channels_last":
        model = model.to(memory_format=torch.channels_last)
    if amp_dtype is not None and os.environ.get("YX_TRAIN_CONV", "1") != "0":
        from pixeltable_yolox_b200 import train_conv

        train_conv.attach_packer(model, amp_dtype)       # every conv weight packed to its 16-bit operands in one launch per step
    n_grad = sum(p.numel() for p in model.parameters() if p.requires_grad)
    net = model
    if world > 1:
        net = torch.nn.parallel.DistributedDataParallel(model, device_ids=[dev.index], broadcast_buffers=False)
    from pixeltable_yolox_b200.optim import FusedSgdEma

    # one rank: no DDP wrapper, so the backward kernels may add weight gradients straight into one flat .grad buffer
    opt = FusedSgdEma(model, lr=1e-3, momentum=0.9, weight_decay=5e-4, nesterov=True, ema=True, ema_decay=0.9998,
                      direct_grads=(world == 1))
    xh, labh, counts = train_batch(args, rank, B)
    xh, labh = xh.pin_memory(), labh.pin_memory()
    x, lab = xh.to(dev), labh.to(dev)
    if args.train_format == "channels_last" and os.environ.get("YX_TRAIN_CONV", "1") == "0":
        x = x.contiguous(memory_format=torch.channels_last)      # (our Focus kernel reads the NCHW image as it arrives)
    clocks = ClockSampler(dev.index)
    clocks.start(); clocks.wait_first()
    w0 = time.perf_counter()
    ms, phases, loss = time_train_steps(net, opt, x, lab, args.steps, args.warmup, amp_dtype, world, dev)
    clocks.mark(w0 + 0.0, time.perf_counter())
    clk = clocks.stop()
    ms_e2e, _, loss_e2e = time_train_steps(net, opt, x, lab, args.steps, 2, amp_dtype, world, dev, host=(xh, labh))

    # ---- the same step as one CUDA graph (our step has no host synchronisation; the reference's cannot be captured)
    graph_line = None
    try:
        gms, gloss, gms_host, gloss_host = time_train_graph(net, opt, x, lab, args.steps, amp_dtype, world, dev, host=(xh, labh))
        graph_line = {"ms_per_step": gms, "images_per_second": world * B / (gms / 1e3), "loss_last_step": gloss,
                      "e2e_ms_per_step": gms_host, "e2e_images_per_second": world * B / (gms_host / 1e3), "e2e_loss_last_step": gloss_host,
                      "what": ("forward + SimOTA + losses + backward + SGD/EMA captured once with torch.cuda.graph and replayed"
                               if world == 1 else
                               "ONE captured graph per step: forward + SimOTA + losses + backward + yx_allreduce_sgd_ema_step (gradient "
                               "all-reduce over NVLink peer memory -- reduce-scatter in rank order, all-gather fused with the SGD + EMA "
                               "update -- as one kernel of ours on the symmetric flat gradient buffer; no NCCL call in the step), on a "
                               "copy of the module without the DDP wrapper"
                               if getattr(time_train_graph, "fused_collective", False) else
                               "two captured graphs (forward + SimOTA + losses + backward | average + SGD/EMA) around one eager "
                               "ncclAllReduce of the flat gradient buffer every .grad is a view of, on a copy of the module "
                               "without the DDP wrapper") + "; lr / EMA decay reach the captured optimizer launch via a device buffer"}
        if world == 1 and amp_dtype is not None and os.environ.get("YX_TRAIN_CONV", "1") != "0":
            # the same graph step fed with uint8 images (the pixels are integers 0..255: exact; the Focus kernel reads them as
            # bytes): a quarter of the upload. The reference's data path hands the trainer fp32 images, so `e2e` stays fp32.
            try:
                xh8 = xh.to(torch.uint8).pin_memory()
                _, _, gms_u8, gloss_u8 = time_train_graph(net, opt, xh8.to(dev), lab, args.steps, amp_dtype, world, dev, host=(xh8, labh))
                graph_line.update({"e2e_uint8_input_ms_per_step": gms_u8, "e2e_uint8_input_images_per_second": B / (gms_u8 / 1e3),
                                   "e2e_uint8_input_h2d_bytes_per_step": xh8.numel() + labh.numel() * 4,
                                   "e2e_uint8_input_loss_last_step": gloss_u8})
            except Exception as e:                    # noqa: BLE001
                graph_line["e2e_uint8_input_failed"] = repr(e)[:200]
    except Exception as e:                            # noqa: BLE001
        import traceback

        graph_line = {"failed": repr(e)[:300]}
        print("# cuda-graph training step failed:\n" + traceback.format_exc(), file=sys.stderr)
        try:
            torch.cuda.synchronize()
        except Exception:                             # noqa: BLE001
            pass

    # ---- our kernels of the step, stand-alone on this rank's head output shape
    model.eval()        # BN statistics are irrelevant here: only shapes and value ranges of the head output matter
    with torch.no_grad():
        from pixeltable_yolox_b200 import synthetic as syn
        from oracle.simota_oracle import anchor_grid          # anchor grid helper only (test infrastructure, not timed)
    hw = [(args.size // s, args.size // s) for s in (8, 16, 32)]
    import numpy as np

    xs, ys, st = (torch.from_numpy(a).to(dev) for a in anchor_grid(hw, (8, 16, 32)))
    pred = torch.from_numpy(syn.train_head_output(B, hw, (8, 16, 32), labh.numpy(), seed=4 + rank)).to(dev)
    asg = ops.simota_assign(pred, lab, xs, ys, st, 80, levels=3)

    def graph_us(fn):
        fn(); torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            fn()
        return timed_us(g.replay, 20)

    t_simota = graph_us(lambda: ops.simota_assign(pred, lab, xs, ys, st, 80, levels=3))
    t_loss = graph_us(lambda: ops.head_losses(pred, lab, asg))
    # ---- the gradient all-reduce alone (one flat fp32 buffer of every gradient)
    t_ar = None
    if world > 1:
        flat = torch.zeros(n_grad, dtype=torch.float32, device=dev)
        t_ar = timed_us(lambda: dist.all_reduce(flat), 20)
        tt = torch.tensor([t_ar], device=dev); dist.all_reduce(tt, op=dist.ReduceOp.MAX); t_ar = float(tt.item())

    # ---- the reference-shaped torch-only step on the same box (unmodified reference module, same optimizer / AMP / DDP)
    ref_line = None
    ref = reference_modules()
    if ref is not None and not args.no_extras:
        try:
            rmodel = reference_model(ref, args.model, sd_cpu, dev).train()
            rnet = rmodel
            if world > 1:
                rnet = torch.nn.parallel.DistributedDataParallel(rmodel, device_ids=[dev.index], broadcast_buffers=False)
            try:
                from yolox.utils import ModelEMA
            except Exception:                         # noqa: BLE001
                ModelEMA = None
            ropt = TorchSgdWithEma(rmodel, ModelEMA)
            try:
                rms, rph, rloss = time_train_steps(rnet, ropt, x, lab, min(args.steps, 10), 2, amp_dtype, world, dev)
                ramp = args.dtype
            except Exception as e:                    # noqa: BLE001 - e.g. an op of the reference without a bf16 kernel
                print(f"# reference train step under autocast({args.dtype}) failed: {e!r}; timing it in fp32", file=sys.stderr)
                rms, rph, rloss = time_train_steps(rnet, ropt, x, lab, min(args.steps, 10), 2, None, world, dev)
                ramp = "fp32"
            ref_line = {"ms_per_step": rms, "images_per_second": world * B / (rms / 1e3), "phases_last_step": rph, "amp": ramp,
                        "loss_last_step": rloss,
                        "what": "unmodified reference YoloxModule.forward(train) (per-image get_assignments loop) + backward + SGD + "
                                "ModelEMA.update, torch eager / cuDNN, same inputs, labels, optimizer and DDP"}
        except Exception as e:                        # noqa: BLE001
            ref_line = {"failed": repr(e)}
    graphed = isinstance(graph_line, dict) and "ms_per_step" in graph_line
    best_ms = graph_line["ms_per_step"] if graphed else ms
    best_e2e_ms = graph_line["e2e_ms_per_step"] if graphed else ms_e2e
    step_mode = ("whole step replayed as a CUDA graph (value, e2e); the op-by-op step is under eager_step" if graphed
                 else "op-by-op (the CUDA-graph capture failed, see cuda_graph_step)")
    if rank == 0:
        pk = peaks()
        A = sum(h * w for h, w in hw)
        sim_bytes = B * A * 85 * 4
        cpu = None
        from pixeltable_yolox_b200.network_blocks import BaseConv as _BaseConv

        n_bn = sum(isinstance(m_, _BaseConv) for m_ in model.modules())
        n_conv = sum(isinstance(m_, torch.nn.Conv2d) and m_.groups == 1 for m_ in model.modules())
        ours_convs = amp_dtype is not None and os.environ.get("YX_TRAIN_CONV", "1") != "0"
        launches_per_step = n_bn * 6 + 6 + 3 + ((4 * n_conv - 1) + 1 + 2 if ours_convs else 0)
        launches_note = (f"ours per step: {n_bn} BaseConv x (3 BatchNorm + activation forward + 3 backward launches) + 6 head-row launches "
                         "+ SimOTA + losses + SGD/EMA" +
                         (f" + {n_conv} convs x (forward, dgrad, wgrad, wgrad reduce; no dgrad for the stem) + 1 weight-packing launch + "
                          "SPP pools forward / backward" if ours_convs else "; the convolutions themselves are cuDNN (YX_TRAIN_CONV=0)"))
        train_tflops = 3 * GFLOP_PER_IMAGE.get(args.model, 0) * 1e9 * B / (best_ms / 1e3) / 1e12
        line = {
            "metric": "images_per_second", "value": world * B / (best_ms / 1e3), "unit": "images/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": best_ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": args.dtype, "data": "synthetic",
            "config": {"workload": workload_name(args), "per_gpu_batch": B, "global_batch": B * world,
                       "labels": f"[{B}, 120, 5] per rank, GT counts on rank 0 {counts}", "amp": args.dtype,
                       "memory_format": args.train_format,
                       "optimizer": "SGD momentum 0.9 nesterov, wd 5e-4 on conv weights (yolox/config.py:307-333) + ModelEMA update "
                                    "(yolox/utils/ema.py:46-58), both arms; ours: one fused launch (yx_sgd_ema_step)",
                       "network_fwd_bwd": ("convolutions: torch autograd / cuDNN (YX_TRAIN_CONV=0)" if os.environ.get("YX_TRAIN_CONV", "1") == "0" or amp_dtype is None
                                           else "convolutions: ours -- forward and dgrad through the tcgen05 implicit-GEMM conv kernel with "
                                                "per-step packed weights, wgrad through the MN-major tcgen05 kernel (yx_conv_wgrad); no cuDNN "
                                                "call in the step") + "; BatchNorm + activation forward / backward, SPP pools: ours",
                       "ours_in_step": "yx_conv_bn_act_fwd (forward + dgrad), yx_conv_wgrad, yx_pack_train_weights, yx_bn_act_train_fwd/bwd (training-mode BatchNorm + SiLU of all 74 BaseConv), yx_head_train_decode "
                                       "fwd/bwd (3 levels), yx_simota_assign (whole batch, one cluster launch, no host sync), "
                                       "yx_head_losses (losses and d/d(pred) in one pass), yx_sgd_ema_step",
                       "collective": ("none (one rank)" if world == 1 else
                                      (f"graph step (value): yx_allreduce_sgd_ema_step, our all-reduce over NVLink 5 / NVSwitch peer memory fused with "
                                       f"SGD + EMA, {n_grad * 4 / 1e6:.1f} MB fp32 per step, no NCCL call; " if getattr(time_train_graph, "fused_collective", False)
                                       else f"graph step (value): one eager ncclAllReduce of the flat {n_grad * 4 / 1e6:.1f} MB fp32 gradient buffer between two graphs; ") +
                                      "eager step: torch DDP buckets (25 MB) -> ncclAllReduce over NVLink/NVSwitch"),
                       "loss_last_step": loss},
            "e2e": {"value": world * B / (best_e2e_ms / 1e3), "unit": "images/s",
                    "h2d_bytes_per_step": xh.numel() * 4 + labh.numel() * 4, "d2h_bytes_per_step": 4,
                    "input": "pinned host fp32 images + labels uploaded every step, loss read back every step", "loss_last_step": loss_e2e},
            "gpu_launches": launches_per_step * args.steps, "launches_per_step": launches_per_step,
            "launches_note": launches_note,
            "step_mode": step_mode,
            "eager_step": {"ms_per_step": ms, "images_per_second": world * B / (ms / 1e3), "e2e_ms_per_step": ms_e2e,
                           "phases_last_step": phases,
                           "what": "the same step launched op by op from Python (torch autograd + our kernels through ctypes)"},
            "cuda_graph_step": graph_line,
            "kernels": {"simota_assign_us": t_simota, "simota_GBps_of_prediction_tensor": sim_bytes / t_simota / 1e3,
                        "head_losses_us": t_loss, "head_losses_GBps": 2 * sim_bytes / t_loss / 1e3,
                        "allreduce_us_standalone": t_ar, "allreduce_share_of_step": (t_ar / 1e3 / ms) if t_ar else None,
                        "allreduce_busbw_GBps": (2 * (world - 1) / world * n_grad * 4 / t_ar / 1e3) if t_ar else None},
            "roofline": {"bound": "tensor", "kernel": "conv family of the training step (conv_tc_kernel forward + dgrad, wgrad_tc_kernel), "
                                                      "timed as the WHOLE step: at 8 images per GPU every layer is a fraction of a wave, "
                                                      "the step is launch- and latency-bound (DESIGN 4.8 has the per-kernel figures: wgrad "
                                                      "128->128 3x3 @80x80 541 TFLOP/s at 8 images, 795 at 64)",
                         "achieved": train_tflops, "peak": pk["tf_sustained"], "unit": "TFLOP/s",
                         "frac": train_tflops / pk["tf_sustained"], "traffic": None,
                         "algorithmic_flops_per_image": 3 * GFLOP_PER_IMAGE.get(args.model, 0) * 1e9,
                         "peak_source": pk["source"] + " bf16 sustained"},
            "hbm_kernel": {"kernel": "head_loss_kernel (losses + gradients)", "achieved_GBps": 2 * sim_bytes / t_loss / 1e3,
                           "frac_of_hbm_peak": 2 * sim_bytes / t_loss / 1e3 / pk["hbm"]},
            "reference_same_box": ref_line, "cpu_baseline": cpu, "clocks": clk,
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def run_reference_train(args, threads):
    """--impl reference --train: the unmodified reference's training step on the host cores (fp32), bounded."""
    import torch

    ref = reference_modules()
    if ref is None:
        print(json.dumps({"impl": "reference", "unavailable": "baseline/_ref missing (python baseline/install_ref.py)"}), flush=True)
        return
    _, model = build_model(args, torch.device("cpu"))
    sd = {k: v.detach().clone() for k, v in model.state_dict().items()}
    rmodel = reference_model(ref, args.model, sd, torch.device("cpu")).train()
    opt = sgd_for(rmodel)
    B = min(args.train_batch, 4)
    x, lab, _ = train_batch(args, 0, B)

    def step():
        out = rmodel(x, lab)
        opt.zero_grad(set_to_none=True)
        out["total_loss"].backward()
        opt.step()

    step()
    steps = max(1, min(args.steps, 3))
    t0 = time.perf_counter()
    for _ in range(steps):
        step()
    dt = time.perf_counter() - t0
    value = B * steps / dt
    line = {"metric": "images_per_second", "impl": "reference", "value": value, "unit": "images/s", "n_gpus": args.gpus,
            "steps": steps, "warmup": 1, "ms_per_step": 1e3 * dt / steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": workload_name(args), "per_gpu_batch": args.train_batch,
                       "reference_arm": f"host CPU fp32, {B} images per step"},
            "cpu_baseline": {"value": value, "unit": "images/s", "cores": threads, "kind": "reference",
                             "sample": f"{steps} steps x {B} images, unmodified reference training step (baseline/_ref), CPU fp32"},
            "e2e": {"value": value, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


def main():
    args = parse()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
