"""-m gpu: the whole drop-in path (YoloxModule.forward / detect / training step) against the
reference goldens and the oracle."""
import numpy as np
import pytest
import torch

import cases

pytestmark = pytest.mark.gpu

import pixeltable_yolox_b200 as yx  # noqa: E402
from oracle import postprocess_oracle as po  # noqa: E402
from oracle import yolox_oracle as yo  # noqa: E402
from pixeltable_yolox_b200 import synthetic as syn  # noqa: E402


def _build(name):
    c = cases.NET_CASES[name]
    cfg = yx.YoloxConfig(name, depth=c["depth"], width=c["width"], depthwise=c["depthwise"])
    model = cfg.get_model()
    x = torch.from_numpy(syn.images(c["batch"], c["h"], c["w"], seed=c["seed"] + 500))
    sd = yo.seeded_state_dict(model.state_dict(), c["seed"], (c["h"], c["w"]), calib_x=x)
    model.load_state_dict(sd)
    return model, sd, x


def _rel(a, b):
    return np.abs(a - b) / np.maximum(np.abs(b), 1.0)


@pytest.mark.parametrize("name", list(cases.NET_CASES))
def test_fp32_forward_within_1e3_of_reference(cuda, name, golden_net):
    """north_star gate: fp32 head outputs within 1e-3 relative of the reference."""
    model, sd, x = _build(name)
    model = model.to(cuda).eval()
    out = model(x.to(cuda)).cpu().numpy()
    ref = golden_net[f"{name}/out"]
    assert out.shape == ref.shape
    err = _rel(out, ref).max()
    # conditioning ceiling: the same fp32 graph in plain torch on this GPU vs the CPU reference
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    ceil = _rel(yo.forward({k: v.to(cuda) for k, v in sd.items()}, x.to(cuda)).cpu().numpy(), ref).max()
    assert err <= 1e-3 or err <= 1.5 * ceil, (err, ceil)     # the depthwise seeded net is ill-conditioned in fp32 itself
    if name != "w25_d33_dw_96":
        assert err <= 1e-3, err
    model.head.decode_in_inference = False
    model.invalidate_engine()
    und = model(x.to(cuda)).cpu().numpy()
    assert _rel(und, golden_net[f"{name}/undecoded"]).max() <= 1e-3


def _torch_native(sd, x, dtype, dev):
    """The reference's own way to run in 16 bit (model.half()/.bfloat16()): plain torch arithmetic."""
    sdd = {k: (v.to(dev).to(dtype) if v.is_floating_point() else v.to(dev)) for k, v in sd.items()}
    a = yo.ACTS["silu"]
    with torch.no_grad():
        o, _ = yo.head(sdd, yo.pafpn(sdd, x.to(dev).to(dtype), a), a)
    return o.float().cpu().numpy()


@pytest.mark.parametrize("name", ["w25_d33_64", "w50_d33_96x128", "w25_d33_dw_96", "w375_d33_64"])
@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float16])
def test_16bit_tcgen05_forward_tracks_reference(cuda, name, dtype, golden_net):
    """16-bit storage perturbs random-weight networks chaotically for the reference too (SURVEY 8c'):
    the gate is relative to the ceiling set by torch's native arithmetic in the same dtype."""
    model, sd, x = _build(name)
    ref = golden_net[f"{name}/out"]
    theirs = _torch_native(sd, x, dtype, cuda)
    model = model.to(cuda).to(dtype).eval()
    out = model(x.to(cuda)).float().cpu().numpy()
    assert np.isfinite(out).all()
    for sl, label in ((slice(0, 4), "boxes"), (slice(4, None), "probabilities")):
        mine = _rel(out[..., sl], ref[..., sl])
        base = _rel(theirs[..., sl], ref[..., sl])
        assert np.median(mine) <= 1.5 * np.median(base) + 1e-3, (label, np.median(mine), np.median(base))
        assert np.quantile(mine, 0.99) <= 2.5 * np.quantile(base, 0.99) + 5e-3, (label, np.quantile(mine, 0.99), np.quantile(base, 0.99))


def test_micro_batching_and_graph_replay_are_deterministic(cuda):
    model, sd, x = _build("w25_d33_64")
    x = torch.cat([x, x.flip(0), x], 0)                # batch 6
    model = model.to(cuda).bfloat16().eval()
    model.micro_batch = 6
    a = model(x.to(cuda))
    model.micro_batch = 4                               # 4 + ragged 2
    model.invalidate_engine()
    b = model(x.to(cuda))
    c = model(x.to(cuda))                               # second call replays the captured graph
    assert torch.equal(a, b) and torch.equal(b, c)
    model.use_cuda_graph = False
    model.invalidate_engine()
    assert torch.equal(model(x.to(cuda)), a)
    assert torch.equal(model(x.to(cuda).to(torch.uint8)), a)     # uint8 image input is the same pixels


def test_detect_equals_forward_plus_postprocess(cuda):
    model, sd, x = _build("w50_d33_96x128")
    model = model.to(cuda).eval()                       # fp32 path: candidates identical to the oracle's forward
    pred = model(x.to(cuda))
    want = yx.postprocess(pred.clone(), 80, 0.05, 0.65, nms_variant="offset")
    dets, idx, cnt = model.detect(x.to(cuda), conf_thre=0.05, nms_thre=0.65, nms_variant="offset")
    for b, w in enumerate(want):
        n = int(cnt[b])
        assert (w is None and n == 0) or (w is not None and torch.equal(dets[b, :n], w))
    ref, _ = po.postprocess(pred.cpu().numpy().copy(), 80, 0.05, 0.65, variant="offset", return_indices=True)
    for w, r in zip(want, ref):
        assert (w is None) == (r is None)
        if w is not None:
            np.testing.assert_array_equal(w.cpu().numpy(), r)


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float16])
@pytest.mark.parametrize("name,micro_batch", [("w50_d33_96x128", None), ("w375_d33_64", 1), ("w25_d33_64", 1)])
def test_detect_with_fused_filter_equals_forward_plus_postprocess(cuda, dtype, name, micro_batch):
    """16-bit paths: detect() runs the score filter inside the head's decode epilogue (+ sort/NMS kernel); the result
    must equal forward() followed by the stand-alone postprocess bit for bit, also when the batch is walked in slices
    (two images, one per slice: the candidate / key / counter pointers of the second slice are offset)."""
    model, sd, x = _build(name)
    model = model.to(cuda).to(dtype).eval()
    model.micro_batch = micro_batch
    pred = model(x.to(cuda))
    for thr in (0.05, 0.3):
        want = yx.postprocess(pred.clone(), 80, thr, 0.65, nms_variant="offset")
        dets, idx, cnt = model.detect(x.to(cuda), conf_thre=thr, nms_thre=0.65, nms_variant="offset")
        assert thr > 0.05 or int(cnt.sum()) > 0
        for b, w in enumerate(want):
            n = int(cnt[b])
            assert (w is None and n == 0) or (w is not None and torch.equal(dets[b, :n], w))


def test_block_level_forward_matches_torch(cuda):
    """BaseConv / CspLayer / SPPBottleneck / Focus called on their own (NCHW in, NCHW out)."""
    from pixeltable_yolox_b200.network_blocks import BaseConv, CspLayer, Focus, SPPBottleneck

    torch.manual_seed(0)
    for blk, x in ((BaseConv(32, 48, 3, 2), torch.randn(2, 32, 20, 24)), (CspLayer(64, 64, n=2), torch.randn(1, 64, 16, 16)),
                   (SPPBottleneck(64, 64), torch.randn(1, 64, 12, 12)), (Focus(3, 32, 3), torch.rand(2, 3, 32, 32) * 255)):
        for m in blk.modules():
            if isinstance(m, torch.nn.BatchNorm2d):
                m.eps = 1e-3
                m.running_mean.normal_(0, 0.5); m.running_var.uniform_(0.5, 2.0)
                m.weight.data.uniform_(0.5, 1.5); m.bias.data.normal_(0, 0.2)
        blk.eval()
        with torch.no_grad():
            want = blk._train_forward(x)                 # torch ops, eval-mode BN
        got = blk.to(cuda)(x.to(cuda)).cpu()
        assert got.shape == want.shape
        assert (_rel(got.numpy(), want.numpy())).max() <= 1e-4, type(blk).__name__


def test_state_dict_roundtrip_and_reload_invalidates_engine(cuda):
    model, sd, x = _build("w25_d33_64")
    model = model.to(cuda).eval()
    a = model(x.to(cuda))
    sd2 = {k: (v * 1.05 if k.endswith("conv.weight") else v) for k, v in sd.items()}
    model.load_state_dict(sd2)
    b = model(x.to(cuda))
    assert not torch.equal(a, b)
    model.load_state_dict(sd)
    assert torch.equal(model(x.to(cuda)), a)
    assert set(model.state_dict()) == set(sd)


def test_training_step_runs_and_backpropagates(cuda):
    model, sd, x = _build("w25_d33_64")
    model = model.to(cuda).train()
    lab = torch.zeros(x.shape[0], 120, 5)
    lab[0, :3] = torch.tensor([[3.0, 20.0, 24.0, 18.0, 22.0], [7.0, 44.0, 40.0, 30.0, 12.0], [0.0, 32.0, 12.0, 10.0, 10.0]])
    out = model(x.to(cuda), lab.to(cuda))
    assert set(out) == {"total_loss", "iou_loss", "l1_loss", "conf_loss", "cls_loss", "num_fg"}
    assert torch.isfinite(out["total_loss"])
    out["total_loss"].backward()
    g = model.head.cls_preds[0].weight.grad
    assert g is not None and torch.isfinite(g).all() and g.abs().sum() > 0


def test_engine_cache_survives_deepcopy_and_weight_changes(cuda):
    """The engine (native plan + packed weights) belongs to one module object: a deep copy / pickle gets none of it and
    builds its own; any weight change while in eval (sub-module load_state_dict, in-place copy_, initialize_biases) is
    picked up by the parameter fingerprint instead of silently serving the old packed weights."""
    import copy
    import io

    model, sd, x = _build("w25_d33_64")
    model = model.to(cuda).bfloat16().eval()
    xd = x.to(cuda)
    base = model(xd).clone()
    twin = copy.deepcopy(model)
    assert twin._engines == {} and len(model._engines) == 1
    assert torch.equal(twin(xd), base) and torch.equal(model(xd), base)
    with torch.no_grad():                                    # change the twin only
        twin.head.cls_preds[0].bias.add_(1.0)
    changed = twin(xd)
    assert not torch.equal(changed, base) and torch.equal(model(xd), base)
    twin.invalidate_engine()                                 # frees the twin's plan only
    assert torch.equal(model(xd), base)
    buf = io.BytesIO(); torch.save(model, buf); buf.seek(0)
    loaded = torch.load(buf, weights_only=False)
    assert loaded._engines == {} and torch.equal(loaded(xd), base)
    # sub-module load_state_dict and initialize_biases while in eval
    model.head.load_state_dict(twin.head.state_dict())
    assert torch.equal(model(xd), changed)
    model.head.initialize_biases(0.5)
    assert not torch.equal(model(xd), changed)
    with pytest.raises(TypeError):
        copy.deepcopy(next(iter(model._engines.values())))


def test_config1_nano_416_user_api_on_gpu(cuda):
    """BASELINE.json config 1 on the GPU path: yolox_nano (depthwise) 416x416 batch 1, fp32 verification mode within 1e-3 of
    the reference's CPU output (or the conditioning ceiling of the same graph in torch-CUDA fp32), bf16 at the torch-bf16
    ceiling; YoloxProcessor.postprocess on the reference's own head tensor returns the reference's Detections exactly."""
    from pathlib import Path

    from PIL import Image

    g = np.load(Path(__file__).resolve().parent / "golden" / "config1.npz")
    c = cases.CONFIG1
    dev = cuda
    img = Image.fromarray(cases.config1_image())
    proc = yx.YoloxProcessor(c["name"])
    proc.nms_variant = "auto_cpu"                  # the fixture was produced by the reference on CPU (torchvision's CPU rule)
    x = proc([img])
    cfg = yx.YoloxConfig.get_named_config(c["name"])
    cfg.model = None
    model = cfg.get_model()
    sd = yo.seeded_state_dict(model.state_dict(), c["seed"], tuple(cfg.test_size), calib_x=x)
    model.load_state_dict(sd)
    model = model.to(dev).eval()
    out = model(x.to(dev)).cpu().numpy()
    ref = g["out"]
    err = _rel(out, ref).max()
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    ceil = _rel(yo.forward({k: v.to(dev) for k, v in sd.items()}, x.to(dev)).cpu().numpy(), ref).max()
    assert err <= 1e-3 or err <= 1.5 * ceil, (err, ceil)
    for thr in c["thresholds"]:
        det = proc.postprocess([img], torch.from_numpy(ref.copy()).to(dev), threshold=thr)[0]
        np.testing.assert_array_equal(np.array(det["bboxes"], dtype=np.float64).reshape(-1, 4), g[f"t{thr}/bboxes"])
        np.testing.assert_array_equal(np.array(det["scores"], dtype=np.float64), g[f"t{thr}/scores"])
        np.testing.assert_array_equal(np.array(det["labels"], dtype=np.int64), g[f"t{thr}/labels"])
    # the whole user-facing call: Yolox.__call__ (processor -> fused detect graph -> formatted detections)
    wrapper = yx.Yolox(model, proc)
    res = wrapper([img], threshold=0.6)[0]
    want = proc.postprocess([img], model(x.to(dev)), threshold=0.6)[0]
    assert res["labels"] == want["labels"] and res["scores"] == want["scores"] and res["bboxes"] == want["bboxes"]
    u8 = model(proc([img]).to(torch.uint8).to(dev)).cpu().numpy()
    assert np.array_equal(u8, out)                 # byte upload: bit-identical


def test_module_on_a_non_current_device(cuda):
    """One process may drive several GPUs: a module on cuda:1 while cuda:0 is the current device must launch on cuda:1
    (library caches are per device, every entry point makes the tensors' device current). Needs two GPUs."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    model, sd, x = _build("w25_d33_64")
    d0, d1 = torch.device("cuda", 0), torch.device("cuda", 1)
    torch.cuda.set_device(0)
    m0 = model.to(d0).bfloat16().eval()
    want = m0(x.to(d0)).cpu()
    import copy

    m1 = copy.deepcopy(m0).to(d1)
    assert torch.cuda.current_device() == 0
    got = m1(x.to(d1))
    assert got.device == d1 and torch.equal(got.cpu(), want)
    dets, _, cnt = m1.detect(x.to(d1), conf_thre=0.05)
    dets0, _, cnt0 = m0.detect(x.to(d0), conf_thre=0.05)
    assert torch.equal(cnt.cpu(), cnt0.cpu()) and torch.equal(dets.cpu(), dets0.cpu())
    pred = torch.from_numpy(syn.dense_scene(1, anchors=2100, seed=3, clusters=20, size=320.0))
    a = yx.postprocess(pred.clone().to(d1), 80, 0.25, 0.65)
    b = yx.postprocess(pred.clone().to(d0), 80, 0.25, 0.65)
    assert torch.equal(a[0].cpu(), b[0].cpu())
    with pytest.raises(RuntimeError, match="is on"):
        ops = __import__("pixeltable_yolox_b200.ops", fromlist=["ops"])
        ops.bboxes_iou_device(torch.zeros(2, 4, device=d0), torch.zeros(2, 4, device=d1), True)
