"""-m gpu: each sm_100a kernel through the C-ABI against a torch fp32 restatement of the same op
(floating-point kernels; tolerance written per test)."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

from pixeltable_yolox_b200 import _lib, ops  # noqa: E402
from pixeltable_yolox_b200.ops import View  # noqa: E402


@pytest.fixture(autouse=True)
def _no_tf32():
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False


def _conv_case(dev, B, H, W, cin, cout, k, s, dtype, res, ups, in_off, out_off, act, simt, seed=0):
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(B, H, W, cin + 2 * in_off, generator=g).to(dev).to(dtype)
    w = (torch.randn(cout, k * k, cin, generator=g) / (k * k * cin) ** 0.5).to(dev).to(dtype)
    bias = torch.randn(cout, generator=g).to(dev)
    pad = (k - 1) // 2
    oh, ow = (H + 2 * pad - k) // s + 1, (W + 2 * pad - k) // s + 1
    xin = View(x, in_off, cin)
    o = torch.full((B, oh, ow, cout + 2 * out_off), 7.0, device=dev, dtype=dtype)
    ov = View(o, out_off, cout)
    r = torch.randn(B, oh, ow, cout, generator=g).to(dev).to(dtype) if res else None
    u = torch.full((B, 2 * oh, 2 * ow, cout), 7.0, device=dev, dtype=dtype) if ups else None
    ops.conv_bn_act(xin, w, bias, ov, k, s, _lib.ACT_CODES[act], res=View(r) if res else None,
                    ups=View(u) if ups else None, simt=simt)
    y = F.conv2d(xin.torch().float().permute(0, 3, 1, 2), w.float().reshape(cout, k, k, cin).permute(0, 3, 1, 2),
                 bias, s, pad)
    y = {"silu": F.silu, "relu": F.relu, "lrelu": lambda t: F.leaky_relu(t, 0.1), None: lambda t: t}[act](y)
    if res:
        y = y + r.float().permute(0, 3, 1, 2)
    y = y.permute(0, 2, 3, 1)
    got = ov.torch().float()
    err = ((got - y).abs() / y.abs().clamp_min(1.0)).max().item()
    if out_off:
        assert (o[..., :out_off] == 7).all() and (o[..., out_off + cout:] == 7).all(), "wrote outside the channel slice"
    if ups:
        for dy in (0, 1):
            for dx in (0, 1):
                assert torch.equal(u[:, dy::2, dx::2], ov.torch()), "2x nearest upsample copy differs"
    return err


TC_CASES = [
    # B, H, W, cin, cout, k, s
    (2, 16, 16, 64, 64, 1, 1), (1, 20, 12, 128, 128, 1, 1), (2, 16, 16, 32, 32, 1, 1), (2, 16, 16, 16, 16, 1, 1),
    (2, 16, 16, 256, 256, 1, 1), (2, 16, 16, 512, 96, 1, 1), (2, 8, 8, 128, 512, 1, 1), (1, 7, 9, 48, 80, 1, 1),
    (2, 16, 16, 64, 64, 3, 1), (2, 20, 20, 128, 128, 3, 1), (1, 40, 40, 128, 128, 3, 1), (1, 80, 80, 32, 64, 3, 1),
    (2, 24, 40, 16, 32, 3, 1), (1, 13, 13, 96, 96, 3, 1), (1, 5, 3, 64, 32, 3, 1),
    (2, 16, 16, 64, 64, 3, 2), (2, 40, 40, 32, 64, 3, 2), (1, 80, 80, 128, 128, 3, 2), (2, 20, 20, 256, 512, 3, 2),
    (1, 64, 48, 16, 32, 3, 2), (1, 26, 26, 48, 96, 3, 2),
]


@pytest.mark.parametrize("case", TC_CASES)
@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float16])
def test_conv_tcgen05_vs_torch(cuda, case, dtype):
    tol = 1e-2 if dtype == torch.bfloat16 else 2e-3      # one rounding of the 16-bit output (+ tanh.approx SiLU)
    err = _conv_case(cuda, *case, dtype, False, False, 0, 0, "silu", simt=False)
    assert err <= tol, err


@pytest.mark.parametrize("k,s", [(1, 1), (3, 1), (3, 2)])
def test_conv_tcgen05_fusions(cuda, k, s):
    """residual add, 2x-upsample second store and channel-sliced in/out buffers."""
    for act in ("silu", "relu", "lrelu", None):
        err = _conv_case(cuda, 2, 16, 24, 64, 64, k, s, torch.bfloat16, True, True, 32, 16, act, simt=False)
        assert err <= 1.5e-2, (act, err)


@pytest.mark.parametrize("k", [1, 3])
def test_conv_two_destinations(cuda, k):
    """yx_conv_desc.out2: the trailing output channels of one GEMM land in a second buffer (stacked CSP conv1|conv2)."""
    g = torch.Generator().manual_seed(3)
    B, H, W, cin, c1, c2 = 2, 20, 24, 64, 32, 48
    x = torch.randn(B, H, W, cin, generator=g).to(cuda).to(torch.bfloat16)
    w = (torch.randn(c1 + c2, k * k, cin, generator=g) / (k * k * cin) ** 0.5).to(cuda).to(torch.bfloat16)
    bias = torch.randn(c1 + c2, generator=g).to(cuda)
    whole = torch.empty(B, H, W, c1 + c2, device=cuda, dtype=torch.bfloat16)
    ops.conv_bn_act(View(x), w, bias, View(whole), k, 1, 1)
    o1 = torch.full((B, H, W, c1), 7.0, device=cuda, dtype=torch.bfloat16)
    o2 = torch.full((B, H, W, 16 + c2), 7.0, device=cuda, dtype=torch.bfloat16)
    ops.conv_bn_act(View(x), w, bias, View(o1), k, 1, 1, out2=View(o2, 16, c2), out2_begin=c1)
    assert torch.equal(o1, whole[..., :c1]) and torch.equal(o2[..., 16:], whole[..., c1:])
    assert (o2[..., :16] == 7).all()


def _bneck_run(dev, B, H, W, c, dtype, use_add, act, in_off=0, out_off=0, seed=0):
    """Fused Bottleneck and its torch reference: fp32 math with the hidden tensor rounded to the 16-bit dtype, exactly
    what the reference's two 16-bit BaseConvs do (network_blocks.py:77-99). Returns (kernel output as fp32, reference,
    the whole output buffer, the kernel's inputs)."""
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(B, H, W, c + 2 * in_off, generator=g).to(dev).to(dtype)
    w1 = (torch.randn(c, 1, c, generator=g) / c ** 0.5).to(dev).to(dtype)
    w2 = (torch.randn(c, 9, c, generator=g) / (9 * c) ** 0.5).to(dev).to(dtype)
    b1 = torch.randn(c, generator=g).to(dev)
    b2 = torch.randn(c, generator=g).to(dev)
    o = torch.full((B, H, W, c + 2 * out_off), 7.0, device=dev, dtype=dtype)
    xin, ov = View(x, in_off, c), View(o, out_off, c)
    ops.bottleneck_fwd(xin, w1, b1, w2, b2, ov, _lib.ACT_CODES[act], use_add)
    f = {"silu": F.silu, "relu": F.relu, "lrelu": lambda t: F.leaky_relu(t, 0.1)}[act]
    xf = xin.torch().float().permute(0, 3, 1, 2)
    h = f(F.conv2d(xf, w1.float().reshape(c, 1, 1, c).permute(0, 3, 1, 2), b1)).to(dtype).float()
    y = f(F.conv2d(h, w2.float().reshape(c, 3, 3, c).permute(0, 3, 1, 2), b2, 1, 1))
    if use_add:
        y = y + xf
    return ov.torch().float(), y.permute(0, 2, 3, 1), o, (xin, w1, b1, w2, b2)


def _bneck_case(dev, B, H, W, c, dtype, use_add, act, in_off=0, out_off=0, seed=0):
    got, y, o, _ = _bneck_run(dev, B, H, W, c, dtype, use_add, act, in_off, out_off, seed)
    if out_off:
        assert (o[..., :out_off] == 7).all() and (o[..., out_off + c:] == 7).all(), "wrote outside the channel slice"
    return ((got - y).abs() / y.abs().clamp_min(1.0)).max().item()


BNECK_CASES = [(2, 16, 16, 64), (1, 80, 80, 64), (3, 40, 40, 32), (1, 160, 160, 32), (2, 13, 21, 16), (1, 5, 3, 64),
               (5, 23, 61, 32), (2, 80, 80, 16)]
# c = 128 has no fused kernel (a streamed-weight version measured slower than the unfused pair: DESIGN 4.6)
C128_CASES = [(2, 40, 40, 128), (1, 13, 21, 128), (9, 20, 20, 128), (1, 3, 5, 128)]


@pytest.mark.parametrize("case", BNECK_CASES)
@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float16])
def test_fused_bottleneck_vs_torch(cuda, case, dtype):
    # tolerance: one 16-bit rounding of the output plus hidden values that round differently at a tie
    # (tanh.approx SiLU vs torch's exp form) propagated through the 3x3 conv
    tol = 2e-2 if dtype == torch.bfloat16 else 4e-3
    for use_add in (True, False):
        err = _bneck_case(cuda, *case, dtype, use_add, "silu")
        assert err <= tol, (use_add, err)


@pytest.mark.parametrize("case", C128_CASES)
def test_fused_bottleneck_rejects_c128(cuda, case):
    with pytest.raises(RuntimeError, match="16, 32 or 64"):
        _bneck_case(cuda, *case, torch.bfloat16, True, "silu")


def test_fused_bottleneck_slices_and_acts(cuda):
    for act in ("silu", "relu", "lrelu"):
        err = _bneck_case(cuda, 2, 24, 40, 32, torch.bfloat16, True, act, in_off=32, out_off=16)
        assert err <= 2e-2, (act, err)


def test_fused_bottleneck_rejects_in_place(cuda):
    x = torch.zeros(1, 8, 8, 64, device=cuda, dtype=torch.bfloat16)
    w1 = torch.zeros(64, 1, 64, device=cuda, dtype=torch.bfloat16)
    w2 = torch.zeros(64, 9, 64, device=cuda, dtype=torch.bfloat16)
    b = torch.zeros(64, device=cuda)
    with pytest.raises(RuntimeError, match="alias"):
        ops.bottleneck_fwd(View(x), w1, b, w2, b, View(x), 1, True)


@pytest.mark.parametrize("case", TC_CASES[::3])
def test_conv_simt_fp32_vs_torch(cuda, case):
    err = _conv_case(cuda, *case, torch.float32, True, True, 16, 16, "silu", simt=True)
    assert err <= 2e-5, err          # fp32 FFMA in a different summation order only


def test_conv_tc_and_simt_agree_bitwise_up_to_rounding(cuda):
    e1 = _conv_case(cuda, 2, 20, 20, 128, 128, 3, 1, torch.bfloat16, False, False, 0, 0, None, simt=False)
    e2 = _conv_case(cuda, 2, 20, 20, 128, 128, 3, 1, torch.bfloat16, False, False, 0, 0, None, simt=True)
    assert abs(e1 - e2) < 1e-3


def test_conv_rejects_bad_arguments(cuda):
    x = torch.zeros(1, 8, 8, 24, device=cuda, dtype=torch.bfloat16)
    w = torch.zeros(16, 1, 24, device=cuda, dtype=torch.bfloat16)
    with pytest.raises(RuntimeError, match="multiple of 16"):
        ops.conv_bn_act(View(x), w, torch.zeros(16, device=cuda), View(torch.zeros(1, 8, 8, 16, device=cuda, dtype=torch.bfloat16)), 1, 1, 1)


@pytest.mark.parametrize("img_dtype", [torch.float32, torch.uint8])
@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float32])
def test_focus_space_to_depth(cuda, img_dtype, dtype):
    g = torch.Generator().manual_seed(1)
    img = torch.randint(0, 256, (2, 3, 32, 48), generator=g).to(img_dtype).to(cuda)
    out = torch.full((2, 16, 24, 16), 9.0, device=cuda, dtype=dtype)
    ops.focus_s2d(img, View(out))
    x = img.float()
    want = torch.cat((x[..., ::2, ::2], x[..., 1::2, ::2], x[..., ::2, 1::2], x[..., 1::2, 1::2]), 1).permute(0, 2, 3, 1)
    assert torch.equal(out[..., :12].float(), want)       # 0..255 integers are exact in bf16
    assert (out[..., 12:] == 0).all()


@pytest.mark.parametrize("img_dtype", [torch.float32, torch.uint8])
@pytest.mark.parametrize("dtype,cout", [(torch.bfloat16, 32), (torch.float16, 64), (torch.bfloat16, 24), (torch.bfloat16, 80)])
def test_fused_focus_stem_matches_focus_then_conv(cuda, img_dtype, dtype, cout):
    """The single-kernel Focus + 3x3 conv + BN + SiLU against the reference composition in torch fp32."""
    from pixeltable_yolox_b200.engine import Builder
    from pixeltable_yolox_b200.network_blocks import Focus

    torch.manual_seed(cout)
    blk = Focus(3, cout, ksize=3)
    bn = blk.conv.bn
    bn.eps = 1e-3
    bn.running_mean.normal_(0, 20.0); bn.running_var.uniform_(500.0, 4000.0)
    bn.weight.data.uniform_(0.5, 1.5); bn.bias.data.normal_(0, 0.2)
    blk.eval()
    g = torch.Generator().manual_seed(3)
    img = torch.randint(0, 256, (3, 3, 96, 160), generator=g).float()
    with torch.no_grad():
        want = blk._train_forward(img)                                       # [B, cout, 48, 80]
    blk = blk.to(cuda).to(dtype)
    b = Builder(cuda, dtype, use_plan=False)
    got = blk.lower_image(b, img.to(img_dtype).to(cuda).contiguous()).to_nchw().float().cpu()
    assert got.shape == want.shape
    # the stem sums 108 products of 0..255 pixels with 16-bit weights: compare relative to the pre-activation scale
    err = (got - want).abs() / want.abs().clamp_min(1.0)
    tol = 4e-2 if dtype == torch.bfloat16 else 6e-3
    assert err.max().item() <= tol, err.max().item()
    assert err.mean().item() <= tol / 8


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float16, torch.float32])
def test_spp_cascade_equals_maxpool_5_9_13(cuda, dtype):
    g = torch.Generator().manual_seed(2)
    c = 32
    buf = torch.zeros(2, 20, 13, 4 * c, device=cuda, dtype=dtype)
    buf[..., :c] = torch.randn(2, 20, 13, c, generator=g).to(cuda).to(dtype)
    ops.spp_maxpool(View(buf), c)
    x = buf[..., :c].float().permute(0, 3, 1, 2)
    for i, k in enumerate((5, 9, 13)):
        want = F.max_pool2d(x, k, 1, k // 2).permute(0, 2, 3, 1)
        assert torch.equal(buf[..., (i + 1) * c:(i + 2) * c].float(), want), k      # max is exact


@pytest.mark.parametrize("stride", [1, 2])
@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float32])
def test_depthwise_conv(cuda, stride, dtype):
    g = torch.Generator().manual_seed(3)
    c = 32
    x = torch.randn(2, 17, 22, c, generator=g).to(cuda).to(dtype)
    w = torch.randn(9, c, generator=g).to(cuda).to(dtype)
    bias = torch.randn(c, generator=g).to(cuda)
    oh, ow = (17 + 2 - 3) // stride + 1, (22 + 2 - 3) // stride + 1
    out = torch.empty(2, oh, ow, c, device=cuda, dtype=dtype)
    ops.dwconv3x3(View(x), w, bias, View(out), stride, _lib.YX_ACT_SILU)
    wt = w.float().t().reshape(c, 1, 3, 3)
    want = F.silu(F.conv2d(x.float().permute(0, 3, 1, 2), wt, bias, stride, 1, 1, c)).permute(0, 2, 3, 1)
    err = ((out.float() - want).abs() / want.abs().clamp_min(1.0)).max().item()
    assert err <= (1e-2 if dtype == torch.bfloat16 else 1e-5), err


def test_pack_weights_folds_bn_like_fuse_conv_and_bn(cuda):
    """utils/model_utils.py:33-75."""
    g = torch.Generator().manual_seed(4)
    o, i, k = 24, 20, 3
    w = torch.randn(o, i, k, k, generator=g)
    gamma, beta = torch.rand(o, generator=g) + 0.5, torch.randn(o, generator=g)
    mean, var = torch.randn(o, generator=g), torch.rand(o, generator=g) + 0.1
    eps = 1e-3
    dst = torch.zeros(32, 9, 32, device=cuda)
    bias = torch.zeros(32, device=cuda)
    ops.pack_weights(w, (gamma, beta, mean, var), None, eps, dst, bias, o_off=4, i_off=8)
    scale = gamma / torch.sqrt(var + eps)
    want_w = (w * scale[:, None, None, None]).permute(0, 2, 3, 1).reshape(o, 9, i)
    torch.testing.assert_close(dst[4:4 + o, :, 8:8 + i].cpu(), want_w, rtol=1e-6, atol=1e-6)
    torch.testing.assert_close(bias[4:4 + o].cpu(), beta - mean * scale, rtol=1e-6, atol=1e-6)
    assert dst[:4].abs().sum() == 0 and dst[:, :, :8].abs().sum() == 0


def test_head_decode_matches_decode_outputs(cuda):
    from oracle import yolox_oracle as yo

    g = torch.Generator().manual_seed(5)
    hw = [(8, 12), (4, 6), (2, 3)]
    A = sum(h * w for h, w in hw)
    raw = torch.randn(2, A, 85, generator=g)
    want = yo.decode_outputs(raw, hw, (8, 16, 32))
    got = ops.head_decode_(raw.to(cuda).clone(), hw, (8, 16, 32)).cpu()
    torch.testing.assert_close(got, want, rtol=1e-6, atol=1e-5)


def test_bboxes_iou_bit_exact(cuda, golden_simota):
    import pixeltable_yolox_b200 as yx

    a, b = torch.from_numpy(golden_simota["iou/a"]).to(cuda), torch.from_numpy(golden_simota["iou/b"]).to(cuda)
    assert np.array_equal(yx.bboxes_iou(a, b, True).cpu().numpy(), golden_simota["iou/xyxy"])
    assert np.array_equal(yx.bboxes_iou(a, b, False).cpu().numpy(), golden_simota["iou/cxcywh"])


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float16])
@pytest.mark.parametrize("thr", [0.5, 0.05])
def test_head_epilogue_fused_score_filter_is_bit_exact(cuda, dtype, thr):
    """Prediction GEMM with the score filter fused into the decode epilogue (yx_conv_desc.head_cand) followed by
    yx_nms_prefiltered == the same GEMM followed by the stand-alone yx_postprocess (filter kernel + NMS), bit for bit:
    detections, kept anchor indices, counts and the in-place corner conversion (boxes.py:31-75). Three levels with
    different strides write one [B, A, 5+nc] tensor; 20x20 and 10x10 make warps straddle image boundaries."""
    g = torch.Generator().manual_seed(11)
    B, nc, c = 3, 80, 64
    levels = [(40, 8.0), (20, 16.0), (10, 32.0)]
    A = sum(hw * hw for hw, _ in levels)
    xs = [(torch.randn(B, hw, hw, c, generator=g) * 0.5).to(cuda).to(dtype) for hw, _ in levels]
    ws_ = [(torch.randn(96, 1, c, generator=g) / c ** 0.5).to(cuda).to(dtype) for _ in levels]
    bs = [torch.cat([torch.randn(4, generator=g) * 0.3, torch.randn(92, generator=g) - 1.0]).to(cuda) for _ in levels]

    def run(post):
        out = torch.zeros(B, A, 5 + nc, device=cuda)
        off = 0
        for (hw, stride), x, w, bias in zip(levels, xs, ws_, bs):
            head = {"out_ptr": out.data_ptr(), "anchors": A, "anchor_off": off, "nc": nc, "decode": 3, "stride": stride}
            head.update(post)
            ops.conv_bn_act(View(x), w, bias, None, 1, 1, 0, head=head)
            off += hw * hw
        return out

    ref_pred = run({})
    plain = ref_pred.clone()
    d0, i0, n0 = ops.postprocess_device(ref_pred, nc, thr, 0.65, 0, inplace_xyxy=True)

    ws = torch.empty(_lib.lib().yx_postprocess_workspace_bytes(B, A), dtype=torch.uint8, device=cuda)
    cand, keys, counts = ops.postprocess_ws_ptrs(ws, B, A)
    ops.postprocess_begin(ws, B, A)
    fused_pred = run({"cand_ptr": cand, "keys_ptr": keys, "counts_ptr": counts, "conf_thre": thr, "xyxy": True})
    d1, i1, n1 = ops.nms_prefiltered(ws, B, A, 0.65, 0)
    torch.cuda.synchronize()
    assert int(n0.sum()) > 0 and torch.equal(n0, n1)
    assert torch.equal(fused_pred, ref_pred)                       # corners in place, obj / cls untouched
    assert torch.equal(fused_pred[..., 4:], plain[..., 4:])
    for b in range(B):
        k = int(n0[b])
        assert torch.equal(d0[b, :k], d1[b, :k]) and torch.equal(i0[b, :k], i1[b, :k])
