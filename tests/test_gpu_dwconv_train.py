"""-m gpu: the depthwise 3x3 convs of the training step (yolox_nano's DWConv) on csrc/yx_dwconv_train.cu: forward, input
gradient and weight gradient against an fp64 depthwise conv and its autograd gradients evaluated on the same 16-bit-rounded
x, dy and weight, so the comparison isolates the kernels' arithmetic (exact 16-bit products, fp32 sums)."""
import copy

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

import pixeltable_yolox_b200 as yx  # noqa: E402
from pixeltable_yolox_b200 import ops, train_conv  # noqa: E402
from pixeltable_yolox_b200 import synthetic as syn  # noqa: E402

# (c, H, W, stride) of the 30 depthwise convs of yolox_nano at 416x416, in forward order: 18 in the backbone and neck, 12 in
# the head towers
NANO_416 = ([(16, 208, 208, 2), (16, 104, 104, 1), (32, 104, 104, 2)] + [(32, 52, 52, 1)] * 3 + [(64, 52, 52, 2)]
            + [(64, 26, 26, 1)] * 3 + [(128, 26, 26, 2), (128, 13, 13, 1), (64, 26, 26, 1), (32, 52, 52, 1), (64, 52, 52, 2),
                                       (64, 26, 26, 1), (128, 26, 26, 2), (128, 13, 13, 1)]
            + [(64, 52, 52, 1)] * 4 + [(64, 26, 26, 1)] * 4 + [(64, 13, 13, 1)] * 4)
assert len(NANO_416) == 30

# (batch, c, H, W, stride): every distinct nano layer shape at batch 2, then odd maps, a channel count that is a multiple of
# 8 but not of 16, and a large pixel sum for dW (8 x 104 x 104 = 86528 products per element)
SHAPES = ([(2,) + s for s in sorted(set(NANO_416))]
          + [(2, 32, 17, 22, 1), (2, 32, 17, 22, 2), (3, 16, 13, 13, 2), (2, 8, 7, 5, 1), (2, 8, 7, 5, 2), (2, 24, 20, 20, 1),
             (2, 24, 19, 21, 2), (8, 16, 104, 104, 1), (1, 512, 9, 9, 2)])


def _cl(t):
    return t.contiguous(memory_format=torch.channels_last)


def _weights(c, gen, cuda):
    """The same values as NCHW-contiguous, channels_last and a tap-major view (channel stride 1)."""
    w = (torch.randn(c, 1, 3, 3, generator=gen) * 0.4).to(cuda)
    tap_major = w.permute(2, 3, 0, 1).contiguous().permute(2, 3, 0, 1)
    return [w, w.contiguous(memory_format=torch.channels_last), tap_major]


def _ulp(ref, dtype):
    """One unit in the last place of `dtype` at |ref| (fp64 tensor)."""
    mant, tiny = (7, 2.0 ** -133) if dtype == torch.bfloat16 else (10, 2.0 ** -24)
    _, e = torch.frexp(ref)
    return torch.ldexp(torch.ones_like(ref), e - 1 - mant).clamp_min(tiny)


def _within_one_ulp(got, ref, abs_terms, dtype, what):
    # one ulp at the fp64 value, plus the bound of the fp32 rounding of the (at most nine-term) sum before the one 16-bit
    # rounding, 8 * 2^-24 * sum |products|: it only matters where the products cancel
    err = (got.double() - ref).abs()
    bound = _ulp(ref, dtype) + 8 * 2.0 ** -24 * abs_terms
    bad = err > bound
    assert not bool(bad.any()), (what, int(bad.sum()), float((err / bound).max()))


def _inputs(shape, dtype, cuda, seed):
    B, c, H, W, s = shape
    g = torch.Generator().manual_seed(seed)
    OH, OW = (H - 1) // s + 1, (W - 1) // s + 1
    x = _cl((torch.randn(B, c, H, W, generator=g) * 0.7 + 0.1).to(dtype).to(cuda))
    dy = _cl((torch.randn(B, c, OH, OW, generator=g) * 0.5).to(dtype).to(cuda))
    return x, dy, _weights(c, g, cuda)


def _reference(x, dy, w16, s):
    """fp64 y, dx, dW of the depthwise conv on the 16-bit-rounded operands, and the sums of |products| of y and dx."""
    c = x.shape[1]
    x64 = x.double().requires_grad_(True)
    w64 = w16.double().requires_grad_(True)
    y = F.conv2d(x64, w64, stride=s, padding=1, groups=c)
    y.backward(dy.double())
    with torch.no_grad():
        y_abs = F.conv2d(x.double().abs(), w16.double().abs(), stride=s, padding=1, groups=c)
        dx_abs = torch.nn.grad.conv2d_input(x.shape, w16.double().abs(), dy.double().abs(), stride=s, padding=1, groups=c)
    return y.detach(), x64.grad, w64.grad, y_abs, dx_abs


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float16])
@pytest.mark.parametrize("shape", SHAPES)
def test_dwconv_forward_dgrad_wgrad_match_fp64(cuda, shape, dtype):
    B, c, H, W, s = shape
    x, dy, ws = _inputs(shape, dtype, cuda, seed=c * 31 + H * 7 + W + s)
    w16 = ws[0].to(dtype)                          # the weight as the kernels round it (autocast's cast)
    y_ref, dx_ref, dw_ref, y_abs, dx_abs = _reference(x, dy, w16, s)
    for w in ws:
        y = ops.dwconv_train_fwd(x, w, s)
        assert y.dtype == dtype and y.shape == y_ref.shape and y.is_contiguous(memory_format=torch.channels_last)
        _within_one_ulp(y, y_ref, y_abs, dtype, "y")
        dx = ops.dwconv_dgrad(dy, w, s, H, W)
        assert dx.dtype == dtype and dx.shape == x.shape
        _within_one_ulp(dx, dx_ref, dx_abs, dtype, "dx")
        dw = ops.dwconv_wgrad(x, dy, w, s)
        assert dw.dtype == torch.float32 and dw.shape == w.shape and dw.stride() == w.stride()
        err = float((dw.double() - dw_ref).abs().max())
        assert err <= 1e-4 * float(dw_ref.abs().max()), (err, float(dw_ref.abs().max()))


def test_dwconv_wgrad_accumulates_into_an_existing_gradient(cuda):
    x, dy, ws = _inputs((2, 64, 26, 26, 2), torch.bfloat16, cuda, seed=5)
    for w in ws:
        plain = ops.dwconv_wgrad(x, dy, w, 2)
        grad = torch.empty_strided(w.shape, w.stride(), device=cuda).copy_(torch.randn(w.shape, device=cuda))  # a non-zero .grad
        want = grad + plain                              # the kernel's `*d + acc` in fp32: bit-identical
        got = ops.dwconv_wgrad(x, dy, w, 2, accumulate_into=grad)
        assert got is grad and torch.equal(grad, want)


def test_dwconv_backward_is_deterministic(cuda):
    x, dy, ws = _inputs((8, 16, 104, 104, 1), torch.bfloat16, cuda, seed=9)
    conv = torch.nn.Conv2d(16, 16, 3, 1, 1, groups=16, bias=False).to(cuda)
    res = []
    for _ in range(2):
        conv.weight.grad = None
        xi = x.clone().requires_grad_(True)
        y = train_conv.conv2d(xi, conv)
        y.backward(dy)
        res.append((conv.weight.grad.clone(), xi.grad.clone(), ops.dwconv_wgrad(x, dy, ws[0], 1)))
    for a, b in zip(*res):
        assert torch.equal(a, b)


@pytest.mark.parametrize("fmt", [torch.contiguous_format, torch.channels_last])
@pytest.mark.parametrize("stride", [1, 2])
def test_dwconv_module_path_under_autocast(cuda, fmt, stride, monkeypatch):
    """train_conv.conv2d routes a depthwise nn.Conv2d to the kernels under bf16 autocast (fp32 input, any memory format):
    y is channels_last bf16, dx comes back in x's dtype, dW in the parameter's strides, all as the kernels compute them."""
    monkeypatch.setenv("YX_TRAIN_CONV", "1")
    torch.manual_seed(stride)
    conv = torch.nn.Conv2d(32, 32, 3, stride, 1, groups=32, bias=False).to(cuda).to(memory_format=fmt)
    x = torch.randn(2, 32, 21, 18, device=cuda).contiguous(memory_format=fmt).requires_grad_(True)
    assert train_conv.usable(x, conv) is None
    with torch.autocast("cuda", dtype=torch.bfloat16):
        assert train_conv.usable_depthwise(x, conv) == torch.bfloat16
        y = train_conv.conv2d(x, conv)
    assert y.dtype == torch.bfloat16 and y.is_contiguous(memory_format=torch.channels_last)
    go = _cl(torch.randn(y.shape, device=cuda).bfloat16())
    y.backward(go)
    xh = _cl(x.detach().bfloat16())
    assert torch.equal(y, ops.dwconv_train_fwd(xh, conv.weight.detach(), stride))
    assert x.grad.dtype == torch.float32
    assert torch.equal(x.grad, ops.dwconv_dgrad(go, conv.weight.detach(), stride, 21, 18).float())
    assert conv.weight.grad.stride() == conv.weight.stride()
    assert torch.equal(conv.weight.grad, ops.dwconv_wgrad(xh, go, conv.weight, stride))


def test_direct_gradients_of_depthwise_weights(cuda):
    """FusedSgdEma(direct_grads=True): the depthwise weight gradients are added into the flat buffer on the side streams and
    autograd gets none for them (no AccumulateGrad: a hook on the weight never fires)."""
    from pixeltable_yolox_b200.optim import FusedSgdEma

    torch.manual_seed(0)
    m = copy.deepcopy(yx.YoloxConfig.get_named_config("yolox_nano").get_model()).float().to(cuda).train()
    m = m.to(memory_format=torch.channels_last)
    x = _cl(torch.from_numpy(syn.images(2, 128, 128, seed=3)).to(cuda))
    lab = torch.from_numpy(syn.labels(2, max_gt=8, seed=5, size=128.0, counts=[3, 5])).to(cuda)
    dws = [mod.weight for mod in m.modules() if isinstance(mod, torch.nn.Conv2d) and mod.groups > 1]
    assert len(dws) == 30
    sd = {k: v.clone() for k, v in m.state_dict().items()}

    def run():
        m.load_state_dict(sd)
        with torch.autocast("cuda", dtype=torch.bfloat16):
            out = m(x, lab)
        out["total_loss"].backward()
        train_conv.join_wgrad()
        return [w.grad.clone() for w in dws]

    m.zero_grad(set_to_none=True)
    want = run()
    for p in m.parameters():
        p.grad = None
    opt = None
    fired = []
    hooks = [w.register_hook(lambda g: fired.append(g is not None)) for w in dws]     # (called with None when none is returned)
    try:
        opt = FusedSgdEma(m, lr=0.01, ema=False, direct_grads=True)
        opt.zero_grad()
        got = run()
        assert not any(fired)
        lo, hi = opt.flat_grad.data_ptr(), opt.flat_grad.data_ptr() + opt.flat_grad.numel() * 4
        for w, a, b in zip(dws, got, want):
            assert lo <= w.grad.data_ptr() < hi and a.stride() == w.stride()
            # (the SPP pool backward adds with fp32 atomics: the last bits of everything upstream of it vary run to run)
            torch.testing.assert_close(a, b, rtol=1e-3, atol=1e-3 * float(b.abs().max()) + 1e-9)
    finally:
        for h in hooks:
            h.remove()
        if opt is not None:
            opt.close()


@pytest.mark.parametrize("case", ["c12", "bias", "env_off"])
def test_fallbacks_are_the_module_forward_bit_for_bit(cuda, case, monkeypatch):
    monkeypatch.setenv("YX_TRAIN_CONV", "0" if case == "env_off" else "1")
    c = 12 if case == "c12" else 16
    torch.manual_seed(4)
    conv = torch.nn.Conv2d(c, c, 3, 1, 1, groups=c, bias=case == "bias").to(cuda)
    x = torch.randn(2, c, 20, 20, device=cuda)
    with torch.autocast("cuda", dtype=torch.bfloat16):
        assert train_conv.usable_depthwise(x, conv) is None
        got = train_conv.conv2d(x, conv)
        want = conv(x)
    assert got.dtype == want.dtype and torch.equal(got, want)


def test_dwconv_c_abi_rejects_bad_shapes(cuda):
    from pixeltable_yolox_b200._lib import YX_BF16, lib, stream_ptr

    x = torch.zeros(1, 8, 8, 16, dtype=torch.bfloat16, device=cuda)
    w = torch.zeros(16, 1, 3, 3, device=cuda)
    L, sp = lib(), stream_ptr(cuda)
    assert L.yx_dwconv3x3_train_fwd(x.data_ptr(), 16, w.data_ptr(), 9, 1, x.data_ptr(), 16, 1, 8, 8, 12, 1, YX_BF16, sp) < 0
    assert b"multiple of 8" in L.yx_last_error()
    assert L.yx_dwconv3x3_dgrad(x.data_ptr(), 16, w.data_ptr(), 9, 1, x.data_ptr(), 16, 1, 8, 8, 16, 3, YX_BF16, sp) < 0
    assert L.yx_dwconv3x3_wgrad_workspace_bytes(1, 8, 8, 12, 1) < 0
    assert L.yx_dwconv3x3_wgrad(x.data_ptr() + 2, 16, x.data_ptr(), 16, YX_BF16, 1, 8, 8, 16, 1, w.data_ptr(), 9, 1, 0,
                                w.data_ptr(), w.numel() * 4, sp) < 0
    assert b"16-byte aligned" in L.yx_last_error()
    torch.cuda.synchronize()


def _nano_step(m, x, lab):
    with torch.autocast("cuda", dtype=torch.bfloat16):
        out = m(x, lab)
    out["total_loss"].backward()
    return out["total_loss"]


def test_nano_training_step_runs_no_depthwise_conv_in_torch(cuda, monkeypatch):
    """Calls of nn.Conv2d._conv_forward with groups > 1 during a bf16 yolox_nano training step: none on the default path,
    all 30 with YX_TRAIN_CONV=0."""
    torch.manual_seed(0)
    m = copy.deepcopy(yx.YoloxConfig.get_named_config("yolox_nano").get_model()).float().to(cuda).train()
    x = torch.from_numpy(syn.images(2, 160, 160, seed=3)).to(cuda)
    lab = torch.from_numpy(syn.labels(2, max_gt=8, seed=5, size=160.0, counts=[3, 5])).to(cuda)
    calls = []
    orig = torch.nn.Conv2d._conv_forward

    def counting(self, input, weight, bias):
        if self.groups > 1:
            calls.append(self)
        return orig(self, input, weight, bias)

    monkeypatch.setattr(torch.nn.Conv2d, "_conv_forward", counting)
    counts = {}
    for flag in ("1", "0"):
        monkeypatch.setenv("YX_TRAIN_CONV", flag)
        calls.clear()
        m.zero_grad(set_to_none=True)
        _nano_step(m, x, lab)
        counts[flag] = len(calls)
    assert counts == {"1": 0, "0": 30}, counts


def test_nano_training_step_captures_as_a_cuda_graph(cuda, monkeypatch):
    """A bf16 yolox_nano forward + backward with direct gradients (depthwise wgrad on the side streams) captured with
    torch.cuda.graph and replayed from the same state: the eager step's loss within 1e-3 relative, finite gradients for every
    parameter. The loss is the mean square of the raw prediction maps: the detection loss goes through SimOTA, whose near-tied
    costs flip an assignment (and move the loss by ~1e-3) on last-bit differences of the torch glue around it."""
    from pixeltable_yolox_b200.optim import FusedSgdEma

    monkeypatch.setenv("YX_TRAIN_CONV", "1")
    torch.manual_seed(0)
    m = copy.deepcopy(yx.YoloxConfig.get_named_config("yolox_nano").get_model()).float().to(cuda).train()
    m = m.to(memory_format=torch.channels_last)
    x = _cl(torch.from_numpy(syn.images(8, 416, 416, seed=3)).to(cuda))
    opt = FusedSgdEma(m, lr=0.01, ema=False, direct_grads=True)
    try:
        def step():
            opt.zero_grad()
            with torch.autocast("cuda", dtype=torch.bfloat16):
                outs = m.head._torch_raw_outputs(m.backbone(x))
            loss = sum(t.float().square().mean() for lvl in outs for t in lvl)
            loss.backward()
            opt.join()
            return loss.detach()

        side = torch.cuda.Stream(cuda)
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for _ in range(3):
                eager = float(step())
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, capture_error_mode="thread_local"):
            loss = step()
        g.replay()
        torch.cuda.synchronize()
        assert abs(float(loss) - eager) <= 1e-3 * abs(eager), (float(loss), eager)
        for n, p in m.named_parameters():
            assert torch.isfinite(p.grad).all(), n
        assert float(opt.flat_grad.abs().sum()) > 0
    finally:
        opt.close()
