"""-m gpu: the tensor-core kernels element by element on the persistent multi-tile schedules the product runs.

The element-wise kernel tests (test_gpu_kernels.py) use maps so small that no CTA walks more than one tile, so the
ring / accumulator-stage / epilogue-group rotation, the split weight-sharing group of G = 2, the padded M tile and
two CTAs per SM never run there. Here every conv case is sized with yx_conv_schedule so that each CTA owns at least
three tiles, the references are fp32 (TF32 off) on the exact 16-bit operands, every element is gated, the slack
around each output is a NaN canary compared bit for bit, and image b of a batch equals a batch-1 run of image b.

Gates, relative to max(|ref|, 1):
  * max over every element: 1e-2 (bf16) / 2e-3 (fp16), the gates of test_gpu_kernels.py (one rounding of the
    16-bit output plus the tanh.approx SiLU);
  * mean over every element: one round-to-nearest errs by at most half an ulp and, uniformly spread, by a quarter
    ulp on average; an ulp is at most 2u|y| (u = 2^-8 bf16, 2^-11 fp16), so the mean relative rounding error is at
    most u/2. tanh.approx.f32 errs by at most 2^-10.99 absolute and SiLU(x) = x/2 (1 + tanh(x/2)) scales that by
    |x|/2; the pre-activations here are about N(0, 1.4^2) (unit-variance GEMM plus an N(0, 1) bias), whose |x| averages
    ~1.1, so the SiLU term adds well under 2^-11 on average. Mean gate: u/2 + 2^-11 = 2.44e-3 (bf16, ~gate / 4) and
    7.3e-4 (fp16, ~gate / 3). What a schedule bug does (a wrong bias slice, a tile stored at another tile's pixels, a
    shifted operand) is O(1) on a whole tile.
"""
import math
from dataclasses import dataclass
from typing import Optional

import ctypes as C
import numpy as np
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

from pixeltable_yolox_b200 import _lib, engine, ops  # noqa: E402
from pixeltable_yolox_b200.ops import View  # noqa: E402

GATE = {torch.bfloat16: 1e-2, torch.float16: 2e-3}
MEAN_GATE = {torch.bfloat16: 2.0 ** -9 + 2.0 ** -11, torch.float16: 2.0 ** -12 + 2.0 ** -11}
CANARY = 0x7FA5                        # a NaN in bf16 and in fp16: no kernel computes it, so any write shows
CTAS_SETTINGS = [None, "1", "2"]       # YX_CTAS_PER_SM unset (the product's choice) / forced 1 / forced 2
TILES_PER_CTA = 3
FIELDS = ["mode", "flat", "b_resident", "G", "ctas", "epi_groups", "acc_stages", "a_slots", "stages", "BN", "n_tiles",
          "m_tiles", "num_tiles", "grid", "tw", "th"]


@pytest.fixture(autouse=True)
def _no_tf32():
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False


def _set_ctas(monkeypatch, ctas):
    if ctas is None:
        monkeypatch.delenv("YX_CTAS_PER_SM", raising=False)
    else:
        monkeypatch.setenv("YX_CTAS_PER_SM", ctas)


def _sms(dev) -> int:
    return torch.cuda.get_device_properties(dev).multi_processor_count


# ------------------------------------------------------------------------------------------------ schedule query
def schedule(d) -> Optional[dict]:
    """yx_conv_schedule of a descriptor; None when the shape does not fit (YX_ERR_UNSUPPORTED)."""
    info = (C.c_int32 * len(FIELDS))()
    n = _lib.lib().yx_conv_schedule(C.byref(d), info, len(FIELDS))
    if n == -2:
        return None
    if n < 0:
        _lib.check(n, "conv_schedule")
    assert n == len(FIELDS), n
    return dict(zip(FIELDS, list(info)))


def cta_ranges(s):
    """[(first unit, end unit)] per CTA: contiguous ranges in the halo / planes modes, strided in the per-tap ring."""
    T, g = s["num_tiles"], s["grid"]
    if s["mode"] == 0:
        return [(i, T) for i in range(g)]
    return [(T * i // g, T * (i + 1) // g) for i in range(g)]


def min_tiles_per_cta(s) -> int:
    if s["mode"] == 0:
        return s["num_tiles"] // s["grid"]
    return min(e - b for b, e in cta_ranges(s))


def locate(s, oh, ow, b, y, x, c) -> str:
    """Output element (image, y, x, channel) of the GEMM -> its M / N tile, work unit and the CTA that owns it."""
    if s["flat"]:
        m = ((b * oh + y) * ow + x) // 128
    else:
        tiles_w, tiles_h = -(-ow // s["tw"]), -(-oh // s["th"])
        m = (b * tiles_h + y // s["th"]) * tiles_w + x // s["tw"]
    n = c // s["BN"]
    G, nt, T, g = s["G"], s["n_tiles"], s["num_tiles"], s["grid"]
    if s["mode"] == 0:
        t = m * nt + n
        cta, pos = t % g, t // g
    else:
        t = ((m // G) * nt + n) * G + m % G
        cta = min(g - 1, t * g // T)
        while T * cta // g > t:
            cta -= 1
        while T * (cta + 1) // g <= t:
            cta += 1
        pos = t - T * cta // g
    return (f"(image {b}, y {y}, x {x}, channel {c}) -> m_tile {m}, n_tile {n}, unit {t}, CTA {cta} "
            f"(its tile #{pos}); schedule {s}")


def _gate(got, ref, dtype, what, where=None):
    """Max and mean of |got - ref| / max(|ref|, 1) over every element; on failure name the worst element."""
    err = (got.float() - ref).abs() / ref.abs().clamp_min(1.0)
    err = torch.nan_to_num(err, nan=float("inf"))
    mx, mean = err.max().item(), err.mean().item()
    if mx <= GATE[dtype] and mean <= MEAN_GATE[dtype]:
        return None
    idx = np.unravel_index(int(err.argmax()), tuple(err.shape))
    loc = where(*idx) if where is not None else str(tuple(int(i) for i in idx))
    return (f"{what}: max err {mx:.3e} (gate {GATE[dtype]:.1e}), mean {mean:.3e} (gate {MEAN_GATE[dtype]:.2e}); worst "
            f"got {got.flatten()[int(err.argmax())].item():.6g} want {ref.flatten()[int(err.argmax())].item():.6g} at {loc}")


# ------------------------------------------------------------------------------------------------ conv cases
@dataclass(frozen=True)
class Conv:
    """One standalone conv: geometry, buffer layout (channel offsets / row pitches) and epilogue."""
    name: str
    H: int
    W: int
    cin: int
    cout: int
    k: int
    s: int
    in_ld: int = 0            # 0: dense (= cin); the input is channels [in_off, in_off + cin) of an in_ld-wide buffer
    in_off: int = 0
    out_ld: int = 0           # 0: dense; the output is channels [out_off, out_off + width) of an out_ld-wide buffer
    out_off: int = 0
    kind: str = "store"       # store / res / ups / out2 / shuffle
    out2_begin: int = 0
    out2_ld: int = 0
    act: int = _lib.YX_ACT_SILU
    odd_m: bool = False       # pick an odd M tile count (the padded tile of G = 2)

    @property
    def oh(self):
        return (self.H + 2 * ((self.k - 1) // 2) - self.k) // self.s + 1

    @property
    def ow(self):
        return (self.W + 2 * ((self.k - 1) // 2) - self.k) // self.s + 1

    @property
    def width(self):          # channels of the first destination
        if self.kind == "out2":
            return self.out2_begin
        if self.kind == "shuffle":
            return self.cout // 4
        return self.cout


class Bufs:
    """Device tensors of one run of a Conv case. Every 16-bit output lives in a flat allocation whose slack -- the
    channels outside the view and 130 rows past the last pixel (where a padded M tile or the flat tail tile would
    land) -- holds the CANARY bit pattern."""

    def __init__(self, case: Conv, B: int, dtype, dev, seed: int, x=None, w=None, bias=None, res=None):
        g = torch.Generator(device=dev).manual_seed(seed)
        c = case
        in_ld = c.in_ld or c.cin
        self.x = x if x is not None else torch.randn(B, c.H, c.W, in_ld, device=dev, generator=g).to(dtype)
        self.xv = View(self.x, c.in_off, c.cin)
        kk = c.k * c.k
        self.w = w if w is not None else (torch.randn(c.cout, kk, c.cin, device=dev, generator=g) / (kk * c.cin) ** 0.5).to(dtype)
        self.bias = bias if bias is not None else torch.randn(c.cout, device=dev, generator=g)
        oh, ow = (2 * c.oh, 2 * c.ow) if c.kind == "shuffle" else (c.oh, c.ow)
        self.out_flat, self.out = self._canary_buf(B, oh, ow, c.out_ld or c.width, dtype, dev)
        self.ov = View(self.out, c.out_off, c.width)
        self.res = self.ups = self.o2 = self.o2v = None
        if c.kind == "res":
            self.res = res if res is not None else torch.randn(B, c.oh, c.ow, c.cout, device=dev, generator=g).to(dtype)
        if c.kind == "ups":
            self.ups = torch.full((B, 2 * c.oh, 2 * c.ow, c.cout), 7.0, device=dev, dtype=dtype)
        if c.kind == "out2":
            self.o2_flat, self.o2 = self._canary_buf(B, c.oh, c.ow, c.out2_ld or c.cout - c.out2_begin, dtype, dev)
            self.o2v = View(self.o2, 0, c.cout - c.out2_begin)

    @staticmethod
    def _canary_buf(B, h, w, ld, dtype, dev):
        flat = torch.full(((B * h * w + 130) * ld,), CANARY, dtype=torch.int16, device=dev).view(dtype)
        return flat, flat[:B * h * w * ld].view(B, h, w, ld)

    def desc(self, case: Conv):
        c = case
        return ops.make_conv_desc(self.xv, self.w, self.bias, self.ov, c.k, 1 if c.kind == "shuffle" else c.s, c.act,
                                  res=View(self.res) if self.res is not None else None,
                                  ups=View(self.ups) if self.ups is not None else None,
                                  out2=self.o2v, out2_begin=c.out2_begin,
                                  shuffle2_c=c.cout // 4 if c.kind == "shuffle" else 0)

    def run(self, case: Conv):
        c = case
        ops.conv_bn_act(self.xv, self.w, self.bias, self.ov, c.k, 1 if c.kind == "shuffle" else c.s, c.act,
                        res=View(self.res) if self.res is not None else None,
                        ups=View(self.ups) if self.ups is not None else None, out2=self.o2v, out2_begin=c.out2_begin,
                        shuffle2_c=c.cout // 4 if c.kind == "shuffle" else 0)

    def result(self, case: Conv):
        """The full GEMM output [B, OH, OW, cout] as the kernel stored it (shuffle: gathered back from the 2x map)."""
        c = case
        if c.kind == "out2":
            return torch.cat([self.ov.torch(), self.o2v.torch()], -1)
        if c.kind == "shuffle":
            sc = c.cout // 4
            o = self.ov.torch()
            return torch.cat([o[:, q >> 1::2, q & 1::2] for q in range(4)], -1)[..., :4 * sc]
        return self.ov.torch()

    def slack_ok(self, case: Conv) -> Optional[str]:
        c = case
        bufs = [(self.out_flat, self.out, c.out_off, c.width)]
        if c.kind == "out2":
            bufs.append((self.o2_flat, self.o2, 0, c.cout - c.out2_begin))
        for flat, t, off, width in bufs:
            n = t.numel()
            tail = flat[n:].view(torch.int16)
            if not bool((tail == CANARY).all()):
                row = int((tail != CANARY).nonzero()[0]) // t.shape[3]
                return f"wrote row {row} past the last pixel (a padded / tail tile)"
            bits = t.view(torch.int16)
            for lo, hi in ((0, off), (off + width, t.shape[3])):
                if hi > lo and not bool((bits[..., lo:hi] == CANARY).all()):
                    return f"wrote outside the channel slice [{off}, {off + width}) (channels {lo}..{hi - 1})"
        return None


def reference(case: Conv, bufs: Bufs) -> torch.Tensor:
    """fp32 (TF32 off) restatement of the conv + bias + act (+ residual) on the exact 16-bit operands: [B, OH, OW, cout]."""
    c = case
    s = 1 if c.kind == "shuffle" else c.s
    pad = (c.k - 1) // 2
    x = bufs.xv.torch().float().permute(0, 3, 1, 2)
    w = bufs.w.float().reshape(c.cout, c.k, c.k, c.cin).permute(0, 3, 1, 2)
    y = F.conv2d(x, w, bufs.bias, s, pad)
    y = {_lib.YX_ACT_SILU: F.silu, _lib.YX_ACT_NONE: lambda t: t, _lib.YX_ACT_RELU: F.relu,
         _lib.YX_ACT_LRELU: lambda t: F.leaky_relu(t, 0.1)}[c.act](y)
    if bufs.res is not None:
        y = y + bufs.res.float().permute(0, 3, 1, 2)
    return y.permute(0, 2, 3, 1)


def pick_batch(case: Conv, dtype, dev, per_cta=TILES_PER_CTA):
    """Smallest batch whose schedule gives every CTA >= per_cta tiles over an uneven split (num_tiles % grid != 0),
    from the schedule query at the current YX_CTAS_PER_SM; (None, None) when the shape does not fit."""
    s1 = schedule(_query_desc(case, 1, dtype, dev))
    if s1 is None:
        return None, None
    target = per_cta * _sms(dev) * s1["ctas"]
    B = max(1, math.ceil(target / s1["num_tiles"]))
    for _ in range(64):
        s = schedule(_query_desc(case, B, dtype, dev))
        if min_tiles_per_cta(s) >= per_cta and s["num_tiles"] % s["grid"] and (s["m_tiles"] % 2 or not case.odd_m):
            return B, s
        B += 1
    raise AssertionError(f"{case.name}: no batch up to {B} gives {per_cta} tiles per CTA: {s}")


_DUMMY = {}


def _query_desc(case: Conv, B: int, dtype, dev):
    """The case's descriptor at batch B, for the schedule query only: every pointer points into one small buffer
    (the query encodes tensor maps, which take addresses and strides but read no memory)."""
    key = (dev, dtype)
    if key not in _DUMMY:
        _DUMMY[key] = torch.zeros(1 << 16, device=dev, dtype=dtype)
    p = _DUMMY[key].data_ptr()
    c = case
    d = _lib.ConvDesc()
    d.batch, d.in_h, d.in_w, d.in_c = B, c.H, c.W, c.cin
    d.out_h, d.out_w, d.out_c = c.oh, c.ow, c.cout
    d.ksize, d.stride = c.k, 1 if c.kind == "shuffle" else c.s
    d.dtype, d.act, d.epilogue = _lib.dtype_code(dtype), c.act, _lib.YX_EPI_STORE
    d.in_, d.in_ld = p + 2 * c.in_off, c.in_ld or c.cin
    d.w, d.bias = p, p
    d.out, d.out_ld = p + 2 * c.out_off, c.out_ld or c.width
    if c.kind == "res":
        d.res, d.res_ld = p, c.cout
    if c.kind == "ups":
        d.ups, d.ups_ld = p, c.cout
    if c.kind == "out2":
        d.out2, d.out2_ld, d.out2_begin = p, c.out2_ld or c.cout - c.out2_begin, c.out2_begin
    if c.kind == "shuffle":
        d.shuffle2_c = c.cout // 4
    return d


def check_conv(case: Conv, B: int, s: dict, dtype, dev, seed=0, invariance=True, w=None, bias=None) -> list:
    """Run the case at batch B once; returns failure messages: element gate, canaries and, where the tiles of a batch-1
    run hold the same pixels in the same accumulator rows, bit-for-bit batch invariance of the first and last image."""
    bufs = Bufs(case, B, dtype, dev, seed, w=w, bias=bias)
    bufs.run(case)
    torch.cuda.synchronize()
    fails = []
    got = bufs.result(case)
    msg = _gate(got, reference(case, bufs), dtype, f"{case.name} B={B} {str(dtype)[6:]}",
                lambda b, y, x, c: locate(s, case.oh, case.ow, b, y, x, c))
    if msg:
        fails.append(msg)
    msg = bufs.slack_ok(case)
    if msg:
        fails.append(f"{case.name} B={B}: {msg}; schedule {s}")
    if case.kind == "ups":
        for dy in (0, 1):
            for dx in (0, 1):
                if not torch.equal(bufs.ups[:, dy::2, dx::2], bufs.ov.torch()):
                    fails.append(f"{case.name} B={B}: the 2x nearest copy differs from the output")
    # flat 1x1 tiles are 128 consecutive pixels of the flattened batch: only maps with H*W % 128 == 0 put every pixel
    # in the same accumulator row at batch 1
    if invariance and not (s["flat"] and (case.oh * case.ow) % 128):
        for b in sorted({0, B - 1}):
            one = Bufs(case, 1, dtype, dev, seed, x=bufs.x[b:b + 1].contiguous(), w=bufs.w, bias=bufs.bias,
                       res=None if bufs.res is None else bufs.res[b:b + 1].contiguous())
            one.run(case)
            torch.cuda.synchronize()
            a, r = got[b:b + 1].view(torch.int16), one.result(case).view(torch.int16)
            if not torch.equal(a, r):
                bad = (a != r).nonzero()[0].tolist()
                fails.append(f"{case.name}: image {b} of the batch-{B} run differs from its batch-1 run at "
                             f"{locate(s, case.oh, case.ow, b, *bad[1:])}")
    return fails


# ------------------------------------------------------------------------------------------------ inventory
INVENTORY_MODELS = [("yolox_s", torch.bfloat16), ("yolox_l", torch.float16)]
_HARVEST = {}


def harvest(name: str, dev):
    """Every conv / fused bottleneck / fused stem shape the lowering of `name` emits, recorded during an eager
    (use_plan=False) batch-1 forward at the config's test size. Convs are deduplicated by
    (in_h, in_w, in_c, out_c, ksize, stride, epilogue kind) and keep the buffer pitches of their first occurrence."""
    if name in _HARVEST:
        return _HARVEST[name]
    import pixeltable_yolox_b200 as yx

    cfg = yx.YoloxConfig.get_named_config(name)
    cfg.model = None
    model = cfg.get_model().eval().to(dev).to(torch.bfloat16)
    cfg.model = None
    convs, bnecks, stems = {}, set(), set()
    B = engine.Builder
    orig = B._emit_conv, B.bottleneck, B.focus_conv

    def emit(self, d):
        if d.epilogue == _lib.YX_EPI_HEAD:
            kind = "head"
        else:
            kind = "res" if d.res else "ups" if d.ups else "out2" if d.out2 else "store"
        key = (d.in_h, d.in_w, d.in_c, d.out_c, d.ksize, d.stride, kind)
        if key not in convs:
            convs[key] = dict(in_ld=d.in_ld, out_ld=d.out_ld, out2_begin=d.out2_begin, out2_ld=d.out2_ld, act=d.act)
        return orig[0](self, d)

    def bneck(self, x, m, out):
        bnecks.add((x.H, x.W, x.segs[0], bool(m.use_add)))
        return orig[1](self, x, m, out)

    def focus(self, img, m, out=None):
        stems.add((img.shape[2], img.shape[3], m.conv.out_channels))
        return orig[2](self, img, m, out)

    h, w = cfg.test_size
    B._emit_conv, B.bottleneck, B.focus_conv = emit, bneck, focus
    try:
        with torch.no_grad():
            b = engine.Builder(dev, torch.bfloat16, use_plan=False)
            feats = model.backbone.lower_image(b, torch.zeros(1, 3, h, w, device=dev))
            A = sum((h // s) * (w // s) for s in model.head.strides)
            model.head.lower(b, list(feats), torch.empty(1, A, 5 + model.head.num_classes, device=dev))
            torch.cuda.synchronize()
    finally:
        B._emit_conv, B.bottleneck, B.focus_conv = orig
    cases = []
    for (ih, iw, ic, oc, k, s, kind), v in sorted(convs.items()):
        if kind == "head":
            continue                      # the prediction GEMMs: test_head_epilogue_at_scale
        in_ld = v["in_ld"] if v["in_ld"] != ic else 0
        out_ld = v["out_ld"] if v["out_ld"] != (v["out2_begin"] if kind == "out2" else oc) else 0
        cases.append(Conv(f"{name}:{k}x{k}s{s} {ic}->{oc} @{ih}x{iw} {kind}", ih, iw, ic, oc, k, s, in_ld=in_ld,
                          out_ld=out_ld, kind=kind, out2_begin=v["out2_begin"], out2_ld=v["out2_ld"], act=v["act"]))
    _HARVEST[name] = (cases, bnecks, stems, sorted(convs))
    del model
    torch.cuda.empty_cache()
    return _HARVEST[name]


def _run_all(cases, ctas, dtype, dev, fails, seen=None):
    ran = 0
    for case in cases:
        B, s = pick_batch(case, dtype, dev)
        if B is None:
            assert ctas == "2", f"{case.name}: does not fit the product's own CTA count (ctas={ctas})"
            continue               # a shape that does not fit two CTAs per SM: only the forced setting may say so
        if seen is not None:
            seen.append((case.name, s))
        fails += check_conv(case, B, s, dtype, dev)
        ran += 1
    return ran


@pytest.mark.parametrize("ctas", CTAS_SETTINGS, ids=["ctas_auto", "ctas_1", "ctas_2"])
@pytest.mark.parametrize("model,dtype", INVENTORY_MODELS, ids=[m for m, _ in INVENTORY_MODELS])
def test_conv_inventory_multi_tile(cuda, monkeypatch, model, dtype, ctas):
    """Every conv shape of the model's lowering, standalone, at a batch where each CTA owns >= 3 tiles."""
    cases = harvest(model, cuda)[0]
    assert len(cases) >= 15, [c.name for c in cases]
    _set_ctas(monkeypatch, ctas)
    fails = []
    ran = _run_all(cases, ctas, dtype, cuda, fails)
    assert ran >= len(cases) // 2
    assert not fails, "\n".join(fails)


# synthetic shapes for combinations the 640x640 inventory cannot reach (checked by test_schedule_coverage)
SYNTH_CASES = [
    # 3x3 128->128 on 26x26: 7 halo tiles per image, streamed weights, G = 2; an odd batch gives an odd m_tiles
    Conv("odd_mtiles_g2 3x3 128->128 @26x26", 26, 26, 128, 128, 3, 1, odd_m=True),
    Conv("odd_mtiles_g2 3x3 128->128 @26x26 fp16 slices", 26, 26, 128, 128, 3, 1, in_ld=192, in_off=32,
         out_ld=176, out_off=16, odd_m=True),
    # channel-sliced input and output views with slack on both sides, one per mode
    Conv("slices 1x1 64->128 @80x80", 80, 80, 64, 128, 1, 1, in_ld=128, in_off=32, out_ld=160, out_off=16),
    Conv("slices 3x3 64->64 @40x40", 40, 40, 64, 64, 3, 1, in_ld=96, in_off=16, out_ld=96, out_off=16),
    Conv("slices 3x3s2 64->128 @80x80", 80, 80, 64, 128, 3, 2, in_ld=96, in_off=16, out_ld=160, out_off=16),
    Conv("slices 1x1 512->256 @20x20 ring", 20, 20, 512, 256, 1, 1, in_ld=544, in_off=16, out_ld=288, out_off=16),
    # residual / 2x upsample / two destinations on multi-tile schedules of each mode
    Conv("res 3x3 64->64 @80x80", 80, 80, 64, 64, 3, 1, kind="res"),
    Conv("res 3x3 128->128 @40x40 G2", 40, 40, 128, 128, 3, 1, kind="res"),
    Conv("ups 1x1 256->128 @40x40", 40, 40, 256, 128, 1, 1, kind="ups"),
    Conv("ups 1x1 512->256 @20x20 ring", 20, 20, 512, 256, 1, 1, kind="ups"),
    Conv("out2 1x1 128->128 @80x80", 80, 80, 128, 128, 1, 1, kind="out2", out2_begin=64, out2_ld=80),
    Conv("out2 3x3 64->96 @40x40", 40, 40, 64, 96, 3, 1, kind="out2", out2_begin=48),
]
SYNTH_DTYPES = {1: torch.float16}      # index -> dtype (default bf16)


@pytest.mark.parametrize("ctas", CTAS_SETTINGS, ids=["ctas_auto", "ctas_1", "ctas_2"])
def test_conv_synthetic_multi_tile(cuda, monkeypatch, ctas):
    _set_ctas(monkeypatch, ctas)
    fails = []
    for i, case in enumerate(SYNTH_CASES):
        B, s = pick_batch(case, SYNTH_DTYPES.get(i, torch.bfloat16), cuda)
        if B is None:
            assert ctas == "2", case.name
            continue
        fails += check_conv(case, B, s, SYNTH_DTYPES.get(i, torch.bfloat16), cuda, seed=i)
    assert not fails, "\n".join(fails)


# the sub-pixel dgrad store of a stride-2 training conv: a stride-1 3x3 conv over dy whose 4*i output channel blocks go
# depth-to-space (dark2 32->64 @320, dark3 64->128 @160, dark5 256->512 @40 of the config-4 step)
SHUFFLE_CASES = [(32, 64, 160), (64, 128, 80), (256, 512, 20)]


@pytest.mark.parametrize("ctas", CTAS_SETTINGS, ids=["ctas_auto", "ctas_1", "ctas_2"])
def test_subpixel_dgrad_store_multi_tile(cuda, monkeypatch, ctas):
    _set_ctas(monkeypatch, ctas)
    fails = []
    for ci, co, oh in SHUFFLE_CASES:
        g = torch.Generator(device=cuda).manual_seed(ci)
        weight = torch.randn(co, ci, 3, 3, device=cuda, generator=g) / (9 * co) ** 0.5
        _, wd = ops.pack_train_weights(weight, torch.bfloat16, co, ci, True, subpixel=True)
        case = Conv(f"shuffle dgrad {co}->{ci} s2 @{oh}x{oh}", oh, oh, co, 4 * ci, 3, 1, kind="shuffle",
                    act=_lib.YX_ACT_NONE)
        B, s = pick_batch(case, torch.bfloat16, cuda)
        if B is None:
            assert ctas == "2", case.name
            continue
        fails += check_conv(case, B, s, torch.bfloat16, cuda, w=wd, bias=torch.zeros(4 * ci, device=cuda))
    assert not fails, "\n".join(fails)


# ------------------------------------------------------------------------------------------------ PDL chain
PDL_CHAINS = [
    (Conv("pdl A 1x1 64->64 @80x80", 80, 80, 64, 64, 1, 1), Conv("pdl B 3x3 64->64 @80x80", 80, 80, 64, 64, 3, 1)),
    (Conv("pdl A 3x3 64->64 @80x80", 80, 80, 64, 64, 3, 1), Conv("pdl B 3x3s2 64->128 @80x80", 80, 80, 64, 128, 3, 2)),
    (Conv("pdl A 3x3 128->128 @40x40", 40, 40, 128, 128, 3, 1), Conv("pdl B 1x1 128->256 @40x40", 40, 40, 128, 256, 1, 1)),
]


@pytest.mark.parametrize("ctas", ["1", "2"], ids=["ctas_1", "ctas_2"])
def test_pdl_chain_consumer_reads_producer_output(cuda, monkeypatch, ctas):
    """Conv A then conv B enqueued back to back on one stream (B reads A's output; programmatic dependent launch lets
    B's prologue and resident-weight loads overlap A's tail). B is checked against the reference applied to A's
    actual output, read after the synchronise. One run per chain."""
    _set_ctas(monkeypatch, ctas)
    fails = []
    for i, (ca, cb) in enumerate(PDL_CHAINS):
        Ba, _ = pick_batch(ca, torch.bfloat16, cuda)
        Bb, sb = pick_batch(cb, torch.bfloat16, cuda)
        if Ba is None or Bb is None:
            assert ctas == "2"
            continue
        B = max(Ba, Bb)
        sb = schedule(_query_desc(cb, B, torch.bfloat16, cuda))
        a = Bufs(ca, B, torch.bfloat16, cuda, 10 + i)
        b = Bufs(cb, B, torch.bfloat16, cuda, 20 + i, x=a.out)
        a.run(ca)
        b.run(cb)                        # no synchronisation between the two launches
        torch.cuda.synchronize()
        msg = _gate(b.result(cb), reference(cb, b), torch.bfloat16, f"{cb.name} after {ca.name} B={B}",
                    lambda bb, y, x, c: locate(sb, cb.oh, cb.ow, bb, y, x, c))
        if msg:
            fails.append(msg)
    assert not fails, "\n".join(fails)


# ------------------------------------------------------------------------------------------------ head epilogue
HEAD_LEVELS = [(80, 8.0), (40, 16.0), (20, 32.0)]
HEAD_C, HEAD_NC = 128, 80
HEAD_A = sum(hw * hw for hw, _ in HEAD_LEVELS)
# fp32 output, no 16-bit rounding: the fp32 accumulation of K = 128 products errs by at most K * 2^-24 * sum|terms|
# (~7.6e-6 * ~10 for these unit-scale operands), which exp() of the w / h channels turns into the same relative error;
# ex2 / rcp.approx and __expf add ~1e-7. Gate 1e-4 on the max, 1e-4 / 8 on the mean.
HEAD_GATE = 1e-4


def _head_query(B, hw, stride, off, decode, dtype, dev):
    c = Conv("head", hw, hw, HEAD_C, 96, 1, 1, act=_lib.YX_ACT_NONE)
    d = _query_desc(c, B, dtype, dev)
    d.epilogue, d.out, d.out_ld = _lib.YX_EPI_HEAD, 0, 0
    d.head_out, d.head_anchors, d.head_anchor_off = d.w, HEAD_A, off
    d.head_nc, d.head_decode, d.head_stride = HEAD_NC, decode, stride
    return d


def _head_batch(hw, stride, off, decode, dtype, dev):
    s1 = schedule(_head_query(1, hw, stride, off, decode, dtype, dev))
    B = max(1, math.ceil(TILES_PER_CTA * _sms(dev) / s1["num_tiles"]))
    while True:
        s = schedule(_head_query(B, hw, stride, off, decode, dtype, dev))
        if min_tiles_per_cta(s) >= TILES_PER_CTA and s["num_tiles"] % s["grid"]:
            return B, s
        B += 1


def _head_inputs(B, dtype, dev, seed):
    g = torch.Generator(device=dev).manual_seed(seed)
    xs = [(torch.randn(B, hw, hw, HEAD_C, device=dev, generator=g) * 0.5).to(dtype) for hw, _ in HEAD_LEVELS]
    ws = [(torch.randn(96, 1, HEAD_C, device=dev, generator=g) / HEAD_C ** 0.5).to(dtype) for _ in HEAD_LEVELS]
    bs = [torch.cat([torch.randn(4, device=dev, generator=g) * 0.3, torch.randn(92, device=dev, generator=g) - 1.0])
          for _ in HEAD_LEVELS]
    return xs, ws, bs


@pytest.mark.parametrize("decode", [0, 3])
@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float16])
def test_head_epilogue_at_scale(cuda, dtype, decode):
    """YX_EPI_HEAD on each level alone, into a [B, A, 85] tensor whose other rows hold a sentinel: the level's rows
    against an fp64 restatement of decode_outputs (yolo_head.py:233-251) on the 16-bit operands, the rest untouched."""
    from oracle import yolox_oracle as yo

    fails = []
    off = 0
    for lvl, (hw, stride) in enumerate(HEAD_LEVELS):
        B, s = _head_batch(hw, stride, off, decode, dtype, cuda)
        xs, ws, bs = _head_inputs(B, dtype, cuda, 40 + lvl)
        out = torch.full((B, HEAD_A, 5 + HEAD_NC), CANARY, dtype=torch.int32, device=cuda).view(torch.float32)
        head = dict(out_ptr=out.data_ptr(), anchors=HEAD_A, anchor_off=off, nc=HEAD_NC, decode=decode, stride=stride)
        ops.conv_bn_act(View(xs[lvl]), ws[lvl], bs[lvl], None, 1, 1, _lib.YX_ACT_NONE, head=head)
        torch.cuda.synchronize()
        raw = torch.einsum("bhwc,oc->bhwo", xs[lvl].double(), ws[lvl][:, 0].double()) + bs[lvl].double()
        raw = raw.reshape(B, hw * hw, 96)[..., :5 + HEAD_NC]
        want = raw
        if decode & 2:
            want = torch.cat([want[..., :4], torch.sigmoid(want[..., 4:])], -1)
        if decode & 1:
            want = yo.decode_outputs(want, [(hw, hw)], [stride])
        got = out[:, off:off + hw * hw]
        err = (got.double() - want).abs() / want.abs().clamp_min(1.0)
        err = torch.nan_to_num(err, nan=float("inf"))
        if err.max().item() > HEAD_GATE or err.mean().item() > HEAD_GATE / 8:
            b, a, ch = np.unravel_index(int(err.argmax()), tuple(err.shape))
            fails.append(f"level {hw}x{hw} decode {decode}: max err {err.max().item():.3e}, mean {err.mean().item():.3e} "
                         f"at {locate(s, hw, hw, int(b), int(a) // hw, int(a) % hw, int(ch))}")
        bits = out.view(torch.int32)
        rest = torch.cat([bits[:, :off], bits[:, off + hw * hw:]], 1)
        if not bool((rest == CANARY).all()):
            fails.append(f"level {hw}x{hw} decode {decode}: wrote rows of another level (B={B})")
        off += hw * hw
    assert not fails, "\n".join(fails)


@pytest.mark.parametrize("thr", [0.3, 0.01])
def test_head_fused_score_filter_at_scale(cuda, thr):
    """The score filter fused into the decode epilogue (head_cand) + yx_nms_prefiltered == the plain decode epilogue
    + postprocess_device, bit for bit, at a batch where the 80x80 level's CTAs own >= 3 tiles each; 0.01 keeps most
    anchors."""
    dtype = torch.bfloat16
    B, _ = _head_batch(80, 8.0, 0, 3, dtype, cuda)
    xs, ws, bs = _head_inputs(B, dtype, cuda, 50)

    def run(post):
        out = torch.zeros(B, HEAD_A, 5 + HEAD_NC, device=cuda)
        off = 0
        for (hw, stride), x, w, bias in zip(HEAD_LEVELS, xs, ws, bs):
            head = dict(out_ptr=out.data_ptr(), anchors=HEAD_A, anchor_off=off, nc=HEAD_NC, decode=3, stride=stride)
            head.update(post)
            ops.conv_bn_act(View(x), w, bias, None, 1, 1, 0, head=head)
            off += hw * hw
        return out

    ref_pred = run({})
    d0, i0, n0 = ops.postprocess_device(ref_pred, HEAD_NC, thr, 0.65, 0, inplace_xyxy=True)
    ws_ = torch.empty(_lib.lib().yx_postprocess_workspace_bytes(B, HEAD_A), dtype=torch.uint8, device=cuda)
    cand, keys, counts = ops.postprocess_ws_ptrs(ws_, B, HEAD_A)
    ops.postprocess_begin(ws_, B, HEAD_A)
    fused_pred = run({"cand_ptr": cand, "keys_ptr": keys, "counts_ptr": counts, "conf_thre": thr, "xyxy": True})
    d1, i1, n1 = ops.nms_prefiltered(ws_, B, HEAD_A, 0.65, 0)
    torch.cuda.synchronize()
    assert int(n0.sum()) > 0 and torch.equal(n0, n1)
    assert torch.equal(fused_pred, ref_pred)
    for b in range(B):
        k = int(n0[b])
        assert torch.equal(d0[b, :k], d1[b, :k]) and torch.equal(i0[b, :k], i1[b, :k]), b
    if thr == 0.01:
        passed = (ref_pred[..., 4:5] * ref_pred[..., 5:].max(-1, keepdim=True).values >= thr).float().mean().item()
        assert passed > 0.5, passed


# ------------------------------------------------------------------------------------------------ bottleneck / stem
def _images_for(pixels_per_image, dev, ctas=2):
    """Batch with B*H*W >= 3 tiles of <= 128 pixels for each of `ctas` CTAs on every SM (no schedule query here)."""
    return math.ceil(TILES_PER_CTA * ctas * 128 * _sms(dev) / pixels_per_image)


# (H, W, c, in_off, out_off): the two fused-bottleneck widths of the inventory at their map sizes, plus a sliced case
BNECK_SCALE = [(160, 160, 32, 0, 0), (80, 80, 64, 0, 0), (80, 80, 32, 32, 16)]
# gates of test_fused_bottleneck_vs_torch (one output rounding plus hidden values that round differently at a tie);
# the mean gate / 8 is above the u/2 + 2^-11 of a single rounding
BNECK_GATE = {torch.bfloat16: 2e-2, torch.float16: 4e-3}


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float16])
@pytest.mark.parametrize("case", BNECK_SCALE, ids=[f"{h}x{w}_c{c}_off{i}" for h, w, c, i, _ in BNECK_SCALE])
def test_fused_bottleneck_at_scale(cuda, case, dtype):
    from tests.test_gpu_kernels import _bneck_run

    H, W, c, in_off, out_off = case
    B = _images_for(H * W, cuda)
    for use_add in (True, False):
        got, want, o, (xin, w1, b1, w2, b2) = _bneck_run(cuda, B, H, W, c, dtype, use_add, "silu", in_off, out_off,
                                                         seed=c + use_add)
        err = (got - want).abs() / want.abs().clamp_min(1.0)
        b, y, x, ch = np.unravel_index(int(err.argmax()), tuple(err.shape))
        where = f"(image {b}, y {y}, x {x}, channel {ch}) of B={B}"
        assert err.max().item() <= BNECK_GATE[dtype], (use_add, err.max().item(), where)
        assert err.mean().item() <= BNECK_GATE[dtype] / 8, (use_add, err.mean().item())
        if out_off:
            assert (o[..., :out_off] == 7).all() and (o[..., out_off + c:] == 7).all(), "wrote outside the channel slice"
        for b in sorted({0, B - 1}):
            one = torch.full((1, H, W, o.shape[3]), 7.0, device=cuda, dtype=dtype)
            ops.bottleneck_fwd(View(xin.t[b:b + 1].contiguous(), xin.c_off, c), w1, b1, w2, b2, View(one, out_off, c),
                               _lib.YX_ACT_SILU, use_add)
            assert torch.equal(one.view(torch.int16), o[b:b + 1].view(torch.int16)), f"image {b} of B={B} != batch-1 run"


@pytest.mark.parametrize("img_dtype", [torch.uint8, torch.float32])
@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float16])
def test_fused_stem_at_scale(cuda, dtype, img_dtype):
    """Focus + 3x3 conv + BN + SiLU as one kernel at 640x640 (102 400 output pixels per image; the fp16 path feeds
    pixels as x/256) against Focus._train_forward in fp32; image b of the batch equals a batch-1 run."""
    from pixeltable_yolox_b200.engine import Builder
    from pixeltable_yolox_b200.network_blocks import Focus

    B = max(2, _images_for(320 * 320, cuda))
    assert B <= 4, B
    torch.manual_seed(5)
    blk = Focus(3, 32, ksize=3)
    bn = blk.conv.bn
    bn.eps = 1e-3
    bn.running_mean.normal_(0, 20.0); bn.running_var.uniform_(500.0, 4000.0)
    bn.weight.data.uniform_(0.5, 1.5); bn.bias.data.normal_(0, 0.2)
    blk = blk.eval().to(cuda)
    g = torch.Generator(device=cuda).manual_seed(3)
    img = torch.randint(0, 256, (B, 3, 640, 640), generator=g, device=cuda).float()
    with torch.no_grad():
        want = blk._train_forward(img)
    blk = blk.to(dtype)
    b = Builder(cuda, dtype, use_plan=False)
    got = blk.lower_image(b, img.to(img_dtype).contiguous()).to_nchw().float()
    # the tolerances of test_fused_focus_stem_matches_focus_then_conv (108 products of 0..255 pixels)
    tol = 4e-2 if dtype == torch.bfloat16 else 6e-3
    err = (got - want).abs() / want.abs().clamp_min(1.0)
    bb, ch, y, x = np.unravel_index(int(err.argmax()), tuple(err.shape))
    assert err.max().item() <= tol, (err.max().item(), f"(image {bb}, y {y}, x {x}, channel {ch})")
    assert err.mean().item() <= tol / 8
    for i in sorted({0, B - 1}):
        one = blk.lower_image(b, img[i:i + 1].to(img_dtype).contiguous()).to_nchw()
        assert torch.equal(one.float(), got[i:i + 1]), f"image {i} of B={B} != batch-1 run"


# ------------------------------------------------------------------------------------------------ training convs
# the config-4 step (8 images at 640x640): stem 12->32 (padded to 16 input channels) @320, dark2 32->64 s2 @320->160,
# 64->64 3x3 @160, dark5 256->512 s2 @40->20 -- forward, the sub-pixel stride-2 dgrad and wgrad
TRAIN_SCALE = [(8, 12, 32, 320, 3, 1), (8, 32, 64, 320, 3, 2), (8, 64, 64, 160, 3, 1), (8, 256, 512, 40, 3, 2)]


@pytest.mark.parametrize("case", TRAIN_SCALE, ids=[f"{ci}to{co}_s{s}_{h}" for _, ci, co, h, _, s in TRAIN_SCALE])
def test_train_conv_at_config4_scale(cuda, case):
    from pixeltable_yolox_b200 import train_conv

    B, ci, co, H, k, s = case
    dtype = torch.bfloat16
    torch.manual_seed(ci * 7 + co)
    conv = torch.nn.Conv2d(ci, co, k, s, (k - 1) // 2, bias=False).to(cuda).to(memory_format=torch.channels_last)
    x = (torch.randn(B, ci, H, H, device=cuda) * 0.8).to(dtype).contiguous(memory_format=torch.channels_last)
    x.requires_grad_(True)
    assert train_conv.usable(x, conv) == dtype
    y = train_conv.conv2d(x, conv)
    go = (torch.randn(y.shape, device=cuda) * 0.3).to(dtype)
    y.backward(go)
    # reference: fp32 autograd of the same rounded operands (test_train_conv_forward_backward_matches_torch)
    xr = x.detach().float().requires_grad_(True)
    wr = conv.weight.detach().to(dtype).float().requires_grad_(True)
    yr = F.conv2d(xr, wr, None, s, (k - 1) // 2)
    yr.backward(go.float())
    tol = dict(rtol=1.6e-2, atol=1.6e-2)
    torch.testing.assert_close(y.float(), yr, **tol)
    torch.testing.assert_close(x.grad.float(), xr.grad, **tol)
    # dW sums B*OH*OW = 51k..205k products here: its reference is fp64 (cuDNN's fp32 weight gradient at these sizes
    # can take transform-based algorithms whose error exceeds the 1e-4 gate), the kernel's fp32 sums stay ~1e-6 relative
    want = torch.nn.grad.conv2d_weight(x.detach().double(), tuple(conv.weight.shape), go.double(), stride=s,
                                       padding=(k - 1) // 2)
    wtol = dict(rtol=1e-4, atol=2e-5 * float(want.abs().max()))
    torch.testing.assert_close(conv.weight.grad.double(), want, **wtol)
    # wgrad alone on the padded operands the training path hands it
    ip, op = -(-ci // 16) * 16, -(-co // 16) * 16
    xp = torch.zeros(B, ip, H, H, device=cuda, dtype=dtype).contiguous(memory_format=torch.channels_last)
    xp[:, :ci] = x.detach()
    dyp = torch.zeros(B, op, *go.shape[2:], device=cuda, dtype=dtype).contiguous(memory_format=torch.channels_last)
    dyp[:, :co] = go
    got = ops.conv_wgrad(xp, dyp, conv.weight, k, s)
    torch.testing.assert_close(got.double(), want, **wtol)


# ------------------------------------------------------------------------------------------------ coverage
def test_schedule_coverage(cuda, monkeypatch):
    """The conv cases above, through the schedule query only (no launches), together reach every combination of the
    persistent schedule that can go wrong; a selector change that drops one fails here and names it."""
    seen = []                                  # (case, dtype-independent schedule)
    for ctas in CTAS_SETTINGS:
        _set_ctas(monkeypatch, ctas)
        groups = [(harvest(m, cuda)[0], dt) for m, dt in INVENTORY_MODELS]
        groups.append((SYNTH_CASES, torch.bfloat16))
        groups.append(([Conv(f"shuffle {co}->{ci}", oh, oh, co, 4 * ci, 3, 1, kind="shuffle", act=_lib.YX_ACT_NONE)
                        for ci, co, oh in SHUFFLE_CASES], torch.bfloat16))
        groups.append(([c for pair in PDL_CHAINS for c in pair], torch.bfloat16))
        for cases, dt in groups:
            for case in cases:
                B, s = pick_batch(case, dt, cuda)
                if B is None:
                    assert ctas == "2", case.name
                    continue
                seen.append((case, s))
        off = 0
        for hw, stride in HEAD_LEVELS:
            B, s = _head_batch(hw, stride, off, 3, torch.bfloat16, cuda)
            seen.append((Conv(f"head {hw}", hw, hw, HEAD_C, 96, 1, 1), s))
            off += hw * hw

    def starts_odd(s):
        return s["G"] == 2 and any(b % 2 for b, _ in cta_ranges(s))

    def ends_inside(s):
        return s["G"] == 2 and any(e % 2 for _, e in cta_ranges(s))

    want = {
        "mode ring": lambda c, s: s["mode"] == 0,
        "mode halo 3x3": lambda c, s: s["mode"] == 1 and not s["flat"],
        "mode halo flat": lambda c, s: s["mode"] == 1 and s["flat"],
        "mode planes C=32": lambda c, s: s["mode"] == 2 and c.cin == 32,
        "mode planes C%64==0": lambda c, s: s["mode"] == 2 and c.cin % 64 == 0,
        "halo resident weights": lambda c, s: s["mode"] == 1 and s["b_resident"],
        "halo streamed weights": lambda c, s: s["mode"] == 1 and not s["b_resident"],
        "G=2, a CTA range starting at an odd unit": lambda c, s: starts_odd(s),
        "G=2, a CTA range ending inside a group": lambda c, s: ends_inside(s),
        "G=2 with odd m_tiles (padded tile)": lambda c, s: s["G"] == 2 and s["m_tiles"] % 2 == 1,
        "ctas_per_sm 1": lambda c, s: s["ctas"] == 1,
        "ctas_per_sm 2": lambda c, s: s["ctas"] == 2,
        "epi_groups 1": lambda c, s: s["epi_groups"] == 1,
        "epi_groups 2": lambda c, s: s["epi_groups"] == 2,
        "epi_groups 3": lambda c, s: s["epi_groups"] == 3,
        "epi_groups 3 on acc_stages 4": lambda c, s: s["epi_groups"] == 3 and s["acc_stages"] == 4,
        "n_tiles > 1": lambda c, s: s["n_tiles"] > 1,
        "uneven ranges (num_tiles % grid != 0)": lambda c, s: s["num_tiles"] % s["grid"] != 0,
    }
    hits = {k: [c.name for c, s in seen if f(c, s)] for k, f in want.items()}
    report = "\n".join(f"  {k}: {len(v)} case(s), e.g. {v[0] if v else '-'}" for k, v in hits.items())
    print(f"schedule combinations over {len(seen)} (case, CTA setting) schedules:\n{report}")
    missing = [k for k, v in hits.items() if not v]
    assert not missing, f"no case reaches: {missing}\n{report}"
    thin = [(c.name, s) for c, s in seen if min_tiles_per_cta(s) < TILES_PER_CTA]
    assert not thin, thin
