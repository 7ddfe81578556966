"""GPU parity of the encoder's bandwidth kernels, one at a time through the stand-alone operators of the C ABI, against
float64 references on the CPU.

The bf16-mode-only kernels (the one-channel score convolution k_conv3x3_c1, the stride-1 depthwise k_depthwise3x3_s1x4 and
the tensor-core attention k_enc_attention_mma, one view or all views in one launch) are held here to bounds set by their
own arithmetic; in the whole-encoder tests they only meet a bound relative to the bf16 rounding of a random BatchNorm network.

Every reference is fed the values the kernel reads: activations rounded to bf16 (bf16 mode) or split into hi + lo bf16
exactly as st_act stores them (bf16x3 mode); depthwise / score-conv weights, BatchNorm scale / shift, LayerNorm parameters
and the positional table in fp32, as the engine uploads them.  What remains is the kernel's own arithmetic and the rounding
of its output, so the bounds are:
  * max pool, subsample: bit-exact in both modes;
  * avg pool (bf16): within one bf16 ulp of the reference;
  * element-wise ops: |y - ref| <= rtol |ref| + atol scale, rtol 2^-8 (bf16) / 2^-15 (bf16x3), `scale` the magnitude
    of the summands of that output (so cancellation does not break a relative bound) and atol the fp32 accumulation;
  * attention: rel-L2 <= 8e-3 per (view, head) block on the tensor-core path (P is rounded to bf16 before P V), the
    element-wise bound with scale sum_j p_j |v_j| on the fp32 CUDA-core path.
Outputs must be finite, and every column and pixel the kernel must not write (filled with -3.5 before the call) unchanged.
FPNMT_KERNEL_ERRORS=<path> merges the worst error of each operator, as a fraction of its bound, into that JSON file.

Measured on one B200 (1000 W power limit), worst error as a fraction of the bound, bf16 / bf16x3:
  max pool, subsample 0 mismatches / 0;  avg pool 0.50 ulp / 0.24;  depthwise 0.99 / 0.23;  scale_shift_relu 1.00 / 0.25;
  score conv 0.94 / -;  co-attention 0.99 / 0.25;  tokens_ln_pos 0.99 / 0.23;  attention, tensor-core: rel-L2 1.9e-3
  (one view and all views) against 8e-3;  attention, CUDA core: 0.98 / 0.12.
In bf16 the output rounding alone reaches 2^-8 |y| at the bottom of a binade, so ratios near 1 there are that rounding;
in bf16x3 the hi + lo storage of the output (~2^-17 relative) is a quarter of rtol.  The file runs in about 10 s.
"""
import numpy as np
import pytest
import torch

import fpnmt_oracle as O
from kernel_check import RTOL, check_elementwise, error_report, gen, q_act  # noqa: F401 (error_report: autouse fixture)
from kernel_check import record as _record

pytestmark = pytest.mark.gpu

PRECS = ["bf16", "bf16x3"]
SENTINEL = -3.5                  # bf16-exact: any write to a column outside the op's view changes it


def view_buffer(shape, C, ld, fill, g):
    """fp32 NHWC buffer with ld channels per pixel: the first C random (`fill(shape + (C,))`), the rest NaN (an input) or
    the sentinel (an output)."""
    buf = torch.full(tuple(shape) + (ld,), float("nan"))
    buf[..., :C] = fill(tuple(shape) + (C,), g)
    return buf


def out_buffer(shape, C, ld):
    """Output buffer: NaN where the kernel must write (catches unwritten elements), the sentinel elsewhere."""
    buf = torch.full(tuple(shape) + (ld,), SENTINEL)
    buf[..., :C] = float("nan")
    return buf.cuda()


def check_untouched(y, C):
    extra = y[..., C:]
    assert bool((extra == SENTINEL).all()), "the kernel wrote %d values outside its channel view" % int((extra != SENTINEL).sum())


def check_elementwise(op, y, ref, scale, rtol, atol, floor=0.0):
    """|y - ref| <= rtol |ref| + atol scale + floor everywhere, y finite."""
    y = y.double()
    assert bool(torch.isfinite(y).all()), "%s: %d non-finite outputs (never written?)" % (op, int((~torch.isfinite(y)).sum()))
    err = (y - ref).abs()
    bound = rtol * ref.abs() + atol * scale + floor
    ratio = err / bound.clamp_min(1e-300)
    worst = float(ratio.max())
    _record(op, worst, 1.0)
    if worst > 1.0:
        i = int(ratio.flatten().argmax())
        idx = np.unravel_index(i, tuple(y.shape))
        raise AssertionError("%s: |y - ref| = %.3g > bound %.3g at %s (y %.8g, ref %.8g, scale %.3g); %d elements over" % (
            op, float(err.flatten()[i]), float(bound.flatten()[i]), idx, float(y.flatten()[i]), float(ref.flatten()[i]),
            float(torch.as_tensor(scale).expand_as(ref).flatten()[i]), int((ratio > 1).sum())))


def nchw(x):
    return x.permute(0, 3, 1, 2)


def nhwc(x):
    return x.permute(0, 2, 3, 1)


# ------------------------------------------------------------------------------------------------------------------------
# depthwise 3x3 (MobileNetV2).  bf16 stride 1 runs k_depthwise3x3_s1x4 (4 outputs per thread along x); bf16x3 and stride 2
# the one-output-per-thread k_depthwise3x3.
DW_CASES = [
    # name, N, H, W, C, in_ld, out_ld, stride, act, bias
    ("s1_w1_c8", 2, 1, 1, 8, 0, 0, 1, 3, True),             # Wo % 4 == 1, one-pixel image
    ("s1_w2_c24", 2, 1, 2, 24, 0, 0, 1, 0, False),          # Wo % 4 == 2
    ("s1_w3_c144", 3, 1, 3, 144, 0, 0, 1, 3, False),        # Wo % 4 == 3
    ("s1_w5_c8", 2, 1, 5, 8, 0, 0, 1, 0, True),             # two x-quads, the second with one output
    ("s1_8x8_c960", 2, 8, 8, 960, 0, 0, 1, 3, True),        # Wo % 4 == 0
    ("s1_7x12_c24", 2, 7, 12, 24, 0, 0, 1, 0, False),
    ("s1_6x11_c144_view", 2, 6, 11, 144, 160, 152, 1, 3, True),   # channel views in and out
    ("s2_8x8_c24", 2, 8, 8, 24, 0, 0, 2, 3, True),          # Keras correct_pad: ((0,1),(0,1)) + valid == pad 0, Ho = H/2
    ("s2_14x14_c144", 2, 14, 14, 144, 0, 0, 2, 0, False),
    ("s2_2x6_c960", 3, 2, 6, 960, 0, 0, 2, 3, False),
    ("s2_10x4_c8_view", 2, 10, 4, 8, 24, 16, 2, 0, True),
]


@pytest.mark.parametrize("prec", PRECS)
@pytest.mark.parametrize("case", DW_CASES, ids=[c[0] for c in DW_CASES])
def test_depthwise3x3(case, prec):
    from fpnmt.engine import depthwise3x3
    name, N, H, W, C, in_ld, out_ld, stride, act, has_bias = case
    in_ld, out_ld = in_ld or C, out_ld or C
    g = gen(len(name) * 31 + C)
    x = view_buffer((N, H, W), C, in_ld, lambda s, g: torch.randn(s, generator=g) * 2, g)
    k = (torch.randn(3, 3, C, 1, generator=g) / 2).numpy()
    b = (torch.randn(C, generator=g) * 0.5).numpy() if has_bias else None
    pad = 1 if stride == 1 else 0
    Ho, Wo = (H, W) if stride == 1 else (H // 2, W // 2)
    y = depthwise3x3(x.cuda(), k, b, stride, (pad, pad), (Ho, Wo), act, C, out_buffer((N, Ho, Wo), C, out_ld), prec).cpu()
    check_untouched(y, C)
    xq = nchw(q_act(x[..., :C], prec)).double()
    pads = ((pad, (Ho - 1) * stride + 3 - pad - H), (pad, (Wo - 1) * stride + 3 - pad - W))
    kd = torch.from_numpy(k).double()
    ref = O.depthwise_conv2d(xq, kd, stride, pads)
    scale = O.depthwise_conv2d(xq.abs(), kd.abs(), stride, pads)
    if b is not None:
        bd = torch.from_numpy(b).double().view(1, -1, 1, 1)
        ref, scale = ref + bd, scale + bd.abs()
    if act == 3:
        ref = O.relu6(ref)
    # fp32 accumulation of <= 10 terms: <= 10 * 2^-24 of the summands' magnitude
    check_elementwise("depthwise3x3/" + prec, y[..., :C], nhwc(ref), nhwc(scale), RTOL[prec], 2.0 ** -19)


# ------------------------------------------------------------------------------------------------------------------------
# pooling: k_maxpool<2|3|0>, k_avgpool2, k_subsample2
MAXPOOL_CASES = [
    # name, N, H, W, C, in_ld, out_ld, k, stride, Keras padding (-inf for 'same' / 'valid', zeros when explicit), input
    ("k2_head_8x8_c256", 2, 8, 8, 256, 0, 0, 2, 2, "valid", "mixed"),              # P6 / P7 and the head pools
    ("k2_odd_5x7_c24", 2, 5, 7, 24, 0, 0, 2, 2, "valid", "mixed"),                 # floor
    ("k3_s2_same_resnet_16x16_c64", 2, 16, 16, 64, 0, 0, 3, 2, "same", "mixed"),   # ResNet pool1 (engine: pad 0, Ho = H/2)
    ("k3_s2_zeropad_densenet_16x16_c64", 2, 16, 16, 64, 0, 256, 3, 2, ((1, 1), (1, 1)), "negative"),  # DenseNet pool1 into
    ("k3_s2_zeropad_odd_9x7_c16", 3, 9, 7, 16, 24, 0, 3, 2, ((1, 1), (1, 1)), "negative"),           # its stage buffer
    ("k5_s2_same_generic_11x11_c8", 2, 11, 11, 8, 0, 0, 5, 2, "same", "negative"),  # k_maxpool<0>, -inf padding
    ("k5_s2_zeropad_generic_9x9_c24", 2, 9, 9, 24, 0, 40, 5, 2, ((2, 2), (2, 2)), "negative"),
]


def _pool_input(kind):
    if kind == "negative":                 # all-negative windows: zero padding changes every border output
        return lambda s, g: -(torch.randn(s, generator=g).abs() + 0.05)
    return lambda s, g: torch.randn(s, generator=g) * 3


@pytest.mark.parametrize("prec", PRECS)
@pytest.mark.parametrize("case", MAXPOOL_CASES, ids=[c[0] for c in MAXPOOL_CASES])
def test_maxpool_bit_exact(case, prec):
    from fpnmt.engine import POOL_MAX, pool
    name, N, H, W, C, in_ld, out_ld, k, s, padding, inp = case
    in_ld, out_ld = in_ld or C, out_ld or C
    g = gen(len(name) * 7 + k)
    x = view_buffer((N, H, W), C, in_ld, _pool_input(inp), g)
    xq = q_act(x[..., :C], prec)
    ref = nhwc(O.max_pool(nchw(xq).double(), k, s, padding))
    Ho, Wo = ref.shape[1], ref.shape[2]
    if padding == "same":
        pt, pl, zero = O.tf_same_pad(H, k, s)[0], O.tf_same_pad(W, k, s)[0], False
    elif padding == "valid":
        pt, pl, zero = 0, 0, False
    else:
        pt, pl, zero = padding[0][0], padding[1][0], True
    y = pool(x.cuda(), POOL_MAX, k, s, (pt, pl), (Ho, Wo), zero, C, out_buffer((N, Ho, Wo), C, out_ld), prec).cpu()
    check_untouched(y, C)
    assert bool(torch.isfinite(y[..., :C]).all())
    if zero:
        assert bool((ref[:, 0] == 0).any()), "the case does not exercise the zero padding"
    diff = int((y[..., :C].double() != ref).sum())
    _record("maxpool/" + prec + " (mismatches)", diff, 1)
    assert diff == 0, "%s %s: %d outputs differ from the max of the inputs" % (name, prec, diff)


SUB_CASES = [
    # name, N, H, W, C, in_ld, out_ld
    ("even_8x8_c256", 2, 8, 8, 256, 0, 0),
    ("odd_7x5_c40", 2, 7, 5, 40, 0, 0),                    # Ho = (H+1)/2 keeps the last row and column
    ("one_1x1_c8", 3, 1, 1, 8, 0, 0),
    ("view_9x6_c16", 2, 9, 6, 16, 32, 24),
]


@pytest.mark.parametrize("prec", PRECS)
@pytest.mark.parametrize("case", SUB_CASES, ids=[c[0] for c in SUB_CASES])
def test_subsample2_bit_exact(case, prec):
    from fpnmt.engine import POOL_SUBSAMPLE2, pool
    name, N, H, W, C, in_ld, out_ld = case
    in_ld, out_ld = in_ld or C, out_ld or C
    g = gen(len(name) * 13 + C)
    x = view_buffer((N, H, W), C, in_ld, lambda s, g: torch.randn(s, generator=g) * 3, g)
    Ho, Wo = (H + 1) // 2, (W + 1) // 2
    y = pool(x.cuda(), POOL_SUBSAMPLE2, channels=C, out=out_buffer((N, Ho, Wo), C, out_ld), precision=prec).cpu()
    check_untouched(y, C)
    ref = q_act(x[:, ::2, ::2, :C], prec)
    diff = int((y[..., :C] != ref).sum())
    _record("subsample2/" + prec + " (mismatches)", diff, 1)
    assert diff == 0, "%s %s: %d outputs differ" % (name, prec, diff)


AVG_CASES = [
    # name, N, H, W, C, in_ld, out_ld
    ("even_8x8_c128_densenet_view", 2, 8, 8, 128, 0, 512),   # DenseNet transition: into the next stage buffer
    ("odd_7x9_c24", 2, 7, 9, 24, 0, 0),                      # floor: the last row and column are dropped
    ("view_in_5x4_c16", 3, 5, 4, 16, 48, 24),
]


@pytest.mark.parametrize("prec", PRECS)
@pytest.mark.parametrize("case", AVG_CASES, ids=[c[0] for c in AVG_CASES])
def test_avgpool2(case, prec):
    from fpnmt.engine import POOL_AVG2, pool
    name, N, H, W, C, in_ld, out_ld = case
    in_ld, out_ld = in_ld or C, out_ld or C
    g = gen(len(name) * 17 + C)
    x = view_buffer((N, H, W), C, in_ld, lambda s, g: torch.randn(s, generator=g) * 3, g)
    Ho, Wo = H // 2, W // 2
    y = pool(x.cuda(), POOL_AVG2, channels=C, out=out_buffer((N, Ho, Wo), C, out_ld), precision=prec).cpu()
    check_untouched(y, C)
    xq = nchw(q_act(x[..., :C], prec)).double()
    ref = nhwc(O.avg_pool2(xq))
    yc = y[..., :C].double()
    assert bool(torch.isfinite(yc).all())
    if prec == "bf16":      # fp32 sum of four bf16 values, * 0.25, rounded once: within one bf16 ulp
        ulp = torch.exp2(torch.floor(torch.log2(ref.abs().clamp_min(2.0 ** -126))) - 7)
        ratio = float(((yc - ref).abs() / ulp).max())
        _record("avgpool2/bf16 (ulps)", ratio, 1.0)
        assert ratio <= 1.0, "%s: %.3g bf16 ulps from the mean" % (name, ratio)
    else:
        check_elementwise("avgpool2/bf16x3", yc, ref, nhwc(O.avg_pool2(xq.abs())), RTOL[prec], 2.0 ** -21)


# ------------------------------------------------------------------------------------------------------------------------
# DenseNet pre-activation BN + ReLU: one 8-channel group per thread walking pixels with stride pix_slots, four in flight.
# pix_slots = ceil(148*2048*2 / (C/8)) capped by the pixel count: with C = 1024, 4736 slots, so 160x160 pixels run the
# grid-stride loop twice and end on a partial group of four.
SSR_CASES = [
    # name, pixel shape, C, in_ld, out_ld
    ("c8_1000px", (2, 20, 25), 8, 0, 0),                    # slots == pixels
    ("c24_ragged_37px", (37,), 24, 0, 0),
    ("c128_densenet_view", (2, 16, 16), 128, 256, 0),        # chan_view(stage buffer, 0, cch)
    ("c1024_below_4slots", (1, 50, 60), 1024, 0, 0),        # 3000 pixels < 4 x 4736
    ("c1024_exactly_4slots", (18944,), 1024, 0, 0),
    ("c1024_grid_stride_160x160", (1, 160, 160), 1024, 0, 0),
    ("c520_view_out", (3, 7, 9), 520, 0, 536),
]


@pytest.mark.parametrize("prec", PRECS)
@pytest.mark.parametrize("case", SSR_CASES, ids=[c[0] for c in SSR_CASES])
def test_scale_shift_relu(case, prec):
    from fpnmt.engine import scale_shift_relu
    name, shape, C, in_ld, out_ld = case
    in_ld, out_ld = in_ld or C, out_ld or C
    g = gen(len(name) * 19 + C)
    x = view_buffer(shape, C, in_ld, lambda s, g: torch.randn(s, generator=g) * 2, g)
    sc = (torch.randn(C, generator=g) * 0.5 + 1).numpy()
    sh = (torch.randn(C, generator=g) * 0.5).numpy()
    y = scale_shift_relu(x.cuda(), sc, sh, C, out_buffer(shape, C, out_ld), prec).cpu()
    check_untouched(y, C)
    xq = q_act(x[..., :C], prec).double()
    scd, shd = torch.from_numpy(sc).double(), torch.from_numpy(sh).double()
    ref = torch.relu(xq * scd + shd)
    check_elementwise("scale_shift_relu/" + prec, y[..., :C], ref, (xq * scd).abs() + shd.abs(), RTOL[prec], 2.0 ** -21)


# ------------------------------------------------------------------------------------------------------------------------
# co-attention score map: k_conv3x3_c1 (bf16 only), 8x8 output tiles with a 10x10 halo
SCORE_CASES = [(2, 1, 1), (2, 2, 2), (3, 4, 7), (2, 7, 9), (2, 9, 4), (2, 64, 64), (2, 9, 64)]


@pytest.mark.parametrize("shape", SCORE_CASES, ids=["%dx%dx%d" % s for s in SCORE_CASES])
def test_score_conv(shape):
    from fpnmt.engine import score_conv
    N, H, W = shape
    g = gen(H * 100 + W)
    x = torch.randn(N, H, W, 256, generator=g)
    k = (torch.randn(3, 3, 256, 1, generator=g) / 48).numpy()
    b = np.array([0.75], np.float32)
    y = score_conv(x.cuda(), k, b, torch.full((N, H, W), float("nan")).cuda()).cpu()
    xq = nchw(q_act(x, "bf16")).double()
    kd = torch.from_numpy(k).double()
    ref = O.conv2d(xq, kd, torch.from_numpy(b).double(), 1, "same")[:, 0]
    scale = O.conv2d(xq.abs(), kd.abs(), None, 1, "same")[:, 0] + 0.75
    # 2304 products summed in fp32 (72 per lane, then a 5-level shuffle tree): <= ~80 * 2^-24 of the summands' magnitude
    check_elementwise("score_conv/bf16", y, ref, scale, RTOL["bf16"], 2.0 ** -17)


def test_score_conv_rejects_bf16x3():
    from fpnmt._lib import ERR_INVALID, FpnmtError
    from fpnmt.engine import score_conv
    with pytest.raises(FpnmtError) as e:
        score_conv(torch.zeros(1, 8, 8, 256).cuda(), np.zeros((3, 3, 256, 1), np.float32), np.zeros(1, np.float32),
                   precision="bf16x3")
    assert e.value.code == ERR_INVALID


# ------------------------------------------------------------------------------------------------------------------------
# co-attention: softmax over the HW scores of an image times the class map.  Pixels per block switch 32 -> 128 -> 256 at
# HW = 1024 and 4096.
COATT_HW = [1, 4, 31, 1023, 1024, 4095, 4096, 4097]
COATT_CASES = ([("hw%d_c8_spread" % hw, hw, 8, "spread") for hw in COATT_HW] +
               [("hw%d_c256_spread" % hw, hw, 256, "spread") for hw in (31, 1023, 1024, 4095, 4096, 4097)] +
               [("hw%d_c256_equal" % hw, hw, 256, "equal") for hw in (4, 1024, 4097)])


@pytest.mark.parametrize("prec", PRECS)
@pytest.mark.parametrize("case", COATT_CASES, ids=[c[0] for c in COATT_CASES])
def test_coattention(case, prec):
    from fpnmt.engine import coattention
    name, HW, C, kind = case
    N = 2
    g = gen(HW * 3 + C)
    if kind == "spread":
        score = (torch.rand(N, HW, generator=g) * 2 - 1) * 80          # weights from 1 down to far below fp32's range
    else:
        score = torch.full((N, HW), 3.7)
    cls = torch.randn(N, HW, C, generator=g) * 2
    out = torch.full((N, HW, C), float("nan")).cuda()
    y = coattention(score.cuda(), cls.cuda(), out, prec).cpu()
    sq, cq = q_act(score, prec).double(), q_act(cls, prec).double()
    ref = O.coattention_cnn(sq.unsqueeze(-1), cq)
    # __expf: ex2.approx of (s - max) * log2(e) rounded to fp32, an error of ~2^-24 |s - max| <= 2^-16.5 for |s - max| <= 160;
    # weights below fp32's normal range are flushed to zero (the floor, 2^-120 absolute)
    check_elementwise("coattention/" + prec, y, ref, ref.abs(), RTOL[prec], 2.0 ** -16, floor=2.0 ** -120)


# ------------------------------------------------------------------------------------------------------------------------
# encoder token pre-amble: one warp per 512-wide row (8 rows per block), LayerNorm + positional table
TLN_CASES = [(3, 1), (3, 4), (3, 16), (2, 64), (1, 256), (1, 1024), (5, 4)]


@pytest.mark.parametrize("prec", PRECS)
@pytest.mark.parametrize("shape", TLN_CASES, ids=["n%d_hw%d" % s for s in TLN_CASES])
def test_tokens_ln_pos(shape, prec):
    from fpnmt.engine import tokens_ln_pos
    N, HW = shape
    rows = N * HW
    g = gen(rows * 11 + HW)
    x = torch.randn(rows, 512, generator=g) * 2 + 0.5
    x[::3] = 100 + torch.randn(x[::3].shape, generator=g) * 1e-2      # large mean, small spread
    gamma = (torch.rand(512, generator=g) + 0.5).numpy()
    beta = (torch.randn(512, generator=g) * 0.1).numpy()
    pos = O.raw_positional_encoding(HW, 512).numpy()
    y = tokens_ln_pos(x.cuda(), HW, gamma, beta, pos, 1e-6, torch.full((rows, 512), float("nan")).cuda(), prec).cpu()
    xq = q_act(x, prec).double()
    gd, bd = torch.from_numpy(gamma).double(), torch.from_numpy(beta).double()
    posd = torch.from_numpy(pos).double().repeat(N, 1)
    ln = O.layer_norm(xq, gd, bd, 1e-6)
    mean, var = xq.mean(-1, keepdim=True), xq.var(-1, unbiased=False, keepdim=True)
    # summands LN + pos; the kernel's fp32 mean carries an error of ~2^-24 |mean| per addition, which LN divides by the
    # row's standard deviation: the |gamma| |mean| / std term (1e4 on the mean-100 rows in bf16x3)
    scale = ln.abs() + posd.abs() + gd.abs() * mean.abs() / torch.sqrt(var + 1e-6)
    check_elementwise("tokens_ln_pos/" + prec, y, ln + posd, scale, RTOL[prec], 2.0 ** -19)


# ------------------------------------------------------------------------------------------------------------------------
# encoder cross-level attention.  Tensor-core path (bf16): one block per (image, head[, view]), warp w walks the 64-key
# tiles w, w+4, ... with an online softmax and the four warps merge at the end - above 256 keys a warp rescales its
# accumulator, below 64 three warps have no tile.  CUDA-core path (bf16x3, or force_simt): fp32 flash-style over chunks of
# 32 keys.
ATT_MODES = [("mma", "bf16", False), ("simt", "bf16", True), ("simt", "bf16x3", False)]


def _att_inputs(B, Tq, tks, heads, kv_ld, k_col, v_col, g):
    """q (B*Tq, nviews*heads*64) and per view K/V (B*Tk, kv_ld) (columns outside [k_col | v_col] NaN).  Every query of an
    (image, view, head) shares a direction u; the last key of the view is u scaled so that its score leads the others by
    about 3-4: the maximum sits in the last tile (for Tk > 256 the second tile of its warp)."""
    nv, w = len(tks), heads * 64
    u = torch.randn(B, nv, heads, 64, generator=g)
    q = (2 * u.unsqueeze(1) + 0.5 * torch.randn(B, Tq, nv, heads, 64, generator=g)).reshape(B * Tq, nv * w)
    kvs = []
    for v, tk in enumerate(tks):
        kv = torch.full((B, tk, kv_ld), float("nan"))
        k = torch.randn(B, tk, heads, 64, generator=g)
        k[:, -1] = 0.6 * u[:, v]
        kv[..., k_col:k_col + w] = k.reshape(B, tk, w)
        kv[..., v_col:v_col + w] = torch.randn(B, tk, w, generator=g)
        kvs.append(kv.reshape(B * tk, kv_ld))
    return q, kvs


def _att_check(op, mode, prec, y, q, kvs, B, Tq, heads, k_col, v_col):
    w = heads * 64
    assert bool(torch.isfinite(y).all()), "%s: non-finite outputs (never written?)" % op
    qq = q_act(q, prec).double().reshape(B, Tq, len(kvs), heads, 64)
    for v, kv in enumerate(kvs):
        tk = kv.shape[0] // B
        kq = q_act(kv, prec).double().reshape(B, tk, -1)
        k = kq[..., k_col:k_col + w].reshape(B, tk, heads, 64).transpose(1, 2)
        vv = kq[..., v_col:v_col + w].reshape(B, tk, heads, 64).transpose(1, 2)
        ref, p = O.scaled_dot_product_attention(qq[:, :, v].transpose(1, 2), k, vv, None)     # (B, heads, Tq, 64)
        yv = y.double().reshape(B, Tq, len(kvs), heads, 64)[:, :, v].transpose(1, 2)
        if mode == "mma":
            for h in range(heads):
                r = float((yv[:, h] - ref[:, h]).norm() / ref[:, h].norm())
                _record(op, r, 8e-3)
                assert r <= 8e-3, "%s: view %d (Tk %d) head %d rel-L2 %.3g" % (op, v, tk, h, r)
        else:
            # fp32 scores of 64-term products (~2^-24 * 64 of |q||k| / 8 each) move p by a relative ~2^-15
            check_elementwise(op, yv, ref, p @ vv.abs(), RTOL[prec], 2.0 ** -15)


ATT_TQ = [1, 4, 16]
ATT_TK = [1, 4, 16, 63, 64, 65, 256, 257, 1024]


@pytest.mark.parametrize("mode,prec,simt", ATT_MODES, ids=["%s_%s" % (m[0], m[1]) for m in ATT_MODES])
@pytest.mark.parametrize("tk", ATT_TK)
@pytest.mark.parametrize("tq", ATT_TQ)
def test_enc_attention_one_view(tq, tk, mode, prec, simt):
    from fpnmt.engine import enc_attention
    B, heads, kv_ld, k_col, v_col = 2, 2, 256, 0, 128
    g = gen(tq * 5000 + tk)
    q, kvs = _att_inputs(B, tq, [tk], heads, kv_ld, k_col, v_col, g)
    y = enc_attention(q.cuda(), [t.cuda() for t in kvs], B, heads, k_col, v_col, simt,
                      torch.full(q.shape, float("nan")).cuda(), prec).cpu()
    _att_check("enc_attention_%s/%s" % (mode, prec), mode, prec, y, q, kvs, B, tq, heads, k_col, v_col)


# the engine's view sets: image 512 -> P3, P4, P5, P7 tokens {1024, 256, 64, 4} with the 16 P6 tokens as queries; image 256 ->
# {256, 64, 16, 1} with 4 queries.  K/V of the last layer of a 6-layer hoisted projection (kv_ld = 6 * 2 * 512).
VIEW_SETS = [("image512", 16, [1024, 256, 64, 4]), ("image256", 4, [256, 64, 16, 1])]


@pytest.mark.parametrize("mode,prec,simt", ATT_MODES, ids=["%s_%s" % (m[0], m[1]) for m in ATT_MODES])
@pytest.mark.parametrize("vs", VIEW_SETS, ids=[v[0] for v in VIEW_SETS])
def test_enc_attention_engine_views(vs, mode, prec, simt):
    from fpnmt.engine import enc_attention
    _, tq, tks = vs
    B, heads, kv_ld, k_col, v_col = 2, 8, 6144, 5 * 1024, 5 * 1024 + 512
    g = gen(tq * 7 + len(tks))
    q, kvs = _att_inputs(B, tq, tks, heads, kv_ld, k_col, v_col, g)
    y = enc_attention(q.cuda(), [t.cuda() for t in kvs], B, heads, k_col, v_col, simt,
                      torch.full(q.shape, float("nan")).cuda(), prec).cpu()
    _att_check("enc_attention_%s_views/%s" % (mode, prec), mode, prec, y, q, kvs, B, tq, heads, k_col, v_col)


@pytest.mark.parametrize("nviews", [1, 4])
@pytest.mark.parametrize("mode,prec,simt", ATT_MODES, ids=["%s_%s" % (m[0], m[1]) for m in ATT_MODES])
def test_enc_attention_rejects_tq17(mode, prec, simt, nviews):
    from fpnmt._lib import ERR_INVALID, FpnmtError
    from fpnmt.engine import enc_attention
    B, heads = 1, 1
    q = torch.zeros(B * 17, nviews * heads * 64).cuda()
    kvs = [torch.zeros(B * 4, 128).cuda() for _ in range(nviews)]
    with pytest.raises(FpnmtError) as e:
        enc_attention(q, kvs, B, heads, 0, 64, simt, precision=prec)
    assert e.value.code == ERR_INVALID
