"""The 16-bit tensor-core convolutions (csrc/conv_tc.cu) against float64 references.

Exact tests: integer activations, weights and biases and offsets on a 1/4 grid.  Every product is then a multiple of a
quantum q (1, or 1/16 for bilinear samples), and check_budget asserts max(S) / q <= 2**20 for S = the same operation
on |inputs|, so every partial sum is an exact fp32 value in any order.  The kernel's output must then be bit-identical
to the float64 reference rounded ONCE (tc_reference.round_rne; torch's float64 -> 16-bit conversion rounds twice).
For the deformable kernels the 16-bit bilinear blend must be exact as well: its partial sums are multiples of 1/16 no
larger than max|x|, so max|x| * 16 <= 2**p (p = 8 for bf16, 11 for fp16) is asserted.

Rounding-model tests: normal data, where the blend rounds.  The reference is the float64 contraction of
tc_reference.emulate_samples (the A operand modelled rounding for rounding), so what remains is fp32 accumulation and
the final rounding: |y - ref| <= ulp/2 + E with E = 2 * 9C * 2**-24 * S for every element, and a bounded share of
outputs that differ from round_rne(ref).
"""
import pytest
import torch
import torch.nn.functional as F

from s2anet_b200 import synth
from tc_reference import (FORMATS, align_offsets, assert_exact, check_budget, contract_samples, deform_grads_ref, dyadic_anchors,
                          emulate_samples, ints, quarter_offsets, round_rne, sampling_positions, ulp)

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
BF16, F16 = torch.bfloat16, torch.float16
DTYPES = [BF16, F16]
# |x| and |w| bounds of the integer data
RANGES = {BF16: (8, 3), F16: (4, 2)}
LEVELS = ((1, 1), (1, 17), (9, 1), (7, 15), (9, 33))
BENCH_LEVELS = ((128, 128), (64, 64), (32, 32), (16, 16), (8, 8))
BENCH_STRIDES = (8, 16, 32, 64, 128)
# Largest share of outputs != round_rne(ref) allowed in the rounding-model tests: 3x the share measured on one B200
# (1,000 W limit) with these seeds -- fp16 with rounded positions 0.548 % / 0.558 % (fp32 / fp16 offsets), bf16 with
# fp32 positions 0.056 % / 0.051 %.
MISMATCH_LIMIT = {(F16, True): 0.017, (BF16, False): 0.0017}


def tv():
    return pytest.importorskip("torchvision")


def cl(t, dtype):
    return t.to(DEV).to(dtype).contiguous(memory_format=torch.channels_last)


def assert_exact_blend(x, dtype, what):
    """The 16-bit bilinear blend of integer data with 1/4-grid weights is exact: partial sums are multiples of 1/16 of
    magnitude <= max|x|."""
    p = FORMATS[dtype][0]
    assert bool((x.double() == x.double().round()).all()), "%s: activations must be integers" % what
    assert float(x.double().abs().max()) * 16 <= 2 ** p, "%s: activations too large for an exact 16-bit blend" % what


def assert_quarter_grid(off, what):
    assert bool((off.double() * 4 == (off.double() * 4).round()).all()), "%s: offsets must lie on a 1/4 grid" % what


# ------------------------------------------------------------------------------------------------------------------
# plain convolutions: conv2d_forward_tc_multi, conv2d_forward_tc_pair, orconv_forward_tc_multi
# ------------------------------------------------------------------------------------------------------------------
def plain_ref(x, w, b, relu):
    ks = w.size(-1)
    x64, w64 = x.double(), w.to(x.device).double()
    ref = F.conv2d(x64, w64, None if b is None else b.to(x.device).double(), padding=ks // 2)
    S = F.conv2d(x64.abs(), w64.abs(), None if b is None else b.to(x.device).double().abs(), padding=ks // 2)
    return (ref.relu() if relu else ref), S


def check_plain(entry, dtype, xs, w, b, relu, ys):
    for l, (x, y) in enumerate(zip(xs, ys)):
        ref, S = plain_ref(x, w, b, relu)
        what = "%s %s level %d (%dx%d)" % (entry, dtype, l, x.size(2), x.size(3))
        check_budget(S, 1.0, dtype, ref, what)
        assert tuple(y.shape) == tuple(ref.shape) and y.dtype == dtype
        assert_exact(y, ref, what)


def plain_case(dtype, B, C, Co, ks, sizes, bias, seed):
    g = torch.Generator().manual_seed(seed)
    xr, wr = RANGES[dtype]
    xs = [cl(ints((B, C, h, w), xr, g), dtype) for h, w in sizes]
    wt = ints((Co, C, ks, ks), wr, g).to(DEV).to(dtype)
    b = ints((Co,), 16, g).float().to(DEV) if bias else None
    return xs, wt, b


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("C,Co,ks,relu,bias", [(8, 32, 3, True, True), (24, 5, 1, False, True), (32, 256, 3, True, True),
                                               (72, 40, 3, False, False), (256, 15, 3, False, True), (256, 5, 1, False, True),
                                               (320, 32, 3, True, False), (512, 96, 1, False, True), (512, 256, 3, True, True),
                                               (256, 96, 3, False, True)])
def test_conv2d_tc_multi_exact(dtype, C, Co, ks, relu, bias):
    """PLAIN / PLAIN_S / 1x1: partial last k-blocks (C % 64), padded output channels, partial and degenerate tiles."""
    from s2anet_b200.conv_tc import conv2d_forward_tc_multi
    xs, wt, b = plain_case(dtype, 2, C, Co, ks, LEVELS, bias, C * 7 + Co + ks)
    check_plain("conv2d_forward_tc_multi", dtype, xs, wt, b, relu, conv2d_forward_tc_multi(xs, wt, b, relu=relu))


@pytest.mark.parametrize("Co,ks", [(64, 3), (15, 3), (40, 1)])
def test_conv2d_tc_multi_exact_many_tiles(Co, ks):
    """405 tiles (odd: a ghost tile) on 148 SMs: the rings and accumulators carry across several tiles per CTA."""
    from s2anet_b200.conv_tc import conv2d_forward_tc_multi
    xs, wt, b = plain_case(BF16, 3, 64, Co, ks, ((136, 120),), True, Co + ks)
    check_plain("conv2d_forward_tc_multi", BF16, xs, wt, b, True, conv2d_forward_tc_multi(xs, wt, b, relu=True))


@pytest.mark.parametrize("dtype,Co,ks,relu", [(BF16, 256, 3, True), (F16, 256, 3, True), (BF16, 15, 3, False),
                                              (BF16, 5, 1, False)])
def test_conv2d_tc_multi_exact_bench_levels(dtype, Co, ks, relu):
    """The five FPN levels of the benchmark (1024^2 images: 128^2 .. 8^2) at batch 2 in one launch."""
    from s2anet_b200.conv_tc import conv2d_forward_tc_multi
    xs, wt, b = plain_case(dtype, 2, 256, Co, ks, BENCH_LEVELS, True, Co + ks + 1)
    check_plain("conv2d_forward_tc_multi", dtype, xs, wt, b, relu, conv2d_forward_tc_multi(xs, wt, b, relu=relu))


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("Co0,Co1,ks", [(256, 256, 3), (15, 5, 1), (15, 5, 3), (32, 32, 3)])
def test_conv2d_tc_pair_exact(dtype, Co0, Co1, ks):
    """Both problems of the paired launch against float64: 15 tiles per problem (odd: a padding tile before the second
    problem), separate and shared inputs, and the fallback to two launches (256 vs 32 input channels)."""
    from s2anet_b200.conv_tc import conv2d_forward_tc_pair
    sizes = ((24, 40), (13, 21), (3, 5), (9, 1))
    xs0, w0, b0 = plain_case(dtype, 1, 128, Co0, ks, sizes, True, Co0 + ks)
    xs1, w1, b1 = plain_case(dtype, 1, 128, Co1, ks, sizes, True, Co1 + ks + 100)
    for a, c in ((xs0, xs1), (xs0, xs0)):
        o0, o1 = conv2d_forward_tc_pair(a, w0, b0, c, w1, b1, relu=True)
        check_plain("conv2d_forward_tc_pair[0]", dtype, a, w0, b0, True, o0)
        check_plain("conv2d_forward_tc_pair[1]", dtype, c, w1, b1, True, o1)
    xs2, w2, b2 = plain_case(dtype, 1, 32, Co1, ks, sizes, True, 5)
    xs3, w3, b3 = plain_case(dtype, 1, 256, Co0, ks, sizes, True, 6)
    o3, o2 = conv2d_forward_tc_pair(xs3, w3, b3, xs2, w2, b2, relu=False)
    check_plain("conv2d_forward_tc_pair[0] (two launches)", dtype, xs3, w3, b3, False, o3)
    check_plain("conv2d_forward_tc_pair[1] (two launches)", dtype, xs2, w2, b2, False, o2)


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("I,O", [(256, 32), (64, 4), (128, 16)])
def test_orconv_tc_multi_exact(dtype, I, O):
    """ORConv2d (8 rotations of an integer bank through the ARF map) with the fused 8-way orientation max."""
    from s2anet_b200.conv_tc import orconv_forward_tc_multi
    from s2anet_b200.orn import ORConv2d
    g = torch.Generator().manual_seed(I + O)
    xr, wr = RANGES[dtype]
    m = ORConv2d(I, O, 3, padding=1, arf_config=(1, 8)).to(DEV)
    with torch.no_grad():
        m.weight.copy_(ints(m.weight.shape, wr, g))
        m.bias.copy_(ints((O * 8,), 16, g))
        arf = m.rotate_arf().detach()                                   # [O*8, I, 3, 3], integers: exact in fp32
    B = 2
    xs = [cl(ints((B, I, h, w), xr, g), dtype) for h, w in LEVELS + ((40, 24),)]
    outs, pooled = orconv_forward_tc_multi(xs, m.weight.to(dtype), m.indices, m.bias, with_pool=True)
    check_plain("orconv_forward_tc_multi", dtype, xs, arf, m.bias.detach(), False, outs)
    for l, (x, p) in enumerate(zip(xs, pooled)):
        ref, _ = plain_ref(x, arf, m.bias.detach(), False)
        assert_exact(p, ref.view(B, O, 8, x.size(2), x.size(3)).max(dim=2)[0],
                     "orconv_forward_tc_multi pooled %s level %d" % (dtype, l))


# ------------------------------------------------------------------------------------------------------------------
# deformable convolutions: AlignConv, the generic deformable conv, its backward
# ------------------------------------------------------------------------------------------------------------------
def deform_ref(x, off, w, relu):
    """float64 torchvision deform_conv2d (+ ReLU) and the same on |x|, |w| (the budget)."""
    x64, off64, w64 = x.double(), off.to(x.device).double(), w.to(x.device).double()
    ref = tv().ops.deform_conv2d(x64, off64, w64, padding=1)
    S = tv().ops.deform_conv2d(x64.abs(), off64, w64.abs(), padding=1)
    return (ref.relu() if relu else ref), S


def check_align(entry, dtype, x, anc, w, stride, y, what):
    off = align_offsets(anc.double(), x.size(2), x.size(3), stride)
    assert_quarter_grid(off, what)
    assert_exact_blend(x, dtype, what)
    ref, S = deform_ref(x, off, w, True)
    check_budget(S, 1 / 16, dtype, ref, what)
    assert_exact(y, ref, what)


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("C,Co", [(64, 32), (256, 256), (128, 96)])
def test_alignconv_tc_multi_exact(dtype, C, Co):
    from s2anet_b200.conv_tc import alignconv_forward_tc, alignconv_forward_tc_multi
    g = torch.Generator().manual_seed(C + Co)
    xr, wr = RANGES[dtype]
    sizes, strides = LEVELS + ((13, 21),), (8, 16, 32, 64, 128, 8)
    B = 2
    xs = [cl(ints((B, C, h, w), xr, g), dtype) for h, w in sizes]
    ancs = [dyadic_anchors(B, h, w, s, g) for (h, w), s in zip(sizes, strides)]
    wt = ints((Co, C, 3, 3), wr, g).to(DEV).to(dtype)
    ys = alignconv_forward_tc_multi(xs, [a.float().to(DEV) for a in ancs], wt, strides)
    for l, (x, a, s, y) in enumerate(zip(xs, ancs, strides, ys)):
        check_align("alignconv_forward_tc_multi", dtype, x, a, wt, s, y,
                    "alignconv_forward_tc_multi %s level %d (%dx%d)" % (dtype, l, x.size(2), x.size(3)))
    y1 = alignconv_forward_tc(xs[-1], ancs[-1].float().to(DEV), wt, strides[-1])
    check_align("alignconv_forward_tc", dtype, xs[-1], ancs[-1], wt, strides[-1], y1, "alignconv_forward_tc %s" % dtype)


@pytest.mark.parametrize("dtype", DTYPES)
def test_alignconv_tc_multi_exact_bench_levels(dtype):
    from s2anet_b200.conv_tc import alignconv_forward_tc_multi
    g = torch.Generator().manual_seed(11)
    xr, wr = RANGES[dtype]
    B, C, Co = 2, 256, 256
    xs = [cl(ints((B, C, h, w), xr, g), dtype) for h, w in BENCH_LEVELS]
    ancs = [dyadic_anchors(B, h, w, s, g) for (h, w), s in zip(BENCH_LEVELS, BENCH_STRIDES)]
    wt = ints((Co, C, 3, 3), wr, g).to(DEV).to(dtype)
    ys = alignconv_forward_tc_multi(xs, [a.float().to(DEV) for a in ancs], wt, BENCH_STRIDES)
    for l, (x, a, s, y) in enumerate(zip(xs, ancs, BENCH_STRIDES, ys)):
        check_align("alignconv_forward_tc_multi", dtype, x, a, wt, s, y,
                    "alignconv_forward_tc_multi %s bench level %d" % (dtype, l))


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("round_positions", [False, True])
@pytest.mark.parametrize("B,C,H,W,Co", [(2, 64, 9, 33, 32), (2, 192, 7, 15, 96), (1, 128, 1, 17, 256), (2, 64, 9, 1, 64),
                                        (2, 128, 20, 36, 128)])
def test_deform_conv_tc_exact(dtype, round_positions, B, C, H, W, Co):
    """Explicit offsets (fp32 and 16-bit), positions exactly on -1, on H - 1 / W - 1, integer positions (lx = 0 with the
    right corner past the edge), just inside -1 and in (W - 1, W); ReLU on and off."""
    from s2anet_b200.conv_tc import deform_conv_forward_tc
    g = torch.Generator().manual_seed(B * 1000 + C + H + W + Co + round_positions)
    xr, wr = RANGES[dtype]
    x = cl(ints((B, C, H, W), xr, g), dtype)
    wt = ints((Co, C, 3, 3), wr, g).to(DEV).to(dtype)
    off = quarter_offsets(B, H, W, g)
    h, w = sampling_positions(off)
    assert (h == -1).any() and (h == -0.75).any() and (h == H - 1).any() and ((w > W - 1) & (w < W)).any()
    if round_positions:
        assert float(torch.maximum(h.abs(), w.abs()).max()) * 4 <= 2 ** FORMATS[dtype][0], "positions not exact in 16 bits"
    what = "deform_conv_forward_tc %s round_positions=%d %dx%d" % (dtype, round_positions, H, W)
    assert_exact_blend(x, dtype, what)
    for relu in (False, True):
        ref, S = deform_ref(x, off, wt, relu)
        check_budget(S, 1 / 16, dtype, ref, what)
        for od in (torch.float32, dtype):
            y = deform_conv_forward_tc(x, off.to(DEV).to(od), wt, relu=relu, round_positions=round_positions)
            assert_exact(y, ref, "%s relu=%d offsets %s" % (what, relu, od))


@pytest.mark.parametrize("dtype", DTYPES)
def test_deform_conv_forward_cuda_half_exact(dtype):
    """The reference-signature entry with 16-bit tensors (NCHW in, NCHW out) routes to the tcgen05 kernel."""
    from s2anet_b200 import dcn
    g = torch.Generator().manual_seed(21)
    xr, wr = RANGES[dtype]
    B, C, H, W, Co = 2, 64, 12, 20, 64
    x = ints((B, C, H, W), xr, g).to(DEV).to(dtype)
    wt = ints((Co, C, 3, 3), wr, g).to(DEV).to(dtype)
    off = quarter_offsets(B, H, W, g)
    out = x.new_empty((B, Co, H, W))
    dcn.deform_conv_forward_cuda(x, wt, off.to(DEV).to(dtype), out, x.new_empty(0), x.new_empty(0), 3, 3, 1, 1, 1, 1, 1, 1,
                                 1, 1, 1)
    ref, S = deform_ref(x, off, wt, False)
    check_budget(S, 1 / 16, dtype, ref, "deform_conv_forward_cuda %s" % dtype)
    assert_exact(out, ref, "deform_conv_forward_cuda %s" % dtype)


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("C,Co,H,W,goff", [(128, 128, 9, 33, True), (256, 64, 13, 21, True), (96, 128, 7, 15, True),
                                           (256, 256, 16, 24, False)])
def test_deform_conv_dgrad_tc_exact(dtype, C, Co, H, W, goff):
    """grad_input and grad_offset (fp32, scattered with atomics) equal the float64 autograd reference exactly; the
    offsets put sampling positions exactly on -1, where the offset gradient follows the reference DCN's rule (0)."""
    from s2anet_b200.conv_tc import deform_conv_dgrad_tc
    g = torch.Generator().manual_seed(C + Co + H)
    B = 2
    x = ints((B, C, H, W), 2, g).to(DEV).to(dtype)
    go = ints((B, Co, H, W), 2, g).to(DEV).to(dtype)
    wt = ints((Co, C, 3, 3), 1, g).to(DEV).to(dtype)
    off = quarter_offsets(B, H, W, g)
    gi_ref, goff_ref, _ = deform_grads_ref(x, off, wt, go)
    gi_S, _, _ = deform_grads_ref(x.abs(), off, wt.abs(), go.abs())
    what = "deform_conv_dgrad_tc %s C=%d Co=%d %dx%d" % (dtype, C, Co, H, W)
    check_budget(gi_S, 1 / 16, what=what + " grad_input")
    if goff:    # gy = hx (D3 - D1) + lx (D4 - D2), D = sum_c col_grad[c] x[c]: |gy| <= 2 max|D|, quantum 1/4
        check_budget(torch.tensor([2.0 * C * Co * 2 * 1 * 2]), 1 / 4, what=what + " grad_offset")
    for od in (torch.float32, dtype):
        gi, gof = deform_conv_dgrad_tc(go, off.to(DEV).to(od), wt, x=x, need_offset_grad=goff)
        assert_exact(gi, gi_ref, "%s offsets %s grad_input" % (what, od))
        if goff:
            assert_exact(gof, goff_ref, "%s offsets %s grad_offset" % (what, od))


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("C,Co,H,W", [(128, 128, 9, 33), (256, 128, 13, 21), (128, 256, 7, 15), (256, 256, 20, 36)])
def test_deform_conv_wgrad_tc_exact(dtype, C, Co, H, W):
    """grad_weight (fp32, accumulated over tiles with atomics) equals torchvision's float64 autograd exactly."""
    from s2anet_b200.conv_tc import deform_conv_wgrad_tc
    g = torch.Generator().manual_seed(C + 2 * Co + W)
    B = 2
    xr = RANGES[dtype][0]
    x = ints((B, C, H, W), xr, g).to(DEV).to(dtype)
    go = ints((B, Co, H, W), 2, g).to(DEV).to(dtype)
    wt = ints((Co, C, 3, 3), 1, g).to(DEV).to(dtype)
    off = quarter_offsets(B, H, W, g)
    what = "deform_conv_wgrad_tc %s C=%d Co=%d %dx%d" % (dtype, C, Co, H, W)
    assert_exact_blend(x, dtype, what)
    _, _, gw_ref = deform_grads_ref(x, off, wt, go)
    _, _, gw_S = deform_grads_ref(x.abs(), off, wt, go.abs())
    check_budget(gw_S, 1 / 16, what=what)
    for od in (torch.float32, dtype):
        assert_exact(deform_conv_wgrad_tc(x, off.to(DEV).to(od), go), gw_ref, "%s offsets %s" % (what, od))


# ------------------------------------------------------------------------------------------------------------------
# rounding model: normal data
# ------------------------------------------------------------------------------------------------------------------
def check_rounding_model(y, samples, wt, dtype, relu, what):
    """|y - ref| <= max(ulp(ref), ulp(y)) / 2 + E everywhere, E = 2 * 9C * 2**-24 * S; returns the share of outputs
    that differ from round_rne(ref)."""
    C = samples.size(-1)
    ref = contract_samples(samples, wt)
    S = contract_samples(samples.abs(), wt.abs())
    if relu:
        ref = ref.relu()
    E = 2.0 * 9 * C * 2.0 ** -24 * S
    y64 = y.double()
    err = (y64 - ref).abs()
    bound = torch.maximum(ulp(ref, dtype), ulp(y64, dtype)) / 2 + E
    bad = err > bound
    if bad.any():
        i = bad.nonzero()[0].tolist()
        raise AssertionError("%s: %d outputs outside ulp/2 + E; first (b, y, x, c)=(%d, %d, %d, %d): got %r, ref %r, bound %r"
                             % (what, int(bad.sum()), i[0], i[2], i[3], i[1], float(y64[tuple(i)]), float(ref[tuple(i)]),
                                float(bound[tuple(i)])))
    return float((y != round_rne(ref, dtype)).double().mean())


@pytest.mark.parametrize("dtype,round_positions", [(F16, True), (BF16, False)])
@pytest.mark.parametrize("off16", [False, True])
def test_deform_conv_tc_rounding_model(dtype, round_positions, off16):
    """Random offsets N(0, 1.5): the kernel against the float64 contraction of its modelled A operand."""
    from s2anet_b200.conv_tc import deform_conv_forward_tc
    g = torch.Generator().manual_seed(31 + off16)
    B, C, H, W, Co = 2, 128, 24, 40, 64
    x = torch.randn(B, C, H, W, generator=g).to(DEV).to(dtype)
    wt = (torch.randn(Co, C, 3, 3, generator=g) * 0.05).to(DEV).to(dtype)
    off = (torch.randn(B, 18, H, W, generator=g) * 1.5).to(DEV)
    if off16:
        off = off.to(dtype)
    y = deform_conv_forward_tc(x, off, wt, round_positions=round_positions)
    samples = emulate_samples(x, off, dtype, round_positions)
    what = "deform_conv_forward_tc %s round_positions=%d offsets %s" % (dtype, round_positions, off.dtype)
    rate = check_rounding_model(y, samples, wt, dtype, False, what)
    print("\n%s: %.4f %% of outputs differ from round_rne(ref)" % (what, 100 * rate))
    assert rate <= MISMATCH_LIMIT[(dtype, round_positions)], "%s: mismatch share %.4f" % (what, rate)


def test_alignconv_rotated_matches_deform_route():
    """Rotated anchors at a benchmark level (64 x 64, stride 16): AlignConv's in-kernel offsets, recomputed with torch
    fp32 ops in the kernel's operation order, fed to the generic deformable kernel.  Both kernels then share every later
    operation, so nearly all outputs agree bit for bit; the rest must satisfy the rounding-model bound.  (Whether torch's
    CUDA cos / sin equal the kernel's cosf / sinf bit for bit is not assumed: disagreements are counted.)"""
    from s2anet_b200.conv_tc import alignconv_forward_tc, deform_conv_forward_tc
    dtype = BF16
    g = torch.Generator().manual_seed(41)
    B, C, H, W, Co, stride = 2, 256, 64, 64, 256, 16
    x = cl(torch.randn(B, C, H, W, generator=g), dtype)
    wt = (torch.randn(Co, C, 3, 3, generator=g) * 0.05).to(DEV).to(dtype)
    anc = torch.from_numpy(synth.refined_anchors(B, H, W, stride, seed=6)).to(DEV).float()
    ax, ay, aw, ah = (anc[..., k] / stride for k in range(4))
    cs, sn = torch.cos(anc[..., 4]), torch.sin(anc[..., 4])
    dw, dh = aw / 3.0, ah / 3.0
    yy = torch.arange(H, device=DEV, dtype=torch.float32).view(1, H, 1)
    xx = torch.arange(W, device=DEV, dtype=torch.float32).view(1, 1, W)
    off = torch.empty(B, 18, H, W, device=DEV)
    for t in range(9):
        fi, fj = float(t // 3 - 1), float(t % 3 - 1)
        txx, tyy = dw * fj, dh * fi
        xr = cs * txx - sn * tyy
        yr = sn * txx + cs * tyy
        xa, ya = xr + ax, yr + ay
        off[:, 2 * t] = ya - (yy + fi)
        off[:, 2 * t + 1] = xa - (xx + fj)
    ya_ = alignconv_forward_tc(x, anc, wt, stride)
    yd = deform_conv_forward_tc(x, off, wt, relu=True, round_positions=False)
    differ = ya_ != yd
    n = int(differ.sum())
    print("\nrotated AlignConv vs deformable route: %d of %d outputs differ" % (n, differ.numel()))
    assert n <= 1e-3 * differ.numel(), "%d of %d outputs differ" % (n, differ.numel())
    if n:
        check_rounding_model(ya_, emulate_samples(x, off, dtype, False), wt, dtype, True, "alignconv_forward_tc rotated")
