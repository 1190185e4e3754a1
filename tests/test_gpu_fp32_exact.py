"""The fp32 convolutions against float64, bit for bit: the 3 x TF32 tensor-core kernel (conv_tc.cu conv_tf32x3_kernel and
its weight packer), the SIMT kernel (conv_f32.cu conv_gather_f32_kernel), the fp32 deformable backward
(deform_bwd.cu + the GEMMs of dcn.py) and the ARF backward (orn.cu).

"Exact" means torch.equal with the float64 result, which assert_exact first checks is an fp32 value.  The data keep
every partial sum exact: integers, offsets on a 1/4 grid (samples are multiples of 1/16) and check_budget's
max(S) / q <= 2**20, which also absorbs the tensor core's truncating additions.

The TF32 split is pinned by three data regimes:
* A: integers.  Samples and weights are TF32 values, so lo == 0 on both sides.
* B: low parts on one side.  x (or w) = +-(1 + odd 2**-11), a TF32 tie with lo = +-2**-11; the other side in
  {-1, 0, 1}; samples are copies of x (integer positions).  The output is exact only if both correction MMAs run.
* C: low parts on both sides and one product per output (one-hot weights).  The kernel computes a*w - a_lo*w_lo with
  the rna split of tc_reference.tf32_split, exactly; that differs from a*w at every nonzero output.
The float64 references run on the GPU (torchvision's deform_conv2d and F.conv2d accept float64 CUDA tensors).
"""
import math

import pytest
import torch
import torch.nn.functional as F

from tc_reference import (align_offsets, assert_exact, check_budget, deform_grads_ref, dyadic_anchors, geom_offsets,
                          geom_positions, ints, odd_fractions, out_size, quarter_offsets, round_rne, tf32_round,
                          tf32_split)

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
MAPS = ((1, 1), (1, 17), (9, 1), (13, 21))
STRIDES = (8, 16, 32, 64)
BENCH_LEVELS = ((128, 128), (64, 64), (32, 32), (16, 16), (8, 8))
BENCH_STRIDES = (8, 16, 32, 64, 128)
Q11 = 2.0 ** -11
# Largest share of rotated-anchor outputs where mode 0 and mode 1 may differ: 3x the share measured on one B200
# (1,000 W limit) with this seed, 9.2 %.
ROTATED_DIFFER_LIMIT = 0.28


def tv():
    return pytest.importorskip("torchvision")


def sm_count():
    return torch.cuda.get_device_properties(DEV).multi_processor_count


@pytest.fixture
def simt():
    """Route fp32 AlignConv / DeformConv / ORConv2d to the SIMT kernel; restore the previous route afterwards."""
    from s2anet_b200 import alignconv
    old = alignconv._FORCE_SIMT_F32
    alignconv.set_fp32_path("simt")
    yield
    alignconv._FORCE_SIMT_F32 = old


@pytest.fixture
def fp32_matmul():
    """The backward's GEMMs in full fp32 (no TF32), as the reference's SGEMMs; restored afterwards."""
    old = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = False
    yield
    torch.backends.cuda.matmul.allow_tf32 = old


def f32bits(t):
    return t.to(torch.float32).contiguous().view(torch.int32)


def dev32(t):
    return t.to(torch.float32).to(DEV)


def arf_bank(weight, indices):
    from s2anet_b200.orn import arf_forward
    return arf_forward(weight.detach(), indices)        # pure data movement (test_gpu_conv checks it against the oracle)


# ------------------------------------------------------------------------------------------------------------------
# 1. the TF32 split of the weights: s2a_conv_pack_weight_tf32
# ------------------------------------------------------------------------------------------------------------------
def mixed_weights(shape, g):
    """Normal values over 40 binades, TF32 ties, subnormals and -0.0 / +0.0, element by element."""
    n = math.prod(shape)
    scale = torch.pow(2.0, torch.randint(-20, 21, (n,), generator=g).float())
    normal = torch.randn(n, generator=g) * scale
    ties = odd_fractions((n,), g).float() * scale
    sign = torch.where(torch.rand(n, generator=g) < 0.5, -1.0, 1.0)
    sub = torch.randint(1, 2 ** 23, (n,), generator=g, dtype=torch.int32).view(torch.float32) * sign
    zero = torch.where(sign < 0, torch.full((n,), -0.0), torch.zeros(n))
    kind = torch.randint(0, 4, (n,), generator=g)
    v = torch.where(kind == 0, normal, torch.where(kind == 1, ties, torch.where(kind == 2, sub, zero)))
    return v.view(shape)


def packed_ref(bank):
    """[Co, C, 3, 3] fp32 -> the model's (hi, lo) planes in the packed layout [Co][tap * C + c]."""
    Co, C = bank.shape[:2]
    return tf32_split(bank.permute(0, 2, 3, 1).reshape(Co, 9 * C))


def check_packed(hi, lo, bank, what):
    want_hi, want_lo = packed_ref(bank)
    assert hi.shape == want_hi.shape and lo.shape == want_lo.shape, what
    # the MMA reads hi as TF32 (it ignores the low 13 bits): lo is only right if hi has none
    assert bool(((f32bits(hi) & 0x1FFF) == 0).all()), "%s: hi has nonzero low 13 bits" % what
    assert bool(((f32bits(lo) & 0x1FFF) == 0).all()), "%s: lo has nonzero low 13 bits" % what
    for got, want, part in ((hi, want_hi, "hi"), (lo, want_lo, "lo")):
        bad = f32bits(got) != f32bits(want)
        if bad.any():
            i = bad.nonzero()[0].tolist()
            raise AssertionError("%s %s: %d of %d differ from the rna split model; first [co=%d, tap=%d, c=%d]: got %r, want %r"
                                 % (what, part, int(bad.sum()), bad.numel(), i[0], i[1] // bank.size(1),
                                    i[1] % bank.size(1), float(got[i[0], i[1]]), float(want[i[0], i[1]])))


def test_pack_weight_tf32_matches_the_split_model():
    """Plain [Co, C, 3, 3] weights: every element a normal value, a tie, a subnormal or a signed zero."""
    from s2anet_b200 import conv_tc
    g = torch.Generator().manual_seed(1)
    for Co, C in ((64, 96), (32, 32), (256, 256)):
        w = dev32(mixed_weights((Co, C, 3, 3), g))
        hi, lo = conv_tc.pack_weight_tf32(w)
        check_packed(hi, lo, w, "pack_weight_tf32 Co=%d C=%d" % (Co, C))
        assert bool((lo != 0).any()) and bool((f32bits(hi) != f32bits(w.permute(0, 2, 3, 1).reshape(Co, -1))).any())


@pytest.mark.parametrize("I,O,nOri", [(32, 32, 1), (4, 4, 8), (12, 28, 8)])
def test_pack_weight_tf32_orconv_bank(I, O, nOri):
    """ORConv2d banks [O, I, nOri, 3, 3] through the ARF map: the model applied to arf_forward(w)."""
    from s2anet_b200 import conv_tc
    from s2anet_b200.orn import ORConv2d
    g = torch.Generator().manual_seed(I + O + nOri)
    m = ORConv2d(I, O, 3, padding=1, arf_config=(nOri, 8)).to(DEV)
    w = dev32(mixed_weights(tuple(m.weight.shape), g))
    hi, lo = conv_tc.pack_weight_tf32(w, m.indices)
    check_packed(hi, lo, arf_bank(w, m.indices), "pack_weight_tf32 ORConv I=%d O=%d nOri=%d" % (I, O, nOri))


# ------------------------------------------------------------------------------------------------------------------
# 2. conv_forward_tf32x3: mode 0 anchors, 1 offsets, 2 regular grid
# ------------------------------------------------------------------------------------------------------------------
def integer_anchors(B, H, W, stride, g):
    """Angle-0 anchors whose nine tap positions are integers: centres on the pixel grid (moved up to +-3 pixels, some
    off the map), sizes 3 * stride * m (dw = m)."""
    yy, xx = torch.meshgrid(torch.arange(H).double(), torch.arange(W).double(), indexing="ij")
    a = torch.zeros(B, H, W, 5, dtype=torch.float64)
    a[..., 0] = (xx + ints((B, H, W), 3, g)) * stride
    a[..., 1] = (yy + ints((B, H, W), 3, g)) * stride
    a[..., 2] = torch.randint(0, 3, (B, H, W), generator=g).double() * 3 * stride
    a[..., 3] = torch.randint(0, 3, (B, H, W), generator=g).double() * 3 * stride
    return a


def tf32x3_aux(mode, B, H, W, stride, g, integer_positions):
    """The float64 aux tensor of a mode (None for the grid) and the float64 offsets the reference samples with."""
    if mode == 2:
        return None, None
    if mode == 1:
        off = ints((B, 18, H, W), 3, g) if integer_positions else quarter_offsets(B, H, W, g)
        return off, off
    anc = integer_anchors(B, H, W, stride, g) if integer_positions else dyadic_anchors(B, H, W, stride, g)
    off = align_offsets(anc, H, W, stride)
    assert bool((off * 4 == (off * 4).round()).all()), "anchor offsets off the 1/4 grid"
    return anc, off


def conv_ref(x, off, w, b, relu):
    """float64 conv (off None) or deformable conv (3x3, pad 1) on the GPU, + bias, + ReLU."""
    x64, w64 = x.to(DEV).double(), w.to(DEV).double()
    b64 = None if b is None else b.to(DEV).double()
    if off is None:
        ref = F.conv2d(x64, w64, b64, padding=1)
    else:
        ref = tv().ops.deform_conv2d(x64, off.to(DEV).double(), w64, bias=b64, padding=1)
    return ref.relu() if relu else ref


def run_tf32x3(mode, x, aux, w, bias, relu, pool, stride, layout, indices=None):
    from s2anet_b200 import conv_tc
    xin = dev32(x)
    if layout == "cl":
        xin = xin.contiguous(memory_format=torch.channels_last)
    packed = conv_tc.pack_weight_tf32(w, indices)
    out = conv_tc.conv_forward_tf32x3(xin, None if aux is None else dev32(aux), mode, packed,
                                      bias=None if bias is None else dev32(bias), relu=relu, stride=float(stride),
                                      with_pool=pool)
    y, p = out if pool else (out, None)
    assert y.dtype == torch.float32 and y.is_contiguous()
    return y, p


def check_out(y, p, ref, what):
    assert tuple(y.shape) == tuple(ref.shape), what
    assert_exact(y, ref, what)
    if p is not None:
        B, Co, H, W = ref.shape
        assert_exact(p, ref.view(B, Co // 8, 8, H, W).amax(dim=2), what + " pooled")


def check_tf32x3_case(mode, x, aux, off, w, bias, relu, pool, stride, layout, q, what, indices=None):
    """Run one call, check the budget of the integer / dyadic data and compare with float64."""
    bank = w if indices is None else arf_bank(w, indices)
    ref = conv_ref(x, off, bank, bias, relu)
    S = conv_ref(x.abs(), off, bank.abs(), None if bias is None else bias.abs(), False)
    check_budget(S, q, what=what)
    y, p = run_tf32x3(mode, x, aux, w, bias, relu, pool, stride, layout, indices)
    check_out(y, p, ref, what)
    return y, ref


TF32X3_A_CASES = [  # mode, C, Co, bias, relu, pool, layout
    (2, 32, 32, True, True, False, "nchw"), (2, 96, 224, False, False, True, "cl"), (2, 256, 64, True, False, True, "nchw"),
    (1, 32, 64, True, False, True, "nchw"), (1, 256, 256, False, True, False, "cl"), (1, 96, 224, True, True, False, "nchw"),
    (0, 96, 32, True, True, False, "cl"), (0, 256, 224, False, False, True, "nchw"), (0, 32, 256, True, False, False, "nchw"),
]


@pytest.mark.parametrize("mode,C,Co,bias,relu,pool,layout", TF32X3_A_CASES)
def test_tf32x3_exact_integer_data(mode, C, Co, bias, relu, pool, layout):
    """Regime A on 1x1, 1x17, 9x1 and 13x21 maps: sampling positions exactly on -1, H - 1, W - 1, in (W - 1, W) and
    off the map; partial tiles; bias, ReLU and the pooled output on and off; NCHW and channels_last input."""
    g = torch.Generator().manual_seed(100 * mode + C + Co)
    B = 2
    w = dev32(ints((Co, C, 3, 3), 3, g))
    b = dev32(ints((Co,), 16, g)) if bias else None
    for (H, W), stride in zip(MAPS, STRIDES):
        x = ints((B, C, H, W), 8, g)
        aux, off = tf32x3_aux(mode, B, H, W, stride, g, False)
        what = "conv_forward_tf32x3 mode %d C=%d Co=%d %dx%d %s" % (mode, C, Co, H, W, layout)
        check_tf32x3_case(mode, x, aux, off, w, b, relu, pool, stride, layout, 1.0 if mode == 2 else 1 / 16, what)


@pytest.mark.parametrize("mode", [0, 1, 2])
def test_tf32x3_exact_bench_levels(mode):
    """The five FPN levels of the benchmark at C = C_out = 256, batch 2.  At 128 x 128, 2 x 128 tiles of 8 x 16 pixels
    exceed the CTA count, so CTAs run several tiles and the barriers go through further phases."""
    g = torch.Generator().manual_seed(200 + mode)
    B, C, Co = 2, 256, 256
    assert B * math.ceil(128 / 8) * math.ceil(128 / 16) > sm_count()
    w = dev32(ints((Co, C, 3, 3), 3, g))
    b = dev32(ints((Co,), 16, g)) if mode == 2 else None
    for (H, W), stride in zip(BENCH_LEVELS, BENCH_STRIDES):
        x = ints((B, C, H, W), 8, g)
        aux, off = tf32x3_aux(mode, B, H, W, stride, g, False)
        what = "conv_forward_tf32x3 mode %d bench level %dx%d" % (mode, H, W)
        check_tf32x3_case(mode, x, aux, off, w, b, mode == 0, mode == 2, stride, "cl", 1.0 if mode == 2 else 1 / 16, what)


@pytest.mark.parametrize("I,O,nOri,layout", [(32, 32, 1, "nchw"), (4, 4, 8, "cl"), (12, 28, 8, "nchw"), (256, 32, 1, "cl")])
def test_tf32x3_orconv_exact(I, O, nOri, layout):
    """ORConv2d through the public fp32 entry (orn.orconv_forward -> mode 2 with the ARF map folded into the packed
    planes), with bias and the fused 8-way orientation max."""
    from s2anet_b200.orn import ORConv2d, orconv_forward
    g = torch.Generator().manual_seed(300 + I + O + nOri)
    m = ORConv2d(I, O, 3, padding=1, arf_config=(nOri, 8)).to(DEV)
    w = dev32(ints(m.weight.shape, 3, g))
    b = dev32(ints((O * 8,), 16, g))
    bank = arf_bank(w, m.indices)
    for H, W in MAPS:
        x = dev32(ints((2, I * nOri, H, W), 8, g))
        xin = x.contiguous(memory_format=torch.channels_last) if layout == "cl" else x
        what = "orconv_forward tf32x3 I=%d O=%d nOri=%d %dx%d" % (I, O, nOri, H, W)
        ref = conv_ref(x, None, bank, b, False)
        check_budget(conv_ref(x.abs(), None, bank.abs(), b.abs(), False), 1.0, what=what)
        y, p = orconv_forward(xin, w, m.indices, b, with_pool=True)
        check_out(y, p, ref, what)


def sparse_mask(Co, K9, nnz, g):
    """[Co, K9] bool with exactly nnz True per row."""
    order = torch.rand(Co, K9, generator=g).argsort(dim=1)
    return order < nnz


def one_sided_case(side, B, C, Co, H, W, g):
    """x, w for regime B: the `side` operand = +-(1 + odd 2**-11) (lo = +-2**-11), the other in {-1, 0, 1}; w has
    exactly nnz nonzeros per output channel so that sum |x||w| / 2**-11 stays within the budget."""
    nnz = min(9 * C * 2 // 3, 192)
    mask = sparse_mask(Co, 9 * C, nnz, g).double().view(Co, 3, 3, C).permute(0, 3, 1, 2)
    if side == "x":
        x = odd_fractions((B, C, H, W), g)
        w = mask * torch.where(torch.rand(Co, C, 3, 3, generator=g) < 0.5, -1.0, 1.0).double()
    else:
        x = ints((B, C, H, W), 1, g)
        w = mask * odd_fractions((Co, C, 3, 3), g)
    return x, w


@pytest.mark.parametrize("mode,side,C,Co", [(2, "x", 32, 32), (2, "w", 256, 64), (1, "x", 256, 256), (1, "w", 32, 224),
                                            (0, "x", 96, 96), (0, "w", 96, 32)])
def test_tf32x3_exact_one_sided_low_parts(mode, side, C, Co):
    """Regime B: a_lo * w_hi (side x) or a_hi * w_lo (side w) carries half of every product's low bits; the output is
    exact only if that correction MMA runs with the right operands.  Integer sampling positions (samples are copies)."""
    g = torch.Generator().manual_seed(400 + 10 * mode + C + Co + (side == "w"))
    B = 2
    for (H, W), stride in zip(((13, 21), (1, 17), (9, 1)), STRIDES):
        x, w = one_sided_case(side, B, C, Co, H, W, g)
        assert bool((tf32_split((x if side == "x" else w).float())[1] != 0).any())
        aux, off = tf32x3_aux(mode, B, H, W, stride, g, True)
        b = ints((Co,), 16, g)
        what = "conv_forward_tf32x3 mode %d lo on %s C=%d Co=%d %dx%d" % (mode, side, C, Co, H, W)
        check_tf32x3_case(mode, x, aux, off, dev32(w), dev32(b), False, False, stride, "nchw", Q11, what)


def tf32_round_rne(v):
    """Round-to-nearest-even TF32 model: what the split would be with cvt.rn instead of cvt.rna."""
    b = v.to(torch.float32).contiguous().view(torch.int32)
    mag = b & 0x7FFFFFFF
    r = ((mag + 0x0FFF + ((mag >> 13) & 1)) & ~0x1FFF) | (b & ~0x7FFFFFFF)
    return r.view(torch.float32)


def tf32_trunc(v):
    """Truncating TF32 model: the low 13 bits masked."""
    return (v.to(torch.float32).contiguous().view(torch.int32) & ~0x1FFF).view(torch.float32)


def split_sensitive(shape, g):
    """Half TF32 ties +-(1 + odd 2**-11) (rna and rne split them differently), half +-(1 + odd 2**-12), 13 significant
    bits and no tie (rna and truncation split them differently): every lo part is nonzero."""
    m = 2 * torch.randint(0, 2048, tuple(shape), generator=g) + 1
    s = torch.where(torch.rand(tuple(shape), generator=g) < 0.5, -1.0, 1.0).double()
    near = s * (1.0 + m.double() * 2.0 ** -12)
    return torch.where(torch.rand(tuple(shape), generator=g) < 0.5, odd_fractions(shape, g), near)


@pytest.mark.parametrize("mode,C,Co", [(2, 32, 32), (2, 256, 256), (1, 96, 224), (0, 32, 64)])
def test_tf32x3_one_product_per_output_pins_the_split(mode, C, Co):
    """Regime C: one-hot weights (one nonzero (tap, channel) per output channel), x and w from split_sensitive.  An
    output is one product a * w; the kernel computes a_hi w_hi + (a_lo w_hi + a_hi w_lo) = a w - a_lo w_lo, each part
    exact (a multiple of 2**-22 below 4), so it must equal that with the rna split exactly -- and differ from a * w.
    On the model, a round-to-nearest-even split and a truncating split each change a large share of these outputs."""
    g = torch.Generator().manual_seed(500 + mode + C + Co)
    B, H, W, stride = 2, 13, 21, 16
    x = split_sensitive((B, C, H, W), g)
    w = torch.zeros(Co, C, 9, dtype=torch.float64)
    w[torch.arange(Co), torch.randint(0, C, (Co,), generator=g), torch.randint(0, 9, (Co,), generator=g)] = 1.0
    w = (w * split_sensitive((Co, C, 9), g)).view(Co, C, 3, 3)
    aux, off = tf32x3_aux(mode, B, H, W, stride, g, True)
    aw = conv_ref(x, off, w, None, False)
    model = lambda rnd: aw - conv_ref((x.float() - rnd(x.float())).double(), off, (w.float() - rnd(w.float())).double(),
                                      None, False)
    want = model(tf32_round)
    what = "conv_forward_tf32x3 mode %d one product per output C=%d Co=%d" % (mode, C, Co)
    y, _ = run_tf32x3(mode, x, aux, dev32(w), None, False, False, stride, "nchw")
    assert_exact(y, want, what)
    nz = aw != 0
    assert float(nz.double().mean()) > 0.3, "%s: too few outputs sample the map" % what
    assert bool((want != aw)[nz].all()), "%s: the dropped a_lo * w_lo term is not visible everywhere" % what
    for name, rnd in (("rne", tf32_round_rne), ("truncating", tf32_trunc)):
        share = float((model(rnd) != want)[nz].double().mean())
        assert share > 0.2, "%s: a %s split changes only %.3f of the outputs" % (what, name, share)


def test_tf32x3_rotated_anchors_match_the_offset_mode():
    """Rotated anchors at a benchmark level (64 x 64, stride 16): mode 0 against mode 1 fed the offsets recomputed with
    torch fp32 ops in the kernel's operation order.  Both then share every later operation, so the outputs agree bit
    for bit wherever torch's cos / sin equal the kernel's cosf / sinf.  They do not always (an ulp of a sampling
    position reaches all 256 channels of a pixel in fp32), so disagreements are counted: at most ROTATED_DIFFER_LIMIT
    of the outputs, each within the fp32 tolerance.  Rotated anchors are only cross-checked, never compared with
    float64 exactly."""
    from s2anet_b200 import conv_tc, synth
    g = torch.Generator().manual_seed(41)
    B, C, H, W, Co, stride = 2, 256, 64, 64, 256, 16
    x = torch.randn(B, C, H, W, generator=g).to(DEV)
    wt = (torch.randn(Co, C, 3, 3, generator=g) * 0.05).to(DEV)
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
        off[:, 2 * t] = (yr + ay) - (yy + fi)
        off[:, 2 * t + 1] = (xr + ax) - (xx + fj)
    packed = conv_tc.pack_weight_tf32(wt)
    ya = conv_tc.conv_forward_tf32x3(x, anc, 0, packed, relu=True, stride=float(stride))
    yd = conv_tc.conv_forward_tf32x3(x, off, 1, packed, relu=True)
    n = int((ya != yd).sum())
    print("\nrotated anchors, tf32x3 mode 0 vs mode 1: %d of %d outputs differ" % (n, ya.numel()))
    assert n <= ROTATED_DIFFER_LIMIT * ya.numel(), "%d of %d outputs differ" % (n, ya.numel())
    assert float((ya - yd).abs().max()) <= 1e-5 + 2e-5 * float(yd.abs().max())


# ------------------------------------------------------------------------------------------------------------------
# 3. the SIMT kernel (conv_f32.cu) through the public entries
# ------------------------------------------------------------------------------------------------------------------
def wide_tile(groups, Co, Ho, Wo, B):
    """conv_f32.cu launch_conv_mode: the 128 x 128 tile when the conv is ungrouped, C_out >= 128 and the wide tiles
    alone fill the GPU."""
    return groups == 1 and Co >= 128 and math.ceil(Ho * Wo / 128) * math.ceil(Co / 128) * B >= sm_count()


def deform_forward(x, w, off, k, stride, pad, dil, groups, dgroups):
    from s2anet_b200 import dcn
    B, Co = x.size(0), w.size(0)
    Ho, Wo = out_size(x.size(2), k, stride, pad, dil), out_size(x.size(3), k, stride, pad, dil)
    out = torch.full((B, Co, Ho, Wo), float("nan"), device=DEV)
    e = torch.empty(0, device=DEV)
    assert dcn.deform_conv_forward_cuda(dev32(x), dev32(w), dev32(off), out, e, e, k, k, stride, stride, pad, pad, dil, dil,
                                        groups, dgroups, B) == 1
    return out


def check_deform_simt(B, C, Co, H, W, geom, g, what):
    k, stride, pad, dil, groups, dgroups = geom
    x = ints((B, C, H, W), 8, g)
    w = ints((Co, C // groups, k, k), 3, g)
    off = geom_offsets(B, H, W, k, stride, pad, dil, dgroups, g)
    h, ww = geom_positions(off, k, stride, pad, dil)
    assert (h == -1).any() and (h == H - 1).any() and ((ww > W - 1) & (ww < W)).any()
    x64, w64, off64 = x.to(DEV), w.to(DEV), off.to(DEV)
    ref = tv().ops.deform_conv2d(x64, off64, w64, stride=stride, padding=pad, dilation=dil)
    S = tv().ops.deform_conv2d(x64.abs(), off64, w64.abs(), stride=stride, padding=pad, dilation=dil)
    check_budget(S, 1 / 16, what=what)
    y = deform_forward(x, w, off, k, stride, pad, dil, groups, dgroups)
    assert_exact(y, ref, what)
    return wide_tile(groups, Co, ref.size(2), ref.size(3), B)


# (k, stride, pad, dilation, groups, deformable groups), C
SIMT_GEOMS = [((3, 1, 1, 1, 1, 1), 12), ((3, 2, 2, 2, 1, 2), 32), ((1, 2, 0, 1, 1, 1), 12), ((2, 1, 0, 1, 1, 1), 12),
              ((3, 1, 0, 1, 1, 4), 32)]


@pytest.mark.parametrize("geom,C,Co", [(gm, c, co) for gm, c in SIMT_GEOMS for co in (40, 72, 200)] +
                         [((3, 1, 1, 1, 2, 1), 24, 128)])
def test_simt_deform_conv_exact(geom, C, Co):
    """DEFORM: kernel sizes 1, 2, 3, stride, padding, dilation, groups (C_out / groups = 64), deformable groups, a
    partial 8-channel chunk (C = 12, C / groups = 12) and partial channel tiles (C_out = 40, 72, 200)."""
    g = torch.Generator().manual_seed(600 + sum(geom) + C + Co)
    check_deform_simt(2, C, Co, 10, 13, geom, g, "deform_conv_forward_cuda SIMT %s C=%d Co=%d" % (geom, C, Co))


def test_simt_deform_conv_exact_both_tiles():
    """C_out = 200 on the narrow (64 x 64) and the wide (128 x 128) tile; the wide one has a partial channel tile."""
    g = torch.Generator().manual_seed(650)
    B, Co = 2, 200
    Wbig = math.ceil(sm_count() / 2) + 2                   # 64 x Wbig: ceil(64 Wbig / 128) * 2 * 2 >= SM count
    seen = set()
    for H, W in ((10, 13), (64, Wbig)):
        seen.add(check_deform_simt(B, 12, Co, H, W, (3, 1, 1, 1, 1, 1), g, "deform_conv_forward_cuda SIMT Co=200 %dx%d" % (H, W)))
    assert seen == {False, True}, "both tile shapes must run"


@pytest.mark.parametrize("C,Co,force", [(24, 40, False), (24, 200, False), (64, 72, True)])
def test_simt_alignconv_exact(C, Co, force, request):
    """ALIGN: C = 24 (tf32x3 refuses it) and C = 64 with the SIMT route forced; dyadic anchors, ReLU."""
    from s2anet_b200.alignconv import alignconv_forward
    if force:
        request.getfixturevalue("simt")
    g = torch.Generator().manual_seed(700 + C + Co)
    B = 2
    w = ints((Co, C, 3, 3), 3, g)
    for (H, W), stride in zip(MAPS + ((64, math.ceil(sm_count() / 2) + 2),), STRIDES + (8,)):
        x = ints((B, C, H, W), 8, g)
        anc = dyadic_anchors(B, H, W, stride, g)
        off = align_offsets(anc, H, W, stride)
        what = "alignconv_forward SIMT C=%d Co=%d %dx%d" % (C, Co, H, W)
        ref = conv_ref(x, off, w, None, True)
        check_budget(conv_ref(x.abs(), off, w.abs(), None, False), 1 / 16, what=what)
        y = alignconv_forward(dev32(x), dev32(anc), dev32(w), stride)
        assert_exact(y, ref, what)


@pytest.mark.parametrize("I,O,nOri,big", [(12, 5, 1, False), (12, 3, 8, False), (12, 20, 1, True), (12, 20, 8, False)])
def test_simt_orconv_exact(I, O, nOri, big, simt):
    """PLAIN (ORConv2d): the ARF map in the weight-tile load, bias, the fused orientation max; O * 8 = 160 on the wide
    tile has a partial channel tile."""
    from s2anet_b200.orn import ORConv2d, orconv_forward
    g = torch.Generator().manual_seed(800 + I + O + nOri)
    m = ORConv2d(I, O, 3, padding=1, arf_config=(nOri, 8)).to(DEV)
    w = dev32(ints(m.weight.shape, 3, g))
    b = dev32(ints((O * 8,), 16, g))
    bank = arf_bank(w, m.indices)
    maps = ((64, math.ceil(sm_count() / 2) + 2),) if big else MAPS
    for H, W in maps:
        x = dev32(ints((2, I * nOri, H, W), 8, g))
        if big:
            assert wide_tile(1, O * 8, H, W, 2)
        what = "orconv_forward SIMT I=%d O=%d nOri=%d %dx%d" % (I, O, nOri, H, W)
        ref = conv_ref(x, None, bank, b, False)
        check_budget(conv_ref(x.abs(), None, bank.abs(), b.abs(), False), 1.0, what=what)
        y, p = orconv_forward(x, w, m.indices, b, with_pool=True)
        check_out(y, p, ref, what)


def test_simt_and_tf32x3_agree_where_both_apply():
    """Shapes both routes take: both exact, so equal to each other bit for bit."""
    from s2anet_b200 import alignconv
    from s2anet_b200.orn import ORConv2d, orconv_forward
    g = torch.Generator().manual_seed(900)
    B, C, Co, H, W = 2, 64, 96, 11, 19
    x, w = ints((B, C, H, W), 8, g), ints((Co, C, 3, 3), 3, g)
    off = quarter_offsets(B, H, W, g)
    m = ORConv2d(8, 4, 3, padding=1, arf_config=(8, 8)).to(DEV)
    wo, bo = dev32(ints(m.weight.shape, 3, g)), dev32(ints((32,), 16, g))
    outs, old = {}, alignconv._FORCE_SIMT_F32
    for path in ("tf32x3", "simt"):
        alignconv.set_fp32_path(path)
        try:
            outs[path] = (deform_forward(x, w, off, 3, 1, 1, 1, 1, 1),) + orconv_forward(dev32(x), wo, m.indices, bo, with_pool=True)
        finally:
            alignconv._FORCE_SIMT_F32 = old
    assert_exact(outs["simt"][0], conv_ref(x, off, w, None, False), "deform_conv_forward_cuda SIMT")
    assert_exact(outs["simt"][1], conv_ref(x, None, arf_bank(wo, m.indices), bo, False), "orconv_forward SIMT")
    for a, b in zip(outs["simt"], outs["tf32x3"]):
        assert torch.equal(a, b)


def test_simt_unsupported_geometries_raise():
    """5x5 kernels, C_out / groups = 24 and C / deformable_groups = 4: an error, not an output."""
    g = torch.Generator().manual_seed(950)
    x = ints((1, 16, 9, 9), 2, g)
    for k, groups, dgroups, Co in ((5, 1, 1, 16), (3, 2, 1, 48), (3, 1, 4, 16)):
        w = ints((Co, 16 // groups, k, k), 1, g)
        off = torch.zeros(1, dgroups * 2 * k * k, 9, 9)
        with pytest.raises(RuntimeError, match="not supported|needs"):
            deform_forward(x, w, off, k, 1, k // 2, 1, groups, dgroups)


# ------------------------------------------------------------------------------------------------------------------
# 4. the fp32 deformable backward: s2a_deform_im2col_f32 / s2a_deform_col2im_f32 + the GEMMs of dcn.py
# ------------------------------------------------------------------------------------------------------------------
BWD_GEOMS = SIMT_GEOMS + [((3, 1, 1, 1, 2, 1), 24), ((5, 1, 2, 1, 1, 1), 12), ((7, 2, 3, 1, 1, 1), 8)]


@pytest.mark.parametrize("geom,C", BWD_GEOMS)
def test_deform_backward_fp32_exact(geom, C, fp32_matmul):
    """deform_conv_backward_input_cuda and deform_conv_backward_parameters_cuda accumulate into the caller's tensors:
    pre-filled with integer patterns, they must hold pattern + gradient (scale 0.5 for the weight) exactly.  Batch 4
    in im2col_step chunks of 2; Ho * Wo is not a multiple of 128."""
    from s2anet_b200 import dcn
    k, stride, pad, dil, groups, dgroups = geom
    g = torch.Generator().manual_seed(1000 + sum(geom) + C)
    B, H, W, step = 4, 11, 13, 2
    Co = 64 * groups if groups > 1 else 40
    Ho, Wo = out_size(H, k, stride, pad, dil), out_size(W, k, stride, pad, dil)
    assert (Ho * Wo) % 128 != 0
    x, w, go = ints((B, C, H, W), 2, g), ints((Co, C // groups, k, k), 1, g), ints((B, Co, Ho, Wo), 2, g)
    off = geom_offsets(B, H, W, k, stride, pad, dil, dgroups, g)
    gi_ref, goff_ref, gw_ref = deform_grads_ref(x.to(DEV), off, w, go, stride, pad, dil)
    gi_S, _, gw_S = deform_grads_ref(x.to(DEV).abs(), off, w.abs(), go.abs(), stride, pad, dil)
    pi, po, pw = ints(x.shape, 64, g).to(DEV), ints(off.shape, 64, g).to(DEV), ints(w.shape, 64, g).to(DEV)
    what = "deform backward fp32 %s C=%d Co=%d" % (geom, C, Co)
    check_budget(gi_S + pi.abs(), 1 / 16, what=what + " grad_input")
    # gy = sum_c gcol_c (hx (v3 - v1) + lx (v4 - v2)): |gcol_c| <= (Co / groups) max|w| max|go|, quantum 1/4
    check_budget(torch.tensor([(C // dgroups) * (Co // groups) * 1 * 2 * 2 * 2 + 64.0]), 1 / 4, what=what + " grad_offset")
    check_budget(pw.abs() + 0.5 * gw_S, 1 / 32, what=what + " grad_weight")
    gI, gO, gW = dev32(pi), dev32(po), dev32(pw)
    e = torch.empty(0, device=DEV)
    xs, offs, gos, ws = dev32(x), dev32(off), dev32(go), dev32(w)
    assert dcn.deform_conv_backward_input_cuda(xs, offs, gos, gI, gO, ws, e, k, k, stride, stride, pad, pad, dil, dil,
                                               groups, dgroups, step) == 1
    assert dcn.deform_conv_backward_parameters_cuda(xs, offs, gos, gW, e, e, k, k, stride, stride, pad, pad, dil, dil,
                                                    groups, dgroups, 0.5, step) == 1
    assert_exact(gI, pi + gi_ref, what + " grad_input")
    assert_exact(gO, po + goff_ref, what + " grad_offset")
    assert_exact(gW, pw + 0.5 * gw_ref, what + " grad_weight")


def test_deform_conv_module_autograd_fp32_exact(fp32_matmul):
    """DeformConv end to end in fp32 (forward on tf32x3 or SIMT, backward through DeformConvFunction): the output, x.grad,
    the offset gradient and weight.grad equal the float64 reference."""
    from s2anet_b200.dcn import DeformConv
    g = torch.Generator().manual_seed(1100)
    for C, Co, k, stride, pad, dil, dgroups in ((32, 64, 3, 1, 1, 1, 1), (16, 40, 3, 2, 2, 2, 2)):
        m = DeformConv(C, Co, k, stride=stride, padding=pad, dilation=dil, deformable_groups=dgroups).to(DEV)
        B, H, W = 2, 10, 13
        w = ints(m.weight.shape, 1, g)
        with torch.no_grad():
            m.weight.copy_(w)
        x = ints((B, C, H, W), 2, g)
        off = geom_offsets(B, H, W, k, stride, pad, dil, dgroups, g)
        Ho, Wo = out_size(H, k, stride, pad, dil), out_size(W, k, stride, pad, dil)
        go = ints((B, Co, Ho, Wo), 2, g)
        xg, og = dev32(x).requires_grad_(True), dev32(off).requires_grad_(True)
        y = m(xg, og)
        y.backward(dev32(go))
        what = "DeformConv fp32 C=%d Co=%d" % (C, Co)
        ref = tv().ops.deform_conv2d(x.to(DEV), off.to(DEV), w.to(DEV), stride=stride, padding=pad, dilation=dil)
        assert_exact(y.detach(), ref, what + " output")
        gi_ref, goff_ref, gw_ref = deform_grads_ref(x.to(DEV), off, w, go, stride, pad, dil)
        assert_exact(xg.grad, gi_ref, what + " x.grad")
        assert_exact(og.grad, goff_ref, what + " offset.grad")
        assert_exact(m.weight.grad, gw_ref, what + " weight.grad")


def test_alignconv_module_autograd_fp32_exact(fp32_matmul):
    """AlignConv in fp32 with gradients: the explicit-offset route (get_offset + DeformConv + ReLU); the anchors carry
    no gradient, so x.grad and weight.grad are compared."""
    from s2anet_b200.alignconv import AlignConv
    g = torch.Generator().manual_seed(1200)
    B, C, Co, H, W, stride = 2, 32, 64, 13, 21, 16
    m = AlignConv(C, Co).to(DEV)
    w = ints(m.deform_conv.weight.shape, 1, g)
    with torch.no_grad():
        m.deform_conv.weight.copy_(w)
    x = ints((B, C, H, W), 2, g)
    anc = dyadic_anchors(B, H, W, stride, g)
    go = ints((B, Co, H, W), 2, g)
    xg = dev32(x).requires_grad_(True)
    y = m(xg, dev32(anc), stride)
    y.backward(dev32(go))
    x64 = x.to(DEV).requires_grad_(True)
    w64 = w.to(DEV).requires_grad_(True)
    ref = tv().ops.deform_conv2d(x64, align_offsets(anc, H, W, stride).to(DEV), w64, padding=1).relu()
    ref.backward(go.to(DEV))
    assert_exact(y.detach(), ref.detach(), "AlignConv fp32 output")
    assert_exact(xg.grad, x64.grad, "AlignConv fp32 x.grad")
    assert_exact(m.deform_conv.weight.grad, w64.grad, "AlignConv fp32 weight.grad")


# ------------------------------------------------------------------------------------------------------------------
# 5. the ARF backward (orn.cu): sum in fp32, round once
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16, torch.float16])
@pytest.mark.parametrize("O,I,nOri", [(32, 256, 1), (3, 5, 8)])
def test_arf_backward_exact(oracle, dtype, O, I, nOri):
    """orn.arf_backward and the active_rotating_filter autograd Function: fp32 equals the oracle exactly on dyadic data;
    bf16 / fp16 equal the float64 sum of the eight rotations rounded once (ties included)."""
    from s2anet_b200.orn import active_rotating_filter, arf_backward
    g = torch.Generator().manual_seed(1300 + O + I + nOri)
    idx = torch.from_numpy(oracle.arf_indices(nOri, 8, 3)).to(DEV)
    r = {torch.float32: 2 ** 12, torch.bfloat16: 2 ** 8, torch.float16: 2 ** 11}[dtype]
    scale = torch.pow(2.0, torch.randint(-3, 1, (O * 8, I * nOri, 3, 3), generator=g).double())
    go = ints((O * 8, I * nOri, 3, 3), r, g) * scale                  # exact in dtype; sums of 8 exact in fp32
    go16 = go.to(dtype).to(DEV)
    assert torch.equal(go16.double().cpu(), go)
    ref = torch.from_numpy(oracle.arf_backward(idx.cpu().numpy(), go.float().numpy(), O, I)).double().to(DEV)
    what = "arf_backward %s O=%d I=%d nOri=%d" % (dtype, O, I, nOri)
    gw = arf_backward(idx, go16)
    assert gw.dtype == dtype and tuple(gw.shape) == (O, I, nOri, 3, 3)
    assert_exact(gw, ref, what)
    if dtype != torch.float32:
        assert bool((round_rne(ref, dtype).double() != ref).any()), "%s: no output needed rounding" % what
    wd = torch.zeros((O, I, nOri, 3, 3), dtype=dtype, device=DEV, requires_grad=True)
    active_rotating_filter(wd, idx).backward(go16)
    assert_exact(wd.grad, ref, what + " (autograd)")
