"""CPU checks of the references in tc_reference.py, which the exact and rounding-model tests of the 16-bit tensor-core
convolutions (test_gpu_tc_exact.py) and the fp32 convolutions (test_gpu_fp32_exact.py) rest on."""
import numpy as np
import pytest
import torch

from tc_reference import (EDGE_POSITIONS, FORMATS, check_budget, emulate_samples, geom_offsets, geom_positions, odd_fractions,
                          out_size, quarter_offsets, round_rne, round_rne64, sampling_positions, tf32_round, tf32_split, ulp)

BF16, F16 = torch.bfloat16, torch.float16


def _bits(t):
    return t.view(torch.int16)


def test_round_rne_fp16_matches_numpy():
    """numpy's float64 -> float16 conversion is correctly rounded: compare on normals, subnormals, midpoints and
    values past the largest finite fp16."""
    rng = np.random.default_rng(0)
    v = [rng.standard_normal(20000) * 10.0 ** rng.uniform(-9, 5, 20000),
         rng.uniform(-2 ** -14, 2 ** -14, 5000),                                   # subnormal range
         (rng.integers(-2 ** 12, 2 ** 12, 5000) + 0.5) * 2.0 ** rng.integers(-26, 5, 5000),   # midpoints of 11-bit grids
         np.array([65504.0, 65519.99, 65520.0, 70000.0, -65520.0, 1e300, -1e300, 2 ** -25, 2 ** -25 + 2 ** -60,
                   3 * 2 ** -26, 2 ** -24, 0.0, -0.0])]
    x = np.concatenate(v)
    with np.errstate(over="ignore"):
        want = x.astype(np.float16)
    got = round_rne(torch.from_numpy(x), F16).numpy()
    assert np.array_equal(got.view(np.uint16), want.view(np.uint16))


def test_round_rne_bf16_matches_torch_on_fp32_inputs():
    """torch's float32 -> bfloat16 conversion rounds once (to nearest even): compare on fp32-representable inputs."""
    g = torch.Generator().manual_seed(1)
    x = torch.randn(50000, generator=g) * torch.pow(10.0, torch.empty(50000).uniform_(-38, 38, generator=g))
    mid = (torch.randint(-2 ** 9, 2 ** 9, (5000,), generator=g) + 0.5) * torch.pow(2.0, torch.randint(-130, 120, (5000,), generator=g).float())
    sub = torch.empty(5000).uniform_(-2 ** -126, 2 ** -126, generator=g)
    x = torch.cat([x, mid.float(), sub, torch.tensor([3.3895314e38, 3.3961e38, 3.3963e38, -3.4e38, 0.0, -0.0])])
    assert torch.equal(_bits(round_rne(x.double(), BF16)), _bits(x.to(BF16)))


@pytest.mark.parametrize("dtype,cases", [
    (BF16, [(1 + 2 ** -8 + 2 ** -30, 1 + 2 ** -7),      # just above a midpoint: up (torch's float64 path gives 1.0)
            (1 + 2 ** -8 - 2 ** -30, 1.0),              # just below: down
            (1 + 2 ** -8, 1.0),                          # the midpoint itself: to even
            (1 + 3 * 2 ** -8, 1 + 2 ** -6),              # midpoint, odd neighbour below: up
            (-(1 + 2 ** -8 + 2 ** -40), -(1 + 2 ** -7))]),
    (F16, [(1 + 2 ** -11 + 2 ** -40, 1 + 2 ** -10),
           (1 + 2 ** -11 - 2 ** -40, 1.0),
           (1 + 2 ** -11, 1.0),
           (2 ** -25 + 2 ** -50, 2 ** -24),              # above half the smallest subnormal
           (2 ** -25, 0.0),                              # exactly half: to even (zero)
           (65520.0 - 2 ** -20, 65504.0),
           (65520.0, float("inf"))]),
])
def test_round_rne_midpoints(dtype, cases):
    x = torch.tensor([c[0] for c in cases], dtype=torch.float64)
    want = torch.tensor([c[1] for c in cases], dtype=torch.float64)
    assert torch.equal(round_rne64(x, dtype), want)
    if dtype == BF16:                                    # torch's own conversion rounds twice here
        assert not torch.equal(x[:1].to(BF16).double(), want[:1])


def test_ulp():
    for dtype, (p, emin, _) in FORMATS.items():
        x = torch.tensor([1.0, 1.5, 2.0 - 2 ** -20, 2.0, -3.0, 0.0, 2.0 ** (emin - 3), 2.0 ** emin], dtype=torch.float64)
        want = [2 ** (1 - p), 2 ** (1 - p), 2 ** (1 - p), 2 ** (2 - p), 2 ** (2 - p), 2 ** (emin + 1 - p),
                2 ** (emin + 1 - p), 2 ** (emin + 1 - p)]
        assert ulp(x, dtype).tolist() == want
        # every value of the format is a multiple of its ulp and the next value is one ulp away
        v = torch.randn(1000, dtype=torch.float64).to(dtype).double()
        u = ulp(v, dtype)
        assert torch.equal(torch.remainder(v, u), torch.zeros_like(v))
        nxt = (v.to(dtype).view(torch.int16) + 1).view(dtype).double()           # sign-magnitude: one step away from 0
        assert torch.equal((nxt - v).abs(), u)


def test_check_budget():
    check_budget(torch.tensor([2.0 ** 20]), 1.0)
    with pytest.raises(AssertionError, match="budget"):
        check_budget(torch.tensor([2.0 ** 20 + 1]), 1.0)
    with pytest.raises(AssertionError, match="budget"):
        check_budget(torch.tensor([2.0 ** 17]), 1 / 16)
    with pytest.raises(AssertionError, match="overflows"):
        check_budget(torch.tensor([100.0]), 1.0, torch.float16, torch.tensor([-70000.0]))


@pytest.mark.parametrize("dtype", [BF16, F16])
@pytest.mark.parametrize("round_positions", [False, True])
def test_emulate_samples_matches_torchvision_on_quarter_offsets(dtype, round_positions):
    """With offsets on a 1/4 grid and small integer activations every position, weight and partial blend is exact, so
    the emulated samples must equal torchvision's float64 deform_conv2d with one-hot weights, tap by tap -- edges
    (h = -1, h = H - 1, positions in (W - 1, W)) included."""
    tv = pytest.importorskip("torchvision")
    g = torch.Generator().manual_seed(3 + round_positions)
    B, C, H, W = 2, 8, 7, 11
    x = torch.randint(-8, 9, (B, C, H, W), generator=g).to(dtype)
    off = quarter_offsets(B, H, W, g)
    for off_dtype in (torch.float32, dtype):
        s, inexact = emulate_samples(x, off.to(off_dtype), dtype, round_positions, return_inexact=True)
        assert inexact == 0 and s.shape == (B, H, W, 9, C)
        for t in range(9):
            wt = torch.zeros(C, C, 3, 3, dtype=torch.float64)
            wt[torch.arange(C), torch.arange(C), t // 3, t % 3] = 1.0
            ref = tv.ops.deform_conv2d(x.double(), off, wt, padding=1)
            assert torch.equal(s[:, :, :, t].permute(0, 3, 1, 2), ref), "tap %d" % t
    # the edge cases are there: exactly -1, exactly H - 1, and strictly between W - 1 and W
    pos_h = off[:, 0::2] + (torch.arange(H).view(1, 1, H, 1) - 1 + torch.arange(9).view(1, 9, 1, 1) // 3)
    pos_w = off[:, 1::2] + (torch.arange(W).view(1, 1, 1, W) - 1 + torch.arange(9).view(1, 9, 1, 1) % 3)
    assert (pos_h == -1).any() and (pos_h == H - 1).any() and ((pos_w > W - 1) & (pos_w < W)).any()


def test_emulate_samples_models_rounding():
    """Off the exact grid the emulator rounds where the kernel does.  A position 5 + 2**-9 stays put in fp32 (the
    sample is 2**-9 of the right neighbour) and becomes 5.0 in bf16 under round_positions (the left pixel alone)."""
    x = torch.zeros(1, 1, 1, 8)
    x[0, 0, 0, 6] = 64.0
    x = x.to(BF16)
    off = torch.zeros(1, 18, 1, 8)
    off[0, 9, 0, 5] = 2 ** -9                    # tap 4 (the centre), dx of pixel (0, 5)
    assert float(emulate_samples(x, off, BF16, False)[0, 0, 5, 4, 0]) == 64.0 * 2 ** -9
    assert float(emulate_samples(x, off, BF16, True)[0, 0, 5, 4, 0]) == 0.0
    # normal data: blend steps round, and the emulator counts them
    g = torch.Generator().manual_seed(5)
    xr = torch.randn(1, 8, 6, 9, generator=g).to(BF16)
    _, inexact = emulate_samples(xr, torch.randn(1, 18, 6, 9, generator=g) * 1.5, BF16, False, return_inexact=True)
    assert inexact > 0


def _f32bits(t):
    return t.to(torch.float32).contiguous().view(torch.int32)


def test_tf32_split_ties_round_away_from_zero():
    """cvt.rna: a tie goes away from zero.  Round-to-nearest-even would give 1, -1 and 1 + 2**-9 here."""
    v = torch.tensor([1 + 2 ** -11, -(1 + 2 ** -11), 1 + 3 * 2 ** -11, 2 - 2 ** -11, 1 + 2 ** -11 - 2 ** -20,
                      1 + 2 ** -11 + 2 ** -20], dtype=torch.float64)
    want = [1 + 2 ** -10, -(1 + 2 ** -10), 1 + 2 ** -9, 2.0, 1.0, 1 + 2 ** -10]
    hi, lo = tf32_split(v.float())
    assert hi.double().tolist() == want
    assert torch.equal(hi.double() + lo.double(), v)
    assert lo.double().tolist()[:4] == [-2 ** -11, 2 ** -11, -2 ** -11, -2 ** -11]


def test_tf32_split_is_exact_below_23_bits():
    """hi + lo == v for every v with at most 22 significant bits whose lo part is not subnormal (a subnormal lo is
    rounded on its own, coarser bits); hi and lo are TF32 values (low 13 bits zero)."""
    g = torch.Generator().manual_seed(7)
    m = torch.randint(2 ** 21, 2 ** 22, (20000,), generator=g).double()
    e = torch.randint(-100, 100, (20000,), generator=g).double()
    s = torch.where(torch.rand(20000, generator=g) < 0.5, -1.0, 1.0).double()
    v = (s * m * torch.pow(2.0, e - 21)).float()
    hi, lo = tf32_split(v)
    assert torch.equal(hi.double() + lo.double(), v.double())
    assert bool(((_f32bits(hi) & 0x1FFF) == 0).all()) and bool(((_f32bits(lo) & 0x1FFF) == 0).all())
    assert bool((lo.double().abs() <= torch.pow(2.0, torch.floor(torch.log2(hi.double().abs())) - 11)).all())
    # 24-bit values: the residual v - hi - lo is what the kernel drops, at most 2**-22 |v|
    w = torch.randn(20000, generator=g)
    hw, lw = tf32_split(w)
    res = (w.double() - hw.double() - lw.double()).abs()
    assert bool((res <= 2.0 ** -22 * w.double().abs()).all()) and bool((res > 0).any())


def test_tf32_split_zeros_and_subnormals():
    z = torch.tensor([0.0, -0.0])
    hi, lo = tf32_split(z)
    assert _f32bits(hi).tolist() == _f32bits(z).tolist()                 # the sign of zero survives in hi
    assert _f32bits(lo).tolist() == [0, 0]                               # -0 - -0 = +0
    # subnormals round on the same bits: 0x1FFF -> 0x2000 (up), 0x0FFF -> 0 (down), 0x1000 -> 0x2000 (tie, away)
    bits = torch.tensor([0x1FFF, 0x0FFF, 0x1000, 0x3000, 0x7FFFFF, 0x00400000 | 0x1000], dtype=torch.int32)
    sub = bits.view(torch.float32)
    hi, lo = tf32_split(sub)
    assert _f32bits(hi).tolist() == [0x2000, 0, 0x2000, 0x4000, 0x800000, 0x00402000]
    # the residuals are subnormal too and round likewise (-1 bit becomes -0): hi + lo need not equal v down here
    neg = lambda b: b - 2 ** 32 if b >= 2 ** 31 else b
    assert _f32bits(lo).tolist() == [neg(0x80000000), 0, neg(0x80002000), neg(0x80002000), neg(0x80000000), neg(0x80002000)]
    assert torch.equal(_f32bits(tf32_round(-sub)), _f32bits(-hi))
    # a carry out of the mantissa moves the exponent: the largest value below 2 rounds to 2
    assert float(tf32_round(torch.tensor([2 - 2 ** -23]))) == 2.0


def test_odd_fractions_are_tf32_ties():
    g = torch.Generator().manual_seed(8)
    v = odd_fractions((5000,), g)
    assert bool(((v.abs() > 1) & (v.abs() < 2)).all())
    hi, lo = tf32_split(v.float())
    assert torch.equal(v.float().double(), v)
    assert torch.equal(lo.double().abs(), torch.full_like(v, 2.0 ** -11))
    assert torch.equal(torch.sign(lo.double()), -torch.sign(v))          # hi is the neighbour away from zero


@pytest.mark.parametrize("k,stride,pad,dil,dgroups", [(3, 1, 1, 1, 1), (3, 2, 2, 2, 2), (1, 2, 0, 1, 1), (2, 1, 0, 1, 1),
                                                      (3, 1, 0, 1, 4), (5, 1, 2, 1, 1), (7, 2, 3, 1, 1)])
def test_geom_offsets_hit_the_edges(k, stride, pad, dil, dgroups):
    """Every draw puts positions exactly on -1, just inside -1, exactly on H - 1 and W - 1, inside (W - 1, W), and off
    the map, in every deformable group; everything lies on the 1/4 grid."""
    g = torch.Generator().manual_seed(k + stride + dgroups)
    B, H, W = 2, 9, 11
    off = geom_offsets(B, H, W, k, stride, pad, dil, dgroups, g)
    Ho, Wo = out_size(H, k, stride, pad, dil), out_size(W, k, stride, pad, dil)
    assert tuple(off.shape) == (B, dgroups * 2 * k * k, Ho, Wo)
    assert torch.equal(off * 4, (off * 4).round())
    h, w = geom_positions(off, k, stride, pad, dil)
    for d in range(dgroups):
        hd, wd = h[:, d], w[:, d]
        assert (hd == -1).any() and (hd == -0.75).any() and (hd == H - 1).any() and (wd == W - 1).any()
        assert ((wd > W - 1) & (wd < W)).any() and ((hd <= -1) | (hd >= H) | (wd <= -1) | (wd >= W)).any()
        for s, (ph, pw) in enumerate(EDGE_POSITIONS(H, W)):
            t, (ho, wo) = s % (k * k), divmod(s // (k * k), Wo)
            assert (float(hd[0, t, ho, wo]), float(wd[0, t, ho, wo])) == (ph, pw)
    if (k, stride, pad, dil) == (3, 1, 1, 1) and dgroups == 1:            # the 3x3 / pad 1 positions agree
        hs, ws = sampling_positions(off)
        assert torch.equal(hs, h[:, 0]) and torch.equal(ws, w[:, 0])
