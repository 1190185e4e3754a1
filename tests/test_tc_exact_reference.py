"""CPU checks of the references in tc_reference.py, which the exact and rounding-model tests of the 16-bit tensor-core
convolutions (test_gpu_tc_exact.py) rest on."""
import numpy as np
import pytest
import torch

from tc_reference import FORMATS, check_budget, emulate_samples, quarter_offsets, round_rne, round_rne64, ulp

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
