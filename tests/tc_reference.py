"""High-precision references for the 16-bit tensor-core convolutions (csrc/conv_tc.cu).

* round_rne / ulp: correct round-to-nearest-even from float64 to bf16 / fp16.  torch's own float64 -> bf16 / fp16
  conversion goes through fp32 and so rounds twice (1 + 2**-8 + 2**-30 becomes 1.0 in bf16, not 1 + 2**-7).
* check_budget: the condition under which a kernel that accumulates in fp32 -- in any order, including the tensor
  core's aligned partial sums -- must reproduce the exact result.
* emulate_samples: the A operand the deformable (ALIGN) kernel builds, rounding for rounding.

Everything works on CPU and CUDA tensors alike.
"""
import torch

# precision (significand bits incl. the implicit one), minimum normal exponent, maximum exponent
FORMATS = {torch.bfloat16: (8, -126, 127), torch.float16: (11, -14, 15)}

# max(S) / q may use 20 of fp32's 24 significand bits: 4 bits of margin for the alignment of partial sums
BUDGET_BITS = 20


def _exponent(a, emin):
    """max(floor(log2 |a|), emin) of a float64 tensor (emin for zeros)."""
    _, e = torch.frexp(a)
    e = torch.where(a > 0, e - 1, torch.full_like(e, emin))
    return torch.clamp(e, min=emin)


def ulp(x, dtype):
    """Spacing of `dtype` values at |x| (float64 tensor): 2**(max(floor(log2|x|), emin) - p + 1); at 0 and in the
    subnormal range the subnormal spacing."""
    p, emin, _ = FORMATS[dtype]
    a = torch.as_tensor(x, dtype=torch.float64).abs()
    e = _exponent(a, emin).to(torch.int64) - (p - 1)
    return ((e + 1023) << 52).view(torch.float64)               # 2**e built from its bits: exact


def round_rne64(x, dtype):
    """x (float64) rounded once, to nearest even, to a `dtype` value; returned as float64 (exact)."""
    p, emin, emax = FORMATS[dtype]
    x = torch.as_tensor(x, dtype=torch.float64)
    q = ulp(x, dtype)
    r = torch.round(x / q) * q                   # x / q and the product are exact (q is a power of two)
    big = (2.0 - 2.0 ** (1 - p)) * 2.0 ** emax   # largest finite value
    r = torch.where(r.abs() > big, torch.copysign(torch.full_like(r, float("inf")), x), r)
    return torch.where(torch.isfinite(x), r, x)


def round_rne(x, dtype):
    """x (float64) rounded once, to nearest even, to `dtype`."""
    return round_rne64(x, dtype).to(dtype)      # exactly representable: the conversion does not round


def check_budget(S, q, dtype=None, ref=None, what=""):
    """Exactness budget.  S = the same operation on |inputs| (bounds every partial sum), q = the quantum every product
    is a multiple of.  max(S) / q <= 2**20 makes every partial sum an exact fp32 value, whatever the summation order.
    For fp16 outputs the exact result must also stay finite."""
    ratio = float(S.max()) / q
    assert ratio <= 2.0 ** BUDGET_BITS, "%s: exactness budget exceeded: max(S)/q = %.0f > 2**%d" % (what, ratio, BUDGET_BITS)
    if dtype == torch.float16 and ref is not None:
        assert float(ref.abs().max()) < 65504.0, "%s: reference overflows fp16" % what


def _fma64(a, b, c):
    """a * b + c for 16-bit values held in float64.  The product is exact (at most 22 significand bits); the sum is
    checked to be exact (TwoSum error term zero), so rounding it to 16 bits afterwards is a single rounding."""
    pr = a * b
    s = pr + c
    bb = s - pr
    err = (pr - (s - bb)) + (c - bb)
    assert bool((err == 0).all()), "emulate_samples: a blend sum is not exact in float64"
    return s


def emulate_samples(x16, offsets, dtype, round_positions, return_inexact=False):
    """The A operand of the tcgen05 deformable conv (conv_tc.cu build_tap_table + blend4) for a 3x3 kernel, pad 1,
    stride 1: samples[b, y, x, t, c] (float64, each a `dtype` value), tap t = 3 * i + j.

    * position h = fp32((y - 1 + i) + offset_h) (likewise w); with round_positions rounded to `dtype`
    * valid when -1 < h < H and -1 < w < W; otherwise every weight is 0
    * ly = h - floor(h), hy = 1 - ly in fp32 (hy, hx rounded to `dtype` first under round_positions only); the four
      corner weights are fp32 products rounded to `dtype`; a corner outside the map has weight 0
    * blend: t = r(w00 * v_tl); t = r(w01 * v_tr + t); t = r(w10 * v_bl + t); t = r(w11 * v_br + t), each r a single
      rounding to `dtype` (HMUL2 / HFMA2)

    This models the KERNEL.  With round_positions it is not the reference's scalar_t = half arithmetic bit for bit: the
    reference multiplies and adds separately in at::Half where the kernel fuses each step.
    x16 [B, C, H, W] of `dtype`; offsets [B, 18, H, W] (dy, dx per tap), fp32 or 16-bit.  With return_inexact, also the
    number of blend steps whose result was not already a `dtype` value."""
    B, C, H, W = x16.shape
    dev = x16.device
    r16 = lambda v: v.to(dtype).to(torch.float32)
    off = offsets.to(torch.float32)
    taps = torch.arange(9, device=dev)
    ti, tj = (taps // 3).view(1, 9, 1, 1), (taps % 3).view(1, 9, 1, 1)
    ys = torch.arange(H, device=dev).view(1, 1, H, 1)
    xs = torch.arange(W, device=dev).view(1, 1, 1, W)
    h = (ys - 1 + ti).to(torch.float32) + off[:, 0::2]          # [B, 9, H, W], one fp32 rounding
    w = (xs - 1 + tj).to(torch.float32) + off[:, 1::2]
    if round_positions:
        h, w = r16(h), r16(w)
    valid = (h > -1) & (w > -1) & (h < H) & (w < W)
    hf, wf = torch.floor(h), torch.floor(w)
    ly, lx = h - hf, w - wf
    hy, hx = 1.0 - ly, 1.0 - lx
    if round_positions:
        hy, hx = r16(hy), r16(hx)
    y0 = torch.where(valid, hf, torch.zeros_like(hf)).to(torch.int64)
    x0 = torch.where(valid, wf, torch.zeros_like(wf)).to(torch.int64)
    t_ok, b_ok, l_ok, r_ok = y0 >= 0, y0 + 1 <= H - 1, x0 >= 0, x0 + 1 <= W - 1
    zero = torch.zeros_like(h)
    wts = [torch.where(valid & a & b, r16(u * v), zero).to(torch.float64)
           for a, b, u, v in ((t_ok, l_ok, hy, hx), (t_ok, r_ok, hy, lx), (b_ok, l_ok, ly, hx), (b_ok, r_ok, ly, lx))]
    X = x16.to(torch.float64).permute(0, 2, 3, 1)                # [B, H, W, C]
    bi = torch.arange(B, device=dev).view(B, 1, 1, 1)
    yt, yb = y0.clamp(0, H - 1), (y0 + 1).clamp(0, H - 1)
    xl, xr = x0.clamp(0, W - 1), (x0 + 1).clamp(0, W - 1)
    corners = [X[bi, yy, xx] for yy, xx in ((yt, xl), (yt, xr), (yb, xl), (yb, xr))]     # [B, 9, H, W, C]
    inexact = 0
    t = None
    for k in range(4):
        e = wts[k][..., None] * corners[k] if t is None else _fma64(wts[k][..., None], corners[k], t)
        t = round_rne64(e, dtype)
        inexact += int((t != e).sum())
    s = t.permute(0, 2, 3, 1, 4).contiguous()                     # [B, H, W, 9, C]
    return (s, inexact) if return_inexact else s


def contract_samples(samples, weight):
    """y[b, co, y, x] = sum_{t, c} samples[b, y, x, t, c] * weight[co, c, t] in float64."""
    B, H, W, _, C = samples.shape
    Co = weight.size(0)
    wm = weight.to(torch.float64).reshape(Co, C, 9).permute(2, 1, 0).reshape(9 * C, Co)
    y = samples.reshape(B * H * W, 9 * C) @ wm.to(samples.device)
    return y.view(B, H, W, Co).permute(0, 3, 1, 2)


def quarter_offsets(B, H, W, g, spread=2.0):
    """[B, 18, H, W] float64 offsets on a 1/4 grid (CPU, from generator g): half of the sampling positions are the
    regular grid moved by up to `spread` pixels, the other half anywhere in [-3, H + 0.25] x [-3, W + 0.25] -- which
    puts positions exactly on -1, on H - 1 and W - 1, strictly between W - 1 and W, and outside the map."""
    off = torch.randint(int(-4 * spread), int(4 * spread) + 1, (B, 18, H, W), generator=g).double() / 4
    taps = torch.arange(9).view(1, 9, 1, 1)
    hh = torch.randint(-8, 4 * H + 5, (B, 9, H, W), generator=g).double() / 4 - 1
    ww = torch.randint(-8, 4 * W + 5, (B, 9, H, W), generator=g).double() / 4 - 1
    pick = torch.rand(B, 9, H, W, generator=g) < 0.5
    off[:, 0::2] = torch.where(pick, hh - (torch.arange(H).view(1, 1, H, 1) - 1 + taps // 3), off[:, 0::2])
    off[:, 1::2] = torch.where(pick, ww - (torch.arange(W).view(1, 1, 1, W) - 1 + taps % 3), off[:, 1::2])
    # and, whatever the draw, pixel (0, 0) of image 0 has these (h, w) at taps 0..5 (tap t sits at (t // 3 - 1, t % 3 - 1))
    for t, (ph, pw) in enumerate(((-1.0, 0.5), (-0.75, 0.25), (H - 1.0, W - 1.0), (0.5, W - 0.75), (H - 0.25, W - 0.25),
                                  (-0.25, -0.75))):
        off[0, 2 * t, 0, 0] = ph - (t // 3 - 1)
        off[0, 2 * t + 1, 0, 0] = pw - (t % 3 - 1)
    return off


def sampling_positions(offsets):
    """(h, w) [B, 9, H, W] of 3x3 / pad 1 offsets, in the offsets' dtype and device."""
    _, _, H, W = offsets.shape
    dev = offsets.device
    taps = torch.arange(9, device=dev).view(1, 9, 1, 1)
    h = offsets[:, 0::2] + (torch.arange(H, device=dev).view(1, 1, H, 1) - 1 + taps // 3)
    w = offsets[:, 1::2] + (torch.arange(W, device=dev).view(1, 1, 1, W) - 1 + taps % 3)
    return h, w
