"""High-precision references for the tensor-core and fp32 convolutions (csrc/conv_tc.cu, csrc/conv_f32.cu,
csrc/deform_bwd.cu).

* round_rne / ulp: correct round-to-nearest-even from float64 to bf16 / fp16.  torch's own float64 -> bf16 / fp16
  conversion goes through fp32 and so rounds twice (1 + 2**-8 + 2**-30 becomes 1.0 in bf16, not 1 + 2**-7).
* check_budget: the condition under which a kernel that accumulates in fp32 -- in any order, including the tensor
  core's aligned partial sums -- must reproduce the exact result.
* emulate_samples: the A operand the deformable (ALIGN) kernel builds, rounding for rounding.
* tf32_split: the hi / lo TF32 split of the fp32 tensor-core kernel (cvt.rna.tf32.f32 twice).
* geom_offsets / geom_positions / deform_grads_ref: offsets on a 1/4 grid and the float64 gradients for any kernel
  size, stride, padding, dilation and (deformable) group count.

Everything works on CPU and CUDA tensors alike.
"""
import pytest
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


# ------------------------------------------------------------------------------------------------------------------
# data and comparison shared by the exact tests
# ------------------------------------------------------------------------------------------------------------------
def ints(shape, r, g):
    return torch.randint(-r, r + 1, tuple(shape), generator=g).double()


def assert_exact(y, ref64, what):
    """y (16-bit, or fp32) == ref64 rounded once to y's dtype; for fp32 y, ref64 must itself be an fp32 value.  On
    failure: the count and the first mismatches with their (b, y, x, channel) for [B, C, H, W] tensors."""
    ref64 = ref64.to(y.device)
    if y.dtype in FORMATS:
        want, got = round_rne(ref64, y.dtype), y
    else:
        assert bool((ref64.float().double() == ref64).all()), "%s: the float64 reference is not an fp32 value" % what
        want, got = ref64, y.double()
    bad = got != want
    n = int(bad.sum())
    if n == 0:
        return
    idx = bad.nonzero()[:5].tolist()
    first = ", ".join("(b, y, x, c)=(%d, %d, %d, %d): got %r, want %r" % (i[0], i[2], i[3], i[1], float(got[tuple(i)]),
                      float(want[tuple(i)])) if len(i) == 4 else "%s: got %r want %r" % (i, float(got[tuple(i)]),
                      float(want[tuple(i)])) for i in idx)
    raise AssertionError("%s: %d of %d outputs differ from the float64 reference; first %s" % (what, n, bad.numel(), first))


def dyadic_anchors(B, H, W, stride, g):
    """[B, H, W, 5] anchors whose tap positions the kernel computes exactly: angle 0 (cosf = 1, sinf = 0), centres on
    a stride/4 grid, sizes 3 * stride * m / 4 (aw / 3.0f exact).  Centres move up to +-3 pixels, some by +-2.75 .. +-4
    (corners leave the 14 x 22 halo), some anchors have zero size and some lie off the map."""
    yy, xx = torch.meshgrid(torch.arange(H).double(), torch.arange(W).double(), indexing="ij")
    a = torch.zeros(B, H, W, 5, dtype=torch.float64)
    dx, dy = ints((B, H, W), 12, g) / 4, ints((B, H, W), 12, g) / 4
    far = torch.tensor([2.75, 3.0, 3.25, 4.0, -2.75, -3.0, -3.25, -4.0], dtype=torch.float64)
    pick = torch.rand(B, H, W, generator=g) < 0.25
    dx = torch.where(pick, far[torch.randint(0, 8, (B, H, W), generator=g)], dx)
    dy = torch.where(pick, far[torch.randint(0, 8, (B, H, W), generator=g)], dy)
    a[..., 0], a[..., 1] = (xx + dx) * stride, (yy + dy) * stride
    a[..., 2] = torch.randint(0, 13, (B, H, W), generator=g).double() * 3 * stride / 4
    a[..., 3] = torch.randint(0, 13, (B, H, W), generator=g).double() * 3 * stride / 4
    off_map = torch.rand(B, H, W, generator=g) < 0.03
    a[..., 0] = torch.where(off_map, torch.full_like(a[..., 0], -6.0 * stride), a[..., 0])
    return a


def align_offsets(anchors, H, W, stride):
    """[B, 18, H, W] AlignConv offsets of [B, H, W, 5] anchors, by the module's own get_offset (in anchors' dtype)."""
    from s2anet_b200.alignconv import AlignConv
    m = AlignConv(8, 8)
    return torch.stack([m.get_offset(anchors[i].reshape(-1, 5), (H, W), stride) for i in range(anchors.size(0))])


# ------------------------------------------------------------------------------------------------------------------
# the 3 x TF32 split (conv_tc.cu tf32_hi: cvt.rna.tf32.f32)
# ------------------------------------------------------------------------------------------------------------------
def tf32_round(v):
    """fp32 -> the nearest TF32 value (10 explicit mantissa bits), ties away from zero, as an fp32 tensor with its low
    13 bits zero: add half a TF32 step (0x1000) to the magnitude bits, clear the low 13 bits, keep the sign.  A carry
    out of the mantissa moves the exponent up, as it should; subnormals round on the same bits."""
    b = v.to(torch.float32).contiguous().view(torch.int32)
    mag = b & 0x7FFFFFFF
    r = ((mag + 0x1000) & ~0x1FFF) | (b & ~0x7FFFFFFF)
    return r.view(torch.float32)


def tf32_split(v):
    """(hi, lo) of fp32 v: hi = tf32_round(v), lo = tf32_round(v - hi) (v - hi is exact in fp32).  hi + lo == v for
    every v with at most 22 significant bits (unless lo is subnormal); for a TF32 tie (12 significant bits) lo is half a
    TF32 step of v, with the sign opposite to v's."""
    v = v.to(torch.float32)
    hi = tf32_round(v)
    return hi, tf32_round(v - hi)


def odd_fractions(shape, g):
    """fp64 values +-(1 + m 2**-11), m odd in [1, 2047]: 12 significant bits, so every one is a TF32 tie whose lo part is
    +-2**-11."""
    m = 2 * torch.randint(0, 1024, tuple(shape), generator=g) + 1
    s = torch.where(torch.rand(tuple(shape), generator=g) < 0.5, -1.0, 1.0).double()
    return s * (1.0 + m.double() * 2.0 ** -11)


# ------------------------------------------------------------------------------------------------------------------
# deformable geometry: any kernel size, stride, padding, dilation, deformable groups
# ------------------------------------------------------------------------------------------------------------------
def out_size(n, k, stride, pad, dil):
    return (n + 2 * pad - (dil * (k - 1) + 1)) // stride + 1


def _tap_bases(Ho, Wo, k, stride, pad, dil, dev=None):
    """Regular-grid positions [k*k, Ho, 1] (rows) and [k*k, 1, Wo] (columns) of each tap: ho*stride - pad + i*dil."""
    taps = torch.arange(k * k, device=dev).view(k * k, 1, 1)
    bh = torch.arange(Ho, device=dev).view(1, Ho, 1) * stride - pad + (taps // k) * dil
    bw = torch.arange(Wo, device=dev).view(1, 1, Wo) * stride - pad + (taps % k) * dil
    return bh, bw


# (h, w) that every geom_offsets draw contains: exactly -1, just inside -1, exactly (H - 1, W - 1), inside (W - 1, W),
# the far corner just inside the map, and a position inside -1 on both axes
EDGE_POSITIONS = lambda H, W: ((-1.0, 0.5), (-0.75, 0.25), (H - 1.0, W - 1.0), (0.5, W - 0.75), (H - 0.25, W - 0.25),
                               (-0.25, -0.75))


def geom_offsets(B, H, W, k, stride, pad, dil, dgroups, g, spread=2.0):
    """[B, dgroups*2*k*k, Ho, Wo] float64 offsets on a 1/4 grid for a k x k deformable conv (CPU, from generator g), in
    the reference's layout (deformable group, tap, (dy, dx)).  As quarter_offsets: half of the positions are the regular
    grid moved by up to `spread` pixels, half anywhere in [-3, H + 0.25] x [-3, W + 0.25]; and in every deformable
    group the first pixels carry EDGE_POSITIONS (entry s at tap s % k*k, pixel s // k*k in raster order)."""
    Ho, Wo = out_size(H, k, stride, pad, dil), out_size(W, k, stride, pad, dil)
    kk = k * k
    bh, bw = (t.double() for t in _tap_bases(Ho, Wo, k, stride, pad, dil))
    off = torch.randint(int(-4 * spread), int(4 * spread) + 1, (B, dgroups, kk, 2, Ho, Wo), generator=g).double() / 4
    hh = torch.randint(-8, 4 * H + 5, (B, dgroups, kk, Ho, Wo), generator=g).double() / 4 - 1
    ww = torch.randint(-8, 4 * W + 5, (B, dgroups, kk, Ho, Wo), generator=g).double() / 4 - 1
    pick = torch.rand(B, dgroups, kk, Ho, Wo, generator=g) < 0.5
    off[:, :, :, 0] = torch.where(pick, hh - bh, off[:, :, :, 0])
    off[:, :, :, 1] = torch.where(pick, ww - bw, off[:, :, :, 1])
    edges = EDGE_POSITIONS(H, W)
    assert Ho * Wo * kk >= len(edges), "geom_offsets: too few (pixel, tap) pairs for the edge positions"
    for s, (ph, pw) in enumerate(edges):
        t, (ho, wo) = s % kk, divmod(s // kk, Wo)
        off[0, :, t, 0, ho, wo] = ph - float(bh[t, ho, 0])
        off[0, :, t, 1, ho, wo] = pw - float(bw[t, 0, wo])
    return off.reshape(B, dgroups * 2 * kk, Ho, Wo)


def geom_positions(off, k, stride, pad, dil):
    """(h, w) [B, dgroups, k*k, Ho, Wo] of [B, dgroups*2*k*k, Ho, Wo] offsets, in the offsets' dtype and device."""
    B, ch, Ho, Wo = off.shape
    o = off.view(B, ch // (2 * k * k), k * k, 2, Ho, Wo)
    bh, bw = _tap_bases(Ho, Wo, k, stride, pad, dil, off.device)
    return o[:, :, :, 0] + bh, o[:, :, :, 1] + bw


def deform_grads_ref(x, off, w, go, stride=1, pad=1, dil=1):
    """torchvision's float64 autograd: (grad_input, grad_offset, grad_weight), with the offset gradient of a sampling
    position outside -1 < h < H, -1 < w < W set to 0.  That is the reference DCN's rule (its coordinate-weight kernel
    moves such positions to -2, where no corner is inside the map) and the one this repository's fp32 col2im and the
    tcgen05 dgrad follow.  torchvision differs only at h == -1 or w == -1 exactly: the sample is 0 there and its
    right-hand derivative is not, and torchvision returns that derivative.  Groups and deformable groups follow from
    the shapes of w and off, as in torchvision."""
    tv = pytest.importorskip("torchvision")
    x64 = x.detach().double().clone().requires_grad_(True)          # (a copy even when x already is float64)
    off64 = off.detach().to(x.device).double().clone().requires_grad_(True)
    w64 = w.detach().to(x.device).double().clone().requires_grad_(True)
    tv.ops.deform_conv2d(x64, off64, w64, stride=stride, padding=pad, dilation=dil).backward(go.to(x.device).double())
    H, W = x.shape[2:]
    h, ww = geom_positions(off64.detach(), w.size(-1), stride, pad, dil)
    outside = ~((h > -1) & (ww > -1) & (h < H) & (ww < W))                     # [B, dg, kk, Ho, Wo]
    outside = outside.unsqueeze(3).expand(-1, -1, -1, 2, -1, -1).reshape(off64.shape)
    goff = torch.where(outside, torch.zeros_like(off64.grad), off64.grad)
    return x64.grad, goff, w64.grad
