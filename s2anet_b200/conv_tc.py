"""Host side of the tcgen05 implicit-GEMM path (csrc/conv_tc.cu): channels-last bookkeeping and the
packed-weight cache.  Activations are bf16 / fp16 tensors in torch.channels_last memory format
(physically NHWC), which is what cuDNN's tensor-core convolutions around these ops produce, so
no layout copies happen inside a channels-last model."""
import weakref

import torch

from . import _lib

# Packed weights are cached per source TENSOR OBJECT (not per address: a freed weight's address is reused by the
# allocator): (id, dtype, kind) -> (weak refs to the sources, their versions, packed result).  An entry is valid only
# while every source is still the same live object at the same in-place version; entries die with their tensors.
_PACK_CACHE = {}


def _stamp(t):
    """What identifies the CONTENT a packed copy was made from.  `_version` alone is not enough: writes through
    `.data` (`w.data.copy_()`, `w.data = ...`, `Module.to()` / `.half()` which reassign `param.data`) do not bump it,
    but they either change the storage (data_ptr / device / dtype) or go through `.data`'s own version counter --
    so the stamp also carries the storage address, device, dtype and the version of the `.data` alias."""
    return (t._version, t.data_ptr(), t.device, t.dtype, tuple(t.shape), tuple(t.stride()))


def _cache_get(key, sources):
    hit = _PACK_CACHE.get(key)
    if hit is None:
        return None
    refs, stamps, value = hit
    if all(r() is t for r, t in zip(refs, sources)) and stamps == tuple(_stamp(t) for t in sources):
        return value
    return None


def _cache_put(key, sources, value):
    if len(_PACK_CACHE) > 256:
        _PACK_CACHE.clear()
    drop = lambda _ref, k=key: _PACK_CACHE.pop(k, None)
    _PACK_CACHE[key] = (tuple(weakref.ref(t, drop) for t in sources), tuple(_stamp(t) for t in sources), value)
    return value


def invalidate_pack_cache():
    """Drop every packed weight.  In-place writes through `.data` that keep the storage (`w.data.add_(1)`, an EMA or
    a clipping step written that way) are invisible to every stamp torch offers; code that does that calls this (or
    trains with grad enabled, which never uses the packed inference path)."""
    _PACK_CACHE.clear()


def _nhwc(x):
    """A [B,C,H,W] tensor whose memory is NHWC-contiguous (no copy if it already is)."""
    if x.dim() != 4:
        raise ValueError("expected a 4-D [B,C,H,W] tensor")
    if x.is_contiguous(memory_format=torch.channels_last):
        return x
    if x.is_cuda and x.is_contiguous() and x.element_size() in (2, 4) and not x.requires_grad:
        # the reference's layout: one pass of the library's own tiled transpose (torch's conversion runs at ~1.8 TB/s)
        B, C, H, W = x.shape
        y = torch.empty_like(x, memory_format=torch.channels_last)
        with torch.cuda.device(x.device):
            rc = _lib.load().s2a_transpose_planes(_lib.ptr(x), _lib.ptr(y), B, C, H * W, x.element_size(),
                                                  _lib.stream_ptr(x.device))
        _lib.check(rc, "transpose_planes")
        return y
    return x.contiguous(memory_format=torch.channels_last)


def nchw_from_nhwc(y, out):
    """Copy a channels_last [B,C,H,W] tensor into the NCHW-contiguous `out` of the same shape and dtype (the layout the
    reference's callers allocate) with the library's transpose; anything else falls back to Tensor.copy_."""
    if (y.is_cuda and y.dim() == 4 and y.shape == out.shape and y.dtype == out.dtype and out.is_contiguous() and
            y.is_contiguous(memory_format=torch.channels_last) and y.element_size() in (2, 4)):
        B, C, H, W = y.shape
        with torch.cuda.device(y.device):
            rc = _lib.load().s2a_transpose_planes(_lib.ptr(y), _lib.ptr(out), B, H * W, C, y.element_size(),
                                                  _lib.stream_ptr(y.device))
        _lib.check(rc, "transpose_planes")
        return out
    out.copy_(y if y.shape == out.shape else y.reshape(out.shape))
    return out


def pack_weight(weight, dtype, indices=None):
    """Pack (and cache) conv weights for the tensor-core kernel; ORConv banks go through the ARF map."""
    sources = (weight,) if indices is None else (weight, indices)
    key = (tuple(id(t) for t in sources), dtype, "arf")
    hit = _cache_get(key, sources)
    if hit is not None:
        return hit
    dev = weight.device
    w = weight.detach().contiguous()
    if indices is None:
        Co, C = w.size(0), w.size(1)
        nOri = nRot = 1
        idx = None
    else:
        O, I, nOri = w.size(0), w.size(1), w.size(2)
        nRot = indices.size(3)
        Co, C = O * nRot, I * nOri
        idx = indices.to(torch.uint8).contiguous()
    packed = torch.empty((Co, 9 * C), dtype=dtype, device=dev)
    with torch.cuda.device(dev):
        rc = _lib.load().s2a_conv_pack_weight(_lib.ptr(w), _lib.dtype_code(w), _lib.ptr(idx), _lib.ptr(packed),
                                              _lib.dtype_code(packed), Co, C, nOri, nRot, _lib.stream_ptr(dev))
    _lib.check(rc, "conv_pack_weight")
    return _cache_put(key, sources, packed)


def alignconv_forward_tc(x, anchors, weight, stride):
    """x [B,C,H,W] bf16/fp16 (channels_last preferred), anchors [B,H,W,5] -> relu(alignconv) as a
    channels_last [B,Co,H,W] tensor of x's dtype."""
    dev = _lib.require_cuda(x, anchors, weight)
    B, C, H, W = x.shape
    Co = weight.size(0)
    xc = _nhwc(x)
    a = anchors.to(torch.float32).contiguous()
    wp = pack_weight(weight, x.dtype)
    out = torch.empty((B, Co, H, W), dtype=x.dtype, device=dev, memory_format=torch.channels_last)
    with torch.cuda.device(dev):
        rc = _lib.load().s2a_alignconv_forward_tc(_lib.ptr(xc), _lib.ptr(a), _lib.ptr(wp), _lib.ptr(out), B, C, H, W, Co,
                                                  float(stride), _lib.dtype_code(xc), _lib.stream_ptr(dev))
    _lib.check(rc, "alignconv_forward_tc")
    return out


def tf32x3_supported(C, Co):
    """Shapes the fp32-on-tensor-cores kernel takes (3x3, stride / pad / dilation 1, one group assumed by the caller)."""
    return C > 0 and C % 32 == 0 and Co % 32 == 0 and 0 < Co <= 256


def pack_weight_tf32(weight, indices=None):
    """fp32 weights -> (hi, lo) TF32 planes [Co][9*C] for conv_forward_tf32x3 (cached); ORConv banks through the ARF map."""
    sources = (weight,) if indices is None else (weight, indices)
    key = (tuple(id(t) for t in sources), torch.float32, "tf32x3")
    hit = _cache_get(key, sources)
    if hit is not None:
        return hit
    dev = weight.device
    w = weight.detach().to(torch.float32).contiguous()
    if indices is None:
        Co, C = w.size(0), w.size(1)
        nOri = nRot = 1
        idx = None
    else:
        O, I, nOri = w.size(0), w.size(1), w.size(2)
        nRot = indices.size(3)
        Co, C = O * nRot, I * nOri
        idx = indices.to(torch.uint8).contiguous()
    hi = torch.empty((Co, 9 * C), dtype=torch.float32, device=dev)
    lo = torch.empty_like(hi)
    with torch.cuda.device(dev):
        rc = _lib.load().s2a_conv_pack_weight_tf32(_lib.ptr(w), _lib.ptr(idx), _lib.ptr(hi), _lib.ptr(lo), Co, C, nOri, nRot,
                                                   _lib.stream_ptr(dev))
    _lib.check(rc, "conv_pack_weight_tf32")
    return _cache_put(key, sources, (hi, lo))


def conv_forward_tf32x3(x, aux, mode, packed, bias=None, relu=False, stride=1.0, with_pool=False, out=None):
    """fp32 3x3 conv on tcgen05 with the 3 x TF32 split: mode 0 AlignConv (aux = anchors [B,H,W,5]), 1 generic
    deformable conv (aux = offsets [B,18,H,W]), 2 regular grid (ORConv2d).  x fp32 [B,C,H,W] (converted to
    channels_last once if it is not); returns NCHW-contiguous fp32 [B,Co,H,W] (+ pooled [B,Co/8,H,W])."""
    dev = _lib.require_cuda(x, aux, bias)
    hi, lo = packed
    B, C, H, W = x.shape
    Co = hi.size(0)
    xc = _nhwc(x.to(torch.float32))
    a = None if aux is None else aux.to(torch.float32).contiguous()
    b = None if bias is None else bias.detach().to(torch.float32).contiguous()
    if out is None or out.dtype != torch.float32 or not out.is_contiguous() or tuple(out.shape) != (B, Co, H, W):
        out = torch.empty((B, Co, H, W), dtype=torch.float32, device=dev)
    pooled = torch.empty((B, Co // 8, H, W), dtype=torch.float32, device=dev) if with_pool else None
    with torch.cuda.device(dev):
        rc = _lib.load().s2a_conv_forward_tf32x3(_lib.ptr(xc), _lib.ptr(a), int(mode), _lib.ptr(hi), _lib.ptr(lo), _lib.ptr(b),
                                                 _lib.ptr(out), _lib.ptr(pooled), B, C, H, W, Co, float(stride),
                                                 1 if relu else 0, _lib.stream_ptr(dev))
    _lib.check(rc, "conv_forward_tf32x3")
    return (out, pooled) if with_pool else out


def deform_conv_tc_supported(C, Co, kH, kW, dH, dW, padH, padW, dilH, dilW, group, deformable_group):
    """Shapes the tcgen05 deformable conv takes (everything S2ANet's AlignConv uses)."""
    return (kH == 3 and kW == 3 and dH == 1 and dW == 1 and padH == 1 and padW == 1 and dilH == 1 and dilW == 1 and
            group == 1 and deformable_group == 1 and C % 64 == 0 and Co % 32 == 0 and Co <= 256)


def deform_conv_forward_tc(x, offset, weight, out=None, relu=False, round_positions=None):
    """Generic 3x3 deformable convolution (explicit [B,18,H,W] offsets) on the tcgen05 kernel: the 16-bit route of
    `deform_conv_forward_cuda`.  x bf16/fp16 [B,C,H,W]; offset fp32 or x's dtype; returns (or fills `out`, if it is a
    channels_last tensor of x's dtype) a channels_last [B,Co,H,W].  round_positions=None: True for fp16 -- the
    reference's half kernel rounds the sampling positions and bilinear weights to half
    (deform_conv_cuda_kernel.cu:94-110, 223-224), which this reproduces -- and False for bf16, a dtype the reference
    does not dispatch (8 mantissa bits would move samples by up to half a pixel)."""
    dev = _lib.require_cuda(x, offset, weight)
    B, C, H, W = x.shape
    Co = weight.size(0)
    if tuple(offset.shape) != (B, 18, H, W):
        raise ValueError("offset must be [B,18,H,W] matching x")
    if round_positions is None:
        round_positions = x.dtype == torch.float16
    xc = _nhwc(x)
    off = offset if offset.dtype in (torch.float32, x.dtype) else offset.to(x.dtype)
    off = off.contiguous()
    wp = pack_weight(weight, x.dtype)
    if out is None or out.dtype != x.dtype or tuple(out.shape) != (B, Co, H, W) or \
            not out.is_contiguous(memory_format=torch.channels_last):
        out = torch.empty((B, Co, H, W), dtype=x.dtype, device=dev, memory_format=torch.channels_last)
    with torch.cuda.device(dev):
        rc = _lib.load().s2a_deform_conv_forward_tc(_lib.ptr(xc), _lib.ptr(off), _lib.dtype_code(off), _lib.ptr(wp),
                                                    _lib.ptr(out), B, C, H, W, Co, 1 if relu else 0,
                                                    1 if round_positions else 0, _lib.dtype_code(xc), _lib.stream_ptr(dev))
    _lib.check(rc, "deform_conv_forward_tc")
    return out


def deform_conv_dgrad_tc(grad_out, offset, weight, x=None, need_offset_grad=False):
    """Deformable-conv backward w.r.t. the input (3x3, stride / pad / dilation 1, one group) on the tcgen05 kernel:
    nine 1x1 implicit GEMMs grad_out x W_t^T whose accumulator tiles are scattered from tensor memory into grad_input
    with the bilinear weights -- no column buffer, no library GEMM.  grad_out [B,Co,H,W] bf16/fp16, offset [B,18,H,W]
    (fp32 or grad_out's dtype), weight [Co,C,3,3]; x [B,C,H,W] is only needed for the offset gradient.
    Returns (grad_input [B,C,H,W] fp32, channels_last; grad_offset [B,18,H,W] fp32 or None)."""
    dev = _lib.require_cuda(grad_out, offset, weight, x)
    B, Co, H, W = grad_out.shape
    C = weight.size(1)
    if tuple(weight.shape) != (Co, C, 3, 3) or tuple(offset.shape) != (B, 18, H, W):
        raise ValueError("deform_conv_dgrad_tc: shapes do not match a 3x3 deformable conv")
    dt = grad_out.dtype
    go = _nhwc(grad_out)
    off = offset if offset.dtype in (torch.float32, dt) else offset.to(dt)
    off = off.contiguous()
    # wd[t][c][co] = weight[co][c][t]: for a 1x1 conv with C_in = Co (a multiple of 64) this IS the packed layout
    wd = weight.detach().to(dt).permute(2, 3, 1, 0).reshape(9, C, Co).contiguous()
    gi = torch.zeros((B, H, W, C), dtype=torch.float32, device=dev)
    goff, xc = None, None
    if need_offset_grad:
        if x is None:
            raise ValueError("deform_conv_dgrad_tc: the offset gradient needs x")
        goff = torch.zeros((B, 18, H, W), dtype=torch.float32, device=dev)
        xc = _nhwc(x.to(dt))
    with torch.cuda.device(dev):
        rc = _lib.load().s2a_deform_conv_dgrad_tc(_lib.ptr(go), _lib.ptr(off), _lib.dtype_code(off), _lib.ptr(wd), _lib.ptr(xc),
                                                  _lib.ptr(gi), _lib.ptr(goff), B, C, H, W, Co, _lib.dtype_code(go),
                                                  _lib.stream_ptr(dev))
    _lib.check(rc, "deform_conv_dgrad_tc")
    return gi.permute(0, 3, 1, 2), goff


def deform_conv_wgrad_tc(x, offset, grad_out):
    """Deformable-conv backward w.r.t. the weight (3x3, stride / pad / dilation 1, one group; C, C_out in {128, 256})
    on tcgen05: dW[co,c,tap] = sum_pixels grad_out[pixel,co] * sample[pixel,tap,c] with both operands as MN-major
    shared-memory tiles and the accumulator in tensor memory -- no column buffer, no library GEMM.
    x [B,C,H,W], grad_out [B,Co,H,W] bf16/fp16; offset [B,18,H,W] fp32 or that dtype.  Returns fp32 [Co,C,3,3]."""
    dev = _lib.require_cuda(x, offset, grad_out)
    B, C, H, W = x.shape
    Co = grad_out.size(1)
    if tuple(offset.shape) != (B, 18, H, W) or tuple(grad_out.shape) != (B, Co, H, W):
        raise ValueError("deform_conv_wgrad_tc: shapes do not match a 3x3 deformable conv")
    dt = x.dtype
    xc, go = _nhwc(x), _nhwc(grad_out.to(dt))
    off = offset if offset.dtype in (torch.float32, dt) else offset.to(dt)
    off = off.contiguous()
    dwt = torch.zeros((9, Co, C), dtype=torch.float32, device=dev)
    with torch.cuda.device(dev):
        rc = _lib.load().s2a_deform_conv_wgrad_tc(_lib.ptr(xc), _lib.ptr(off), _lib.dtype_code(off), _lib.ptr(go), _lib.ptr(dwt),
                                                  B, C, H, W, Co, _lib.dtype_code(xc), _lib.stream_ptr(dev))
    _lib.check(rc, "deform_conv_wgrad_tc")
    return dwt.permute(1, 2, 0).reshape(Co, C, 3, 3)


def deform_conv_wgrad_tc_supported(C, Co, kH, kW, dH, dW, padH, padW, dilH, dilW, group, deformable_group):
    return (kH == 3 and kW == 3 and dH == 1 and dW == 1 and padH == 1 and padW == 1 and dilH == 1 and dilW == 1 and
            group == 1 and deformable_group == 1 and C in (128, 256) and Co in (128, 256))


def deform_conv_dgrad_tc_supported(C, Co, kH, kW, dH, dW, padH, padW, dilH, dilW, group, deformable_group):
    return (kH == 3 and kW == 3 and dH == 1 and dW == 1 and padH == 1 and padW == 1 and dilH == 1 and dilW == 1 and
            group == 1 and deformable_group == 1 and C % 32 == 0 and C <= 256 and Co % 64 == 0)


def orconv_forward_tc(x, weight, indices, bias, with_pool=False):
    dev = _lib.require_cuda(x, weight, indices, bias)
    B, C, H, W = x.shape
    O, I, nOri = weight.shape[:3]
    nRot = indices.size(3)
    Co = O * nRot
    if C != I * nOri:
        raise ValueError("input channels (%d) != I*nOrientation (%d)" % (C, I * nOri))
    xc = _nhwc(x)
    wp = pack_weight(weight, x.dtype, indices)
    b = None if bias is None else bias.detach().to(torch.float32).contiguous()
    out = torch.empty((B, Co, H, W), dtype=x.dtype, device=dev, memory_format=torch.channels_last)
    pooled = torch.empty((B, Co // 8, H, W), dtype=x.dtype, device=dev,
                         memory_format=torch.channels_last) if with_pool else None
    with torch.cuda.device(dev):
        rc = _lib.load().s2a_orconv_forward_tc(_lib.ptr(xc), _lib.ptr(wp), _lib.ptr(b), _lib.ptr(out), _lib.ptr(pooled),
                                               B, C, H, W, Co, _lib.dtype_code(xc), _lib.stream_ptr(dev))
    _lib.check(rc, "orconv_forward_tc")
    return (out, pooled) if with_pool else out


def _ptr_array(tensors):
    import ctypes as C
    return (C.c_void_p * len(tensors))(*[None if t is None else t.data_ptr() for t in tensors])


def _int_array(vals):
    import ctypes as C
    return (C.c_int * len(vals))(*[int(v) for v in vals])


def alignconv_forward_tc_multi(xs, anchors, weight, strides):
    """All FPN levels in one persistent launch: xs[l] [B,C,H_l,W_l] (16-bit), anchors[l] [B,H_l,W_l,5]."""
    import ctypes as C
    dev = _lib.require_cuda(*xs, *anchors, weight)
    B, Cc = xs[0].shape[:2]
    Co = weight.size(0)
    xc = [_nhwc(x) for x in xs]
    an = [a.to(torch.float32).contiguous() for a in anchors]
    wp = pack_weight(weight, xs[0].dtype)
    outs = [torch.empty((B, Co, x.size(2), x.size(3)), dtype=x.dtype, device=dev, memory_format=torch.channels_last)
            for x in xs]
    st = (C.c_float * len(xs))(*[float(s) for s in strides])
    with torch.cuda.device(dev):
        rc = _lib.load().s2a_alignconv_forward_tc_multi(len(xs), _ptr_array(xc), _ptr_array(an), _lib.ptr(wp),
                                                        _ptr_array(outs), _int_array([x.size(2) for x in xs]),
                                                        _int_array([x.size(3) for x in xs]), st, B, Cc, Co,
                                                        _lib.dtype_code(xc[0]), _lib.stream_ptr(dev))
    _lib.check(rc, "alignconv_forward_tc_multi")
    return outs


def orconv_forward_tc_multi(xs, weight, indices, bias, with_pool=False):
    dev = _lib.require_cuda(*xs, weight, indices, bias)
    B, Cc = xs[0].shape[:2]
    O, I, nOri = weight.shape[:3]
    nRot = indices.size(3)
    Co = O * nRot
    xc = [_nhwc(x) for x in xs]
    wp = pack_weight(weight, xs[0].dtype, indices)
    b = None if bias is None else bias.detach().to(torch.float32).contiguous()
    outs = [torch.empty((B, Co, x.size(2), x.size(3)), dtype=x.dtype, device=dev, memory_format=torch.channels_last)
            for x in xs]
    pooled = [torch.empty((B, Co // 8, x.size(2), x.size(3)), dtype=x.dtype, device=dev,
                          memory_format=torch.channels_last) for x in xs] if with_pool else [None] * len(xs)
    with torch.cuda.device(dev):
        rc = _lib.load().s2a_orconv_forward_tc_multi(len(xs), _ptr_array(xc), _lib.ptr(wp), _lib.ptr(b), _ptr_array(outs),
                                                     _ptr_array(pooled), _int_array([x.size(2) for x in xs]),
                                                     _int_array([x.size(3) for x in xs]), B, Cc, Co,
                                                     _lib.dtype_code(xc[0]), _lib.stream_ptr(dev))
    _lib.check(rc, "orconv_forward_tc_multi")
    return (outs, pooled) if with_pool else outs


def pack_conv2d_weight(weight, bias, dtype):
    """Pack (and cache) a stock [Co,C,ks,ks] conv weight (+ fp32 bias padded to Co_pad) for conv2d_forward_tc_multi."""
    sources = (weight,) if bias is None else (weight, bias)
    key = (tuple(id(t) for t in sources), dtype, "conv2d")
    hit = _cache_get(key, sources)
    if hit is not None:
        return hit
    dev = weight.device
    w = weight.detach().contiguous()
    Co, C, ks, ks2 = w.shape
    if ks != ks2 or ks not in (1, 3):
        raise ValueError("conv2d_forward_tc: square kernels of size 1 or 3 only")
    Co_pad, Cp = (Co + 31) // 32 * 32, (C + 63) // 64 * 64
    packed = torch.empty((Co_pad, ks * ks * Cp), dtype=dtype, device=dev)
    with torch.cuda.device(dev):
        rc = _lib.load().s2a_conv2d_pack_weight(_lib.ptr(w), _lib.dtype_code(w), _lib.ptr(packed), _lib.dtype_code(packed),
                                                Co, C, ks, _lib.stream_ptr(dev))
    _lib.check(rc, "conv2d_pack_weight")
    b = None
    if bias is not None:
        b = torch.zeros((Co_pad,), dtype=torch.float32, device=dev)
        b[:Co] = bias.detach().float()
    return _cache_put(key, sources, (packed, b, Co_pad, ks))


def conv2d_forward_tc_multi(xs, weight, bias=None, relu=False):
    """nn.Conv2d(C, Co, ks, stride 1, padding ks//2) (+ReLU) on all FPN levels in one persistent tcgen05 launch.
    xs[l] [B,C,H_l,W_l] bf16/fp16 -> [B,Co,H_l,W_l] channels_last views (of a Co_pad-channel buffer when Co % 32)."""
    dev = _lib.require_cuda(*xs, weight, bias)
    B, C = xs[0].shape[:2]
    if weight.size(1) != C:
        raise ValueError("conv2d_forward_tc: input has %d channels, weight expects %d" % (C, weight.size(1)))
    if C % 8:
        raise ValueError("conv2d_forward_tc: C must be a multiple of 8")
    packed, b, Co_pad, ks = pack_conv2d_weight(weight, bias, xs[0].dtype)
    xc = [_nhwc(x) for x in xs]
    outs = [torch.empty((B, Co_pad, x.size(2), x.size(3)), dtype=x.dtype, device=dev, memory_format=torch.channels_last)
            for x in xs]
    with torch.cuda.device(dev):
        rc = _lib.load().s2a_conv2d_forward_tc_multi(len(xs), _ptr_array(xc), _lib.ptr(packed), _lib.ptr(b), _ptr_array(outs),
                                                     _int_array([x.size(2) for x in xs]), _int_array([x.size(3) for x in xs]),
                                                     B, C, Co_pad, ks, 1 if relu else 0, _lib.dtype_code(xc[0]),
                                                     _lib.stream_ptr(dev))
    _lib.check(rc, "conv2d_forward_tc_multi")
    Co = weight.size(0)
    return outs if Co == Co_pad else [o[:, :Co] for o in outs]


def conv2d_forward_tc_fam_decode(xs, head, strides, anchor_scale, anchor_angle, wh_ratio_clip=1e-6):
    """decode.fam_decode(conv2d_forward_tc_multi(xs, head.weight, head.bias), strides, ...) in ONE launch, bit for bit,
    without writing the deltas: the FAM regression head (nn.Conv2d(C, 5, 1) with bias) decodes its output against the
    grid anchors in its epilogue.  xs[l] [B,C,H_l,W_l] bf16/fp16 -> refined anchors [B,H_l,W_l,5] fp32 per level."""
    w, b = head.weight, head.bias
    if w.dim() != 4 or tuple(w.shape[0:1]) + tuple(w.shape[2:]) != (5, 1, 1) or b is None:
        raise ValueError("conv2d_forward_tc_fam_decode: needs a 5-channel 1x1 head with bias")
    if tuple(head.stride) != (1, 1) or tuple(head.padding) != (0, 0) or tuple(head.dilation) != (1, 1) or head.groups != 1:
        raise ValueError("conv2d_forward_tc_fam_decode: the head must have stride 1, no padding, dilation 1, one group")
    if len(strides) != len(xs):
        raise ValueError("conv2d_forward_tc_fam_decode: one anchor stride per level")
    B, C = xs[0].shape[:2]
    if any(x.dim() != 4 or x.size(1) != w.size(1) for x in xs):
        raise ValueError("conv2d_forward_tc_fam_decode: inputs must be [B,%d,H,W]" % w.size(1))
    if C % 8:
        raise ValueError("conv2d_forward_tc_fam_decode: C must be a multiple of 8")
    dev = _lib.require_cuda(*xs, w, b)
    packed, bp, Co_pad, _ = pack_conv2d_weight(w, b, xs[0].dtype)
    xc = [_nhwc(x) for x in xs]
    refined = [torch.empty((B, x.size(2), x.size(3), 5), dtype=torch.float32, device=dev) for x in xs]
    import ctypes as C_
    st = (C_.c_float * len(xs))(*[float(s) for s in strides])
    with torch.cuda.device(dev):
        rc = _lib.load().s2a_conv2d_forward_tc_fam_decode(len(xs), _ptr_array(xc), _lib.ptr(packed), _lib.ptr(bp),
                                                          _ptr_array(refined), _int_array([x.size(2) for x in xs]),
                                                          _int_array([x.size(3) for x in xs]), st, B, C, Co_pad,
                                                          float(anchor_scale), float(anchor_angle), float(wh_ratio_clip),
                                                          _lib.dtype_code(xc[0]), _lib.stream_ptr(dev))
    _lib.check(rc, "conv2d_forward_tc_fam_decode")
    return refined


def conv2d_forward_tc_pair(xs0, weight0, bias0, xs1, weight1, bias1, relu=False):
    """Two convolutions of one shape class -- same C, padded C_out, kernel size, ReLU and batch, e.g. the
    classification and the regression tower layer of the head -- in ONE persistent launch (two launches of 682 tile
    groups fill the 74 CTA pairs to 92 %, one launch of 1,364 to 97 %).  Falls back to two launches when the shapes
    differ or the levels do not fit one launch.  Returns (outs0, outs1) like two conv2d_forward_tc_multi calls."""
    same = (weight0.shape[1:] == weight1.shape[1:] and (weight0.size(0) + 31) // 32 == (weight1.size(0) + 31) // 32 and
            xs0[0].dtype == xs1[0].dtype and xs0[0].size(0) == xs1[0].size(0) and len(xs0) + len(xs1) <= 16 and
            (bias0 is None) == (bias1 is None))
    if not same:
        return (conv2d_forward_tc_multi(xs0, weight0, bias0, relu=relu), conv2d_forward_tc_multi(xs1, weight1, bias1, relu=relu))
    xs = list(xs0) + list(xs1)
    dev = _lib.require_cuda(*xs, weight0, weight1, bias0, bias1)
    B, C = xs[0].shape[:2]
    if weight0.size(1) != C or any(x.size(1) != C for x in xs):
        raise ValueError("conv2d_forward_tc: input has %d channels, weight expects %d" % (C, weight0.size(1)))
    if C % 8:
        raise ValueError("conv2d_forward_tc: C must be a multiple of 8")
    p0, b0, Co_pad, ks = pack_conv2d_weight(weight0, bias0, xs[0].dtype)
    p1, b1, _, _ = pack_conv2d_weight(weight1, bias1, xs[0].dtype)
    xc = [_nhwc(x) for x in xs]
    outs = [torch.empty((B, Co_pad, x.size(2), x.size(3)), dtype=x.dtype, device=dev, memory_format=torch.channels_last)
            for x in xs]
    with torch.cuda.device(dev):
        rc = _lib.load().s2a_conv2d_forward_tc_multi2(len(xs), len(xs0), _ptr_array(xc), _lib.ptr(p0), _lib.ptr(p1),
                                                      _lib.ptr(b0), _lib.ptr(b1), _ptr_array(outs),
                                                      _int_array([x.size(2) for x in xs]), _int_array([x.size(3) for x in xs]),
                                                      B, C, Co_pad, ks, 1 if relu else 0, _lib.dtype_code(xc[0]),
                                                      _lib.stream_ptr(dev))
    _lib.check(rc, "conv2d_forward_tc_multi2")
    n0 = len(xs0)
    o0 = outs[:n0] if weight0.size(0) == Co_pad else [o[:, :weight0.size(0)] for o in outs[:n0]]
    o1 = outs[n0:] if weight1.size(0) == Co_pad else [o[:, :weight1.size(0)] for o in outs[n0:]]
    return o0, o1
