"""numpy/ctypes front-end of the CPU oracle (oracle/s2a_oracle.c) and of oracle/_ref.

TEST INFRASTRUCTURE ONLY: imported by tests/, __graft_entry__.smoke() and bench.py's
cpu_baseline / --impl reference legs -- never by s2anet_b200/.
"""
import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
_f32p = np.ctypeslib.ndpointer(dtype=np.float32, flags="C_CONTIGUOUS")
_i64p = np.ctypeslib.ndpointer(dtype=np.int64, flags="C_CONTIGUOUS")
_u8p = np.ctypeslib.ndpointer(dtype=np.uint8, flags="C_CONTIGUOUS")

_lib = None


def lib():
    global _lib
    if _lib is None:
        path = os.path.join(HERE, "libs2a_oracle.so")
        if not os.path.exists(path):
            from . import build_oracle
            build_oracle.build_oracle()
        L = C.CDLL(path)
        L.s2a_oracle_single_iou.restype = C.c_float
        L.s2a_oracle_single_iou.argtypes = [_f32p, _f32p]
        L.s2a_oracle_box_iou_rotated.restype = None
        L.s2a_oracle_box_iou_rotated.argtypes = [_f32p, C.c_int64, _f32p, C.c_int64, _f32p]
        L.s2a_oracle_nms_rotated.restype = C.c_int64
        L.s2a_oracle_nms_rotated.argtypes = [_f32p, _f32p, C.c_void_p, C.c_int64, C.c_float, C.c_int, _i64p]
        L.s2a_oracle_arf_forward.restype = None
        L.s2a_oracle_arf_forward.argtypes = [_f32p, _u8p] + [C.c_int] * 6 + [_f32p]
        L.s2a_oracle_arf_backward.restype = None
        L.s2a_oracle_arf_backward.argtypes = [_f32p, _u8p] + [C.c_int] * 6 + [_f32p]
        L.s2a_oracle_ri_pool.restype = None
        L.s2a_oracle_ri_pool.argtypes = [_f32p] + [C.c_int] * 5 + [_f32p]
        L.s2a_oracle_deform_conv_forward.restype = C.c_int
        L.s2a_oracle_deform_conv_forward.argtypes = [_f32p, _f32p, _f32p, _f32p] + [C.c_int] * 16
        L.s2a_oracle_alignconv_offset.restype = None
        L.s2a_oracle_alignconv_offset.argtypes = [_f32p, C.c_int, C.c_int, C.c_float, _f32p]
        L.s2a_oracle_alignconv_forward.restype = C.c_int
        L.s2a_oracle_alignconv_forward.argtypes = [_f32p, _f32p, _f32p, _f32p] + [C.c_int] * 5 + [C.c_float]
        L.s2a_oracle_conv2d.restype = None
        L.s2a_oracle_conv2d.argtypes = [_f32p, _f32p, C.c_void_p, _f32p] + [C.c_int] * 9
        L.s2a_oracle_orconv_forward.restype = None
        L.s2a_oracle_orconv_forward.argtypes = [_f32p, _f32p, _u8p, C.c_void_p, _f32p, C.c_void_p] + [C.c_int] * 11
        _lib = L
    return _lib


def _f32(a):
    return np.ascontiguousarray(a, dtype=np.float32)


def single_iou(b1, b2):
    return float(lib().s2a_oracle_single_iou(_f32(b1), _f32(b2)))


def box_iou_rotated(boxes1, boxes2):
    b1, b2 = _f32(boxes1).reshape(-1, 5), _f32(boxes2).reshape(-1, 5)
    out = np.empty((b1.shape[0], b2.shape[0]), np.float32)
    if out.size:
        lib().s2a_oracle_box_iou_rotated(b1, b1.shape[0], b2, b2.shape[0], out)
    return out


def nms_rotated(dets, scores, thr, labels=None, ge=False):
    """keep indices (int64, original order ids, descending score).  labels=None -> nms_rotated,
    else ml_nms_rotated.  ge=True selects the reference CPU build's >= predicate."""
    d, s = _f32(dets).reshape(-1, 5), _f32(scores).reshape(-1)
    n = d.shape[0]
    keep = np.empty(max(n, 1), np.int64)
    lab = None
    if labels is not None:
        lab = _f32(labels).reshape(-1)
    nk = lib().s2a_oracle_nms_rotated(d, s, None if lab is None else lab.ctypes.data, n, float(thr),
                                      int(bool(ge)), keep)
    return keep[:nk].copy()


def multiclass_nms_rotated(bboxes, scores, score_thr=0.05, iou_thr=0.5, max_per_img=2000):
    """utils/bbox_nms_rotated.py:5-64 restated on numpy: strict score threshold, row-major
    (box, class) expansion, ml-NMS, optional top-max_per_img re-sort.
    Returns (dets [k,6] = x,y,w,h,theta,score ; labels [k] float32)."""
    b, s = _f32(bboxes).reshape(-1, 5), _f32(scores)
    mask = s > np.float32(score_thr)
    bi, ci = np.nonzero(mask)                      # row-major order == torch boolean-mask order
    if bi.size == 0:
        return np.zeros((0, 6), np.float32), np.zeros((0,), np.float32)
    cb, cs, cl = b[bi], s[bi, ci], ci.astype(np.float32)
    keep = nms_rotated(cb, cs, iou_thr, labels=cl)
    cb, cs, cl = cb[keep], cs[keep], cl[keep]
    if keep.size > max_per_img:
        order = np.argsort(-cs, kind="stable")[:max_per_img]
        cb, cs, cl = cb[order], cs[order], cl[order]
    return np.concatenate([cb, cs[:, None]], 1), cl


def arf_forward(w, indices):
    w = _f32(w)
    O, I, nOri, kH, kW = w.shape
    idx = np.ascontiguousarray(indices, np.uint8)
    nRot = idx.shape[-1]
    out = np.zeros((O * nRot, I * nOri, kH, kW), np.float32)
    lib().s2a_oracle_arf_forward(w, idx.reshape(-1), O, I, nOri, kH, kW, nRot, out)
    return out


def arf_backward(indices, gout, O, I):
    idx = np.ascontiguousarray(indices, np.uint8)
    nOri, kH, kW, nRot = idx.shape
    g = _f32(gout)
    out = np.zeros((O, I, nOri, kH, kW), np.float32)
    lib().s2a_oracle_arf_backward(g, idx.reshape(-1), O, I, nOri, kH, kW, nRot, out)
    return out


def ri_pool(x, n_ori=8):
    x = _f32(x)
    B, Cc, H, W = x.shape
    out = np.empty((B, Cc // n_ori, H, W), np.float32)
    lib().s2a_oracle_ri_pool(x, B, Cc, H, W, n_ori, out)
    return out


def deform_conv_forward(x, offset, w, stride=(1, 1), padding=(0, 0), dilation=(1, 1), groups=1,
                        deformable_groups=1, relu=False):
    x, offset, w = _f32(x), _f32(offset), _f32(w)
    B, Cc, H, W = x.shape
    Co, _, kH, kW = w.shape
    Ho = (H + 2 * padding[0] - (dilation[0] * (kH - 1) + 1)) // stride[0] + 1
    Wo = (W + 2 * padding[1] - (dilation[1] * (kW - 1) + 1)) // stride[1] + 1
    out = np.empty((B, Co, Ho, Wo), np.float32)
    rc = lib().s2a_oracle_deform_conv_forward(x, offset, w, out, B, Cc, H, W, Co, kH, kW, stride[0], stride[1],
                                              padding[0], padding[1], dilation[0], dilation[1], groups,
                                              deformable_groups, int(relu))
    if rc != 0:
        raise ValueError("bad deform-conv geometry")
    return out


def alignconv_offset(anchors, H, W, stride):
    a = _f32(anchors).reshape(-1, 5)
    out = np.empty((18, H, W), np.float32)
    lib().s2a_oracle_alignconv_offset(a, H, W, float(stride), out)
    return out


def alignconv_forward(x, anchors, w, stride):
    x, anchors, w = _f32(x), _f32(anchors), _f32(w)
    B, Cc, H, W = x.shape
    Co = w.shape[0]
    out = np.empty((B, Co, H, W), np.float32)
    rc = lib().s2a_oracle_alignconv_forward(x, anchors, w, out, B, Cc, H, W, Co, float(stride))
    if rc != 0:
        raise ValueError("bad alignconv geometry")
    return out


def conv2d(x, w, bias=None, pad=1):
    x, w = _f32(x), _f32(w)
    B, Cc, H, W = x.shape
    Co, _, kH, kW = w.shape
    out = np.empty((B, Co, H + 2 * pad - kH + 1, W + 2 * pad - kW + 1), np.float32)
    b = None if bias is None else _f32(bias)
    lib().s2a_oracle_conv2d(x, w, None if b is None else b.ctypes.data, out, B, Cc, H, W, Co, kH, kW, pad, pad)
    return out


def orconv_forward(x, w, indices, bias=None, pad=1, pool_group=0):
    x, w = _f32(x), _f32(w)
    O, I, nOri, kH, kW = w.shape
    idx = np.ascontiguousarray(indices, np.uint8)
    nRot = idx.shape[-1]
    B, _, H, W = x.shape
    Ho, Wo = H + 2 * pad - kH + 1, W + 2 * pad - kW + 1
    out = np.empty((B, O * nRot, Ho, Wo), np.float32)
    pooled = np.empty((B, O * nRot // pool_group, Ho, Wo), np.float32) if pool_group else None
    b = None if bias is None else _f32(bias)
    lib().s2a_oracle_orconv_forward(x, w, idx.reshape(-1), None if b is None else b.ctypes.data, out,
                                    None if pooled is None else pooled.ctypes.data, B, H, W, O, I, nOri, kH, kW,
                                    nRot, pad, pool_group)
    return (out, pooled) if pool_group else out


def arf_indices(n_orientation=1, n_rotation=8, k=3):
    """models/orn/modules/ORConv.py:41-75 (get_indices) restated: uint8 [nOri, k, k, nRot],
    1-based destination entry for source tap l under rotation 45deg*r."""
    import math
    table = {
        1: {a: (1,) for a in range(0, 360, 45)},
        3: {0: (1, 2, 3, 4, 5, 6, 7, 8, 9), 45: (2, 3, 6, 1, 5, 9, 4, 7, 8), 90: (3, 6, 9, 2, 5, 8, 1, 4, 7),
            135: (6, 9, 8, 3, 5, 7, 2, 1, 4), 180: (9, 8, 7, 6, 5, 4, 3, 2, 1), 225: (8, 7, 4, 9, 5, 1, 6, 3, 2),
            270: (7, 4, 1, 8, 5, 2, 9, 6, 3), 315: (4, 1, 2, 7, 5, 3, 8, 9, 6)},
    }
    d_ori, d_rot = 360 / n_orientation, 360 / n_rotation
    idx = np.zeros((n_orientation * k * k, n_rotation), np.uint8)
    for i in range(n_orientation):
        for j in range(k * k):
            for r in range(n_rotation):
                angle = d_rot * r
                layer = (i + math.floor(angle / d_ori)) % n_orientation
                idx[i * k * k + j, r] = int(layer * k * k + table[k][int(angle)][j])
    return idx.reshape(n_orientation, k, k, n_rotation)


# ---- oracle/_ref: the reference's own code compiled in place (see build_oracle.py) -------

def ref_lib(tag, sem):
    """tag in {iou, nms, ml}; sem in {cpu, cudasem}.  Returns (CDLL, prefix) or None if absent."""
    path = os.path.join(HERE, "_ref", "libref_%s_%s.so" % (tag, sem))
    if not os.path.exists(path):
        return None
    L = C.CDLL(path)
    pre = "ref_%s_%s_" % (tag, sem)
    f = getattr(L, pre + "single_iou")
    f.restype, f.argtypes = C.c_float, [_f32p, _f32p]
    g = getattr(L, pre + "pairwise")
    g.restype, g.argtypes = None, [_f32p, C.c_int64, _f32p, C.c_int64, _f32p]
    return L, pre


def ref_pairwise(tag, sem, boxes1, boxes2):
    r = ref_lib(tag, sem)
    if r is None:
        return None
    L, pre = r
    st = 6 if tag == "ml" else 5
    b1, b2 = _f32(boxes1).reshape(-1, st), _f32(boxes2).reshape(-1, st)
    out = np.empty((b1.shape[0], b2.shape[0]), np.float32)
    getattr(L, pre + "pairwise")(b1, b1.shape[0], b2, b2.shape[0], out)
    return out


# ------------------------------------------------------------------------------------------------
# box decode stages (numpy restatement; fp32 step by step like the reference's elementwise torch ops)
# ------------------------------------------------------------------------------------------------
def norm_angle(a):
    """utils/general.py:925-930: (a - (-pi/4)) % pi + (-pi/4) in fp32 (Python/torch remainder sign rule)."""
    a = _f32(a)
    lo = np.float32(-np.pi / 4)
    return (np.mod(a - lo, np.float32(np.pi)) + lo).astype(np.float32)


def delta2bbox_rotated(anchors, deltas, wh_ratio_clip=16 / 1000):
    """models/boxes.py:82-162 (is_encode_relative=True).  anchors [...,5] fp32; deltas [...,5] float32 or
    float16 -- a float16 input keeps the reference's half-precision steps (clamp, exp and pi*dangle are
    evaluated on the half tensor, SURVEY Appendix A.7) before meeting the fp32 anchors."""
    anchors = _f32(anchors)
    dt = np.float16 if deltas.dtype == np.float16 else np.float32
    d = np.asarray(deltas, dtype=dt)
    lim = dt(abs(np.log(wh_ratio_clip)))                       # torch.clamp converts its bounds to the tensor dtype
    dx, dy = d[..., 0].astype(np.float32), d[..., 1].astype(np.float32)
    dw = np.clip(d[..., 2], -lim, lim)
    dh = np.clip(d[..., 3], -lim, lim)
    with np.errstate(over="ignore"):               # fp16 exp overflows to inf at the 1e-6 clip, as in torch
        ew = np.exp(dw.astype(np.float32)).astype(dt).astype(np.float32)
        eh = np.exp(dh.astype(np.float32)).astype(dt).astype(np.float32)
    pda = (d[..., 4].astype(np.float32) * np.float32(np.pi)).astype(dt).astype(np.float32)
    rx, ry, rw, rh, ra = (anchors[..., i] for i in range(5))
    cosa, sina = np.cos(ra), np.sin(ra)
    gx = dx * rw * cosa - dy * rh * sina + rx
    gy = dx * rw * sina + dy * rh * cosa + ry
    gw = rw * ew
    gh = rh * eh
    ga = norm_angle(pda + ra)
    return np.stack([gx, gy, gw, gh, ga], axis=-1).astype(np.float32)


def grid_anchors(H, W, stride, scale=4.0, angle=0.0):
    """models/anchors.py:75-126 for one square anchor per location -> [H, W, 5] fp32."""
    s = np.float32(stride)
    xs = np.arange(W, dtype=np.float32) * s + np.float32(0.5) * (s - np.float32(1))
    ys = np.arange(H, dtype=np.float32) * s + np.float32(0.5) * (s - np.float32(1))
    a = np.zeros((H, W, 5), np.float32)
    a[..., 0] = xs[None, :]
    a[..., 1] = ys[:, None]
    a[..., 2] = a[..., 3] = s * np.float32(scale)
    a[..., 4] = np.float32(angle)
    return a


def fam_decode(fam_bbox_pred, stride, scale=4.0, angle=0.0, wh_ratio_clip=1e-6):
    """models/head.py:27-52: fam_bbox_pred [B,5,H,W] -> refined anchors [B,H,W,5]."""
    B, _, H, W = fam_bbox_pred.shape
    d = np.transpose(fam_bbox_pred, (0, 2, 3, 1))
    return delta2bbox_rotated(grid_anchors(H, W, stride, scale, angle)[None], d, wh_ratio_clip)


def sigmoid_in(x):
    dt = np.float16 if x.dtype == np.float16 else np.float32
    xf = np.asarray(x, np.float32)
    return (np.float32(1) / (np.float32(1) + np.exp(-xf))).astype(dt)


def select_decode(cls_preds, bbox_preds, anchors, topk=2000, wh_ratio_clip=16 / 1000):
    """models/head.py:684-717 for a batch: per level sigmoid, top-k by best class score (descending, NaN
    first, ties by ascending location), gather; concatenate levels; decode.  Returns (bboxes [B,n,5] fp32,
    scores [B,n,C] fp32, index [B,n] int32)."""
    B = cls_preds[0].shape[0]
    out_b, out_s, out_i = [], [], []
    for b in range(B):
        sl, dl, al, il = [], [], [], []
        for cls, reg, anc in zip(cls_preds, bbox_preds, anchors):
            C, H, W = cls.shape[1:]
            sc = sigmoid_in(np.transpose(cls[b], (1, 2, 0)).reshape(H * W, C))
            de = np.transpose(reg[b], (1, 2, 0)).reshape(H * W, 5)
            an = _f32(anc[b]).reshape(H * W, 5)
            idx = np.arange(H * W)
            if topk > 0 and H * W > topk:
                best = sc.max(axis=1).astype(np.float32)                # NaN if any class is NaN, like torch.max
                idx = np.lexsort((idx, -best, ~np.isnan(best)))[:topk]  # NaN first, like torch.topk
            sl.append(sc[idx].astype(np.float32)); dl.append(de[idx]); al.append(an[idx]); il.append(idx.astype(np.int32))
        out_b.append(delta2bbox_rotated(np.concatenate(al), np.concatenate(dl), wh_ratio_clip))
        out_s.append(np.concatenate(sl)); out_i.append(np.concatenate(il))
    return np.stack(out_b), np.stack(out_s), np.stack(out_i)


def assign_labels(anchors, gt_boxes, imgs_size=(1024, 1024), pos_iou_thr=0.5, neg_iou_thr=0.4, min_pos_iou_thr=0,
                  gt_max_assign_all=True, filter_invalid_anchors=True, ious=None):
    """models/utils.py:33-147 restated with numpy on top of the oracle IoU (or a given IoU matrix)."""
    anchors, gt_boxes = _f32(anchors), _f32(gt_boxes)
    M, N = anchors.shape[0], gt_boxes.shape[0]
    out = np.full(M, -2, np.int64)
    flags = np.ones(M, bool)
    if filter_invalid_anchors:                                                        # :71-77
        flags = ((anchors[:, 0] >= 0) & (anchors[:, 1] >= 0) & (anchors[:, 0] <= imgs_size[1]) & (anchors[:, 1] <= imgs_size[0])
                 & (anchors[:, 2] < imgs_size[1]) & (anchors[:, 3] < imgs_size[0]))
    if N == 0:                                                                        # :79-86
        out[flags] = -1
        return out
    iou = (box_iou_rotated(anchors, gt_boxes) if ious is None else np.array(ious, np.float32)).copy()
    iou[(iou < 0) | (iou > 1)] = -0.5                                                 # :89-96
    iou[~flags] = -0.5                                                                # :99-100
    mx, arg = iou.max(axis=1), iou.argmax(axis=1)                                     # :115 (first index of the maximum)
    out[(mx >= 0) & (mx < neg_iou_thr)] = -1                                          # :116
    pos = mx >= pos_iou_thr
    out[pos] = arg[pos]                                                               # :122-123
    gmx, garg = iou.max(axis=0), iou.argmax(axis=0)                                   # :128
    for i in range(N):                                                                # :130-144
        if gmx[i] > min_pos_iou_thr:
            if gt_max_assign_all:
                out[iou[:, i] == gmx[i]] = i
            else:
                out[garg[i]] = i
    return out


# ---- DOTA result-merging NMS (fp64 polygons): oracle/poly_oracle.c and oracle/_ref/libref_polyiou.so -----------

_f64p = np.ctypeslib.ndpointer(dtype=np.float64, flags="C_CONTIGUOUS")


def _poly_lib():
    L = lib()
    if not getattr(L, "_poly_ready", False):
        L.s2a_oracle_poly_iou_pairs.restype = None
        L.s2a_oracle_poly_iou_pairs.argtypes = [_f64p, _f64p, C.c_int64, _f64p]
        L.s2a_oracle_poly_nms.restype = C.c_int64
        L.s2a_oracle_poly_nms.argtypes = [_f64p, C.c_int64, C.c_int64, C.c_double, _i64p]
        L._poly_ready = True
    return L


def poly_iou_pairs(p, q):
    """polyiou.cpp:110-126 for n pairs: p, q [n, 8] float64 -> [n]."""
    p = np.ascontiguousarray(p, dtype=np.float64)
    q = np.ascontiguousarray(q, dtype=np.float64)
    out = np.empty((p.shape[0],), dtype=np.float64)
    _poly_lib().s2a_oracle_poly_iou_pairs(p, q, p.shape[0], out)
    return out


def poly_nms(dets, thresh):
    """ResultMerge_multi_process.py:62-123: dets [n, 9] float64 -> kept row indices (descending score)."""
    dets = np.ascontiguousarray(dets, dtype=np.float64)
    n = dets.shape[0]
    keep = np.empty((max(n, 1),), dtype=np.int64)
    k = _poly_lib().s2a_oracle_poly_nms(dets, dets.shape[1], n, float(thresh), keep)
    return keep[:k].copy()


def ref_polyiou():
    """The reference's own iou_poly compiled in place (oracle/_ref/libref_polyiou.so), or None."""
    path = os.path.join(HERE, "_ref", "libref_polyiou.so")
    if not os.path.exists(path):
        return None
    L = C.CDLL(path)
    L.ref_iou_poly_pairs.restype = None
    L.ref_iou_poly_pairs.argtypes = [_f64p, _f64p, C.c_int64, _f64p]
    return L


def ref_poly_iou_pairs(p, q):
    L = ref_polyiou()
    if L is None:
        return None
    p = np.ascontiguousarray(p, dtype=np.float64)
    q = np.ascontiguousarray(q, dtype=np.float64)
    out = np.empty((p.shape[0],), dtype=np.float64)
    L.ref_iou_poly_pairs(p, q, p.shape[0], out)
    return out


def ref_py_cpu_nms_poly_fast(dets, thresh=0.5):
    """py_cpu_nms_poly_fast line by line (ResultMerge_multi_process.py:62-123), numpy as in the reference, with the
    reference's compiled iou_poly for the pair values.  Used to generate and to pin the golden keep lists."""
    L = ref_polyiou()
    assert L is not None, "oracle/_ref/libref_polyiou.so is not built"
    dets = np.asarray(dets, dtype=np.float64)
    obbs = dets[:, 0:-1]
    x1 = np.min(obbs[:, 0::2], axis=1)
    y1 = np.min(obbs[:, 1::2], axis=1)
    x2 = np.max(obbs[:, 0::2], axis=1)
    y2 = np.max(obbs[:, 1::2], axis=1)
    scores = dets[:, 8]
    areas = (x2 - x1 + 1) * (y2 - y1 + 1)
    order = scores.argsort()[::-1]
    keep = []
    while order.size > 0:
        i = order[0]
        keep.append(int(i))
        xx1 = np.maximum(x1[i], x1[order[1:]])
        yy1 = np.maximum(y1[i], y1[order[1:]])
        xx2 = np.minimum(x2[i], x2[order[1:]])
        yy2 = np.minimum(y2[i], y2[order[1:]])
        w = np.maximum(0.0, xx2 - xx1)
        h = np.maximum(0.0, yy2 - yy1)
        hbb_inter = w * h
        hbb_ovr = hbb_inter / (areas[i] + areas[order[1:]] - hbb_inter)
        h_inds = np.where(hbb_ovr > 0)[0]
        tmp_order = order[h_inds + 1]
        if tmp_order.size:
            pi = np.ascontiguousarray(np.repeat(obbs[i][None, :], tmp_order.size, axis=0))
            hbb_ovr[h_inds] = ref_poly_iou_pairs(pi, np.ascontiguousarray(obbs[tmp_order]))
        inds = np.where(hbb_ovr <= thresh)[0]
        order = order[inds + 1]
    return np.asarray(keep, dtype=np.int64)
