"""nms_rotated / ml_nms_rotated / multiclass_nms_rotated with the reference's Python signatures.

reference: utils/nms_rotated/__init__.py:6-11, utils/ml_nms_rotated/__init__.py:1,
utils/bbox_nms_rotated.py:5-64 and the CUDA hosts they call (nms_rotated_cuda.cu:72-132,
ml_nms_rotated/src/nms_rotated_cuda.cu:74-137).
"""
import torch

from . import _lib, _torch_ext


def _nms_impl(dets, scores, labels, iou_threshold):
    dev = _lib.require_cuda(dets, scores, labels)
    n = dets.size(0)
    if n == 0:
        return torch.empty((0,), dtype=torch.int64, device=dev)
    if dets.dim() != 2 or dets.size(1) != 5:
        raise ValueError("dets must be [N,5]")
    ext = _torch_ext.module()
    if ext is not None:                 # the torch-extension binding: same C-ABI call, less host code per call
        keep = ext.nms_rotated(dets, scores, float(iou_threshold)) if labels is None else \
            ext.ml_nms_rotated(dets, scores, labels, float(iou_threshold))
        _lib.check(0, "nms_rotated")                                 # (launch accounting of bench.py's gpu_launches)
        return keep
    if dets.dtype != torch.float32 or dets.stride(1) != 1:
        dets = dets.to(torch.float32).contiguous()
    if scores.dtype != torch.float32:          # fp16 scores under half-precision validation (SURVEY A.7)
        scores = scores.to(torch.float32)
    if labels is not None and (labels.dtype != torch.float32 or labels.stride(0) != 1):
        labels = labels.to(torch.float32).contiguous()
    lib = _lib.load()
    ws_bytes = lib.s2a_nms_rotated_workspace_bytes(n)
    ws = torch.empty((ws_bytes,), dtype=torch.uint8, device=dev)
    keep = torch.empty((n,), dtype=torch.int64, device=dev)
    num = torch.empty((1,), dtype=torch.int32, device=dev)
    with torch.cuda.device(dev):
        rc = lib.s2a_nms_rotated(_lib.ptr(dets), dets.stride(0), _lib.ptr(scores), scores.stride(0),
                                 _lib.ptr(labels), n, float(iou_threshold), _lib.ptr(keep), _lib.ptr(num),
                                 _lib.ptr(ws), ws_bytes, _lib.stream_ptr(dev))
    _lib.check(rc, "nms_rotated")
    return keep[: int(num.item())]       # the only host sync: 4 bytes (the result's length)


def nms_rotated_op(dets, scores, iou_threshold):
    """extension-level call: `nms_rotated_cuda.nms_rotated(dets[N,5], scores[N], thr) -> keep int64`."""
    return _nms_impl(dets, scores, None, iou_threshold)


def ml_nms_rotated(dets, scores, labels, iou_threshold):
    """`ml_nms_rotated_cuda.ml_nms_rotated(dets[N,5], scores[N], labels[N], thr) -> keep int64`."""
    return _nms_impl(dets, scores, labels, iou_threshold)


def nms_rotated(dets, iou_thr):
    """reference wrapper utils/nms_rotated/__init__.py:6-11: dets [N,6] -> (dets[keep], keep);
    returns the bare (empty) tensor when N == 0, exactly like the reference."""
    if dets.shape[0] == 0:
        return dets
    keep_inds = nms_rotated_op(dets[:, :5], dets[:, 5], iou_thr)
    dets = dets[keep_inds, :]
    return dets, keep_inds


# kMcMaxBoxes in csrc/nms_rotated.cu: the most boxes per image whose per-class selection runs in one CTA.  The fused
# path takes any n; above this it selects with a device-wide segmented sort instead.
MC_FUSED_MAX_BOXES = 6144


def multiclass_nms_rotated_batched(bboxes, scores, score_thr=0.05, iou_thr=0.5, max_per_img=2000):
    """Fused, sync-free, batched form: bboxes [B,n,5], scores [B,n,C] ->
    (dets [B,max_per_img,6], labels [B,max_per_img] float32, counts [B] int32); rows >= counts[b]
    are unspecified.  No host round trip at any n: one call = 6 kernel launches for the whole batch up to
    MC_FUSED_MAX_BOXES boxes per image, plus the segmented sort's passes above it."""
    dev = _lib.require_cuda(bboxes, scores)
    B, n, _ = bboxes.shape
    C = scores.size(2)
    bboxes = bboxes.to(torch.float32).contiguous()
    scores = scores.to(torch.float32).contiguous()
    max_out = int(max(1, min(n * C, max_per_img)))
    dets = torch.empty((B, max_out, 6), dtype=torch.float32, device=dev)
    labels = torch.empty((B, max_out), dtype=torch.float32, device=dev)
    counts = torch.zeros((B,), dtype=torch.int32, device=dev)
    if B == 0 or n == 0 or C == 0:
        return dets, labels, counts
    if not (iou_thr >= 0):
        # A negative threshold, which the fused kernel does not take: per image, the reference's own composition on
        # the generic ml_nms_rotated kernel (one 4-byte host read per image), written into the same fixed-shape outputs.
        for b in range(B):
            d, l = _multiclass_composed(bboxes[b], scores[b], score_thr, iou_thr, max_per_img)
            k = d.size(0)
            if k:
                dets[b, :k] = d
                labels[b, :k] = l.reshape(-1)
            counts[b] = k
        return dets, labels, counts
    lib = _lib.load()
    ws_bytes = lib.s2a_multiclass_nms_rotated_workspace_bytes(n, C, B)
    ws = torch.empty((ws_bytes,), dtype=torch.uint8, device=dev)
    with torch.cuda.device(dev):
        rc = lib.s2a_multiclass_nms_rotated(_lib.ptr(bboxes), _lib.ptr(scores), n, C, B, float(score_thr),
                                            float(iou_thr), int(max_per_img), _lib.ptr(dets), _lib.ptr(labels),
                                            _lib.ptr(counts), max_out, _lib.ptr(ws), ws_bytes,
                                            _lib.stream_ptr(dev))
    _lib.check(rc, "multiclass_nms_rotated")
    if n > MC_FUSED_MAX_BOXES:
        _lib.launches += 1        # (a key and a gather kernel in place of the select kernel)
    return dets, labels, counts


def multiclass_nms_rotated_packed(bboxes, scores, dests, slot0=0, score_thr=0.05, iou_thr=0.5, max_per_img=2000, K=None):
    """The batched NMS writing PACKED rows into one or several [slots, K+1, 8] buffers (see
    s2a_multiclass_nms_rotated_packed): `dests` is a list of fp32 tensors and / or raw device pointers (ints: the
    NVLink-mapped buffers of peer ranks, dist.DetectionExchange.targets()); image b lands in slot slot0 + b.
    K (rows per image) defaults to dests[0].size(1) - 1.  Sync-free and graph-capturable at any n."""
    import ctypes as C
    dev = _lib.require_cuda(bboxes, scores)
    B, n, _ = bboxes.shape
    nc = scores.size(2)
    if K is None:
        K = dests[0].size(1) - 1
    if not (iou_thr >= 0):
        raise NotImplementedError("multiclass_nms_rotated_packed: the fused path takes iou_thr >= 0; "
                                  "use multiclass_nms_rotated_batched + dist.gather_detections")
    bboxes = bboxes.to(torch.float32).contiguous()
    scores = scores.to(torch.float32).contiguous()
    ptrs = (C.c_void_p * len(dests))(*[d.data_ptr() if torch.is_tensor(d) else int(d) for d in dests])
    lib = _lib.load()
    ws_bytes = lib.s2a_multiclass_nms_rotated_workspace_bytes(n, nc, B)
    ws = torch.empty((ws_bytes,), dtype=torch.uint8, device=dev)
    with torch.cuda.device(dev):
        rc = lib.s2a_multiclass_nms_rotated_packed(_lib.ptr(bboxes), _lib.ptr(scores), n, nc, B, float(score_thr),
                                                   float(iou_thr), int(max_per_img), ptrs, len(dests), int(slot0), int(K),
                                                   _lib.ptr(ws), ws_bytes, _lib.stream_ptr(dev))
    _lib.check(rc, "multiclass_nms_rotated_packed")
    if n > MC_FUSED_MAX_BOXES:
        _lib.launches += 1        # (a key and a gather kernel in place of the select kernel)


def _multiclass_composed(bboxes, scores, score_thr, iou_thr, max_per_img):
    """Negative thresholds, which the fused kernel does not take, and the tests' witness for it: the reference's
    own composition (utils/bbox_nms_rotated.py:24-64) on top of the generic ml_nms_rotated kernel."""
    num_classes = scores.size(1)
    boxes = bboxes[:, None].expand(-1, num_classes, 5)
    mask = scores > score_thr
    sc = scores[mask]
    boxes = boxes[mask]
    labels = mask.nonzero(as_tuple=False)[:, 1].to(boxes)
    if boxes.shape[0] == 0:
        return bboxes.new_zeros((0, 6)), bboxes.new_zeros((0, 1), dtype=torch.long)
    keep = ml_nms_rotated(boxes, sc, labels, iou_thr)
    boxes, sc, labels = boxes[keep], sc[keep], labels[keep]
    if keep.size(0) > max_per_img:
        boxes, sc, labels = boxes[:max_per_img], sc[:max_per_img], labels[:max_per_img]   # already score-sorted
    return torch.cat([boxes, sc[:, None]], dim=1), labels


def multiclass_nms_rotated(bboxes, scores, score_thr=0.05, iou_thr=0.5, max_per_img=2000):
    """reference signature (utils/bbox_nms_rotated.py:5-64): bboxes [n,5], scores [n,C] ->
    (dets [k,6], labels [k]); labels are float like the reference's `labels.to(bboxes)`, and the
    empty case returns ([0,6], [0,1] int64) like the reference's else-branch (:60-64)."""
    assert bboxes.shape[1] == 5
    if not (iou_thr >= 0):
        return _multiclass_composed(bboxes, scores, score_thr, iou_thr, max_per_img)
    dets, labels, counts = multiclass_nms_rotated_batched(bboxes[None], scores[None], score_thr, iou_thr,
                                                          max_per_img)
    k = int(counts[0].item())
    if k == 0:
        return bboxes.new_zeros((0, 6)), bboxes.new_zeros((0, 1), dtype=torch.long)
    return dets[0, :k].to(bboxes.dtype), labels[0, :k].to(bboxes.dtype)
