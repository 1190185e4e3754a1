"""Fused multiclass NMS above 6,144 boxes per image, exactly.

Up to MC_FUSED_MAX_BOXES boxes per image a segment's candidates are selected and sorted inside one CTA; above it they
are appended as rank keys and sorted by a device-wide segmented sort (csrc/nms_rotated.cu, mc_key_kernel).  The output
must not depend on the route: descending score, equal scores by ascending box, then ascending class, -0.0 == +0.0, as
oracle.multiclass_nms_rotated and the composition on the generic ml_nms_rotated kernel (`_multiclass_composed`) define
it.  The sizes are those of larger inputs: 6,720 boxes at 1536^2 and 21,824 at 1024^2 without the per-level top-k.
"""
import ctypes as C

import numpy as np
import pytest
import torch

from conftest import bits
from s2anet_b200 import synth

DEV = "cuda:0"
pytestmark = pytest.mark.gpu


def _sig(logits, dtype):
    return torch.sigmoid(torch.from_numpy(np.asarray(logits, np.float32)).to(dtype)).float().numpy()


def _boxes(n, seed):
    b = synth.clustered_boxes(n_seed=n // 4 + 1, rep=4, seed=seed)[0][:n]
    assert b.shape[0] == n
    return b


def _far_apart_boxes(n):
    """n boxes 100 px apart, 20 px wide: no pair overlaps, so nothing is suppressed"""
    i = np.arange(n)
    return np.stack([50.0 + 100.0 * (i % 40), 50.0 + 100.0 * (i // 40), np.full(n, 20.0), np.full(n, 12.0),
                     np.full(n, 0.3)], 1).astype(np.float32)


def check_multiclass(oracle, bb, sc, score_thr, iou_thr=0.5, max_per_img=2000):
    """multiclass_nms_rotated_batched on [B, n, 5] / [B, n, C] against the oracle (bits) and the generic composition
    (torch.equal), per image.  Returns the per-image counts."""
    from s2anet_b200.nms_rotated import _multiclass_composed, multiclass_nms_rotated_batched
    tb, ts = torch.from_numpy(bb).to(DEV), torch.from_numpy(sc).to(DEV)
    dets, labels, counts = multiclass_nms_rotated_batched(tb, ts, score_thr, iou_thr, max_per_img)
    out = []
    for b in range(bb.shape[0]):
        rd, rl = oracle.multiclass_nms_rotated(bb[b], sc[b], score_thr, iou_thr, max_per_img)
        k = int(counts[b])
        assert k == rd.shape[0], "image %d: %d detections, the oracle has %d" % (b, k, rd.shape[0])
        assert np.array_equal(bits(dets[b, :k].cpu().numpy()), bits(rd)), "image %d: dets differ from the oracle" % b
        assert np.array_equal(labels[b, :k].cpu().numpy(), rl)
        cd, cl = _multiclass_composed(tb[b], ts[b], score_thr, iou_thr, max_per_img)
        assert cd.shape[0] == k
        if k:
            assert torch.equal(dets[b, :k], cd) and torch.equal(labels[b, :k], cl.reshape(-1))
        out.append(k)
    return out


def _bench_density_batch(n, dtype, seed):
    """Batch 3, 15 classes: bench-density logits (about 0.56 candidates per box), no candidates, and the same density
    on logits rounded to steps of 0.25, so that a few scores are shared by most candidates of every class."""
    rng = np.random.default_rng(seed)
    C = 15
    bb = np.stack([_boxes(n, seed + i) for i in range(3)])
    logits = np.empty((3, n, C))
    logits[0] = rng.normal(-5.6, 1.5, (n, C))
    logits[1] = -10.0
    logits[2] = np.round(rng.normal(-5.6, 1.5, (n, C)) * 4.0) / 4.0
    return bb, _sig(logits, dtype)


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float16], ids=["bf16", "f16"])
@pytest.mark.parametrize("n", [6145, 6720, 8193, 21824])
def test_multiclass_many_boxes_on_tied_16bit_scores(oracle, dtype, n):
    bb, sc = _bench_density_batch(n, dtype, 300 + n)
    counts = check_multiclass(oracle, bb, sc, 0.05)
    assert counts[1] == 0 and counts[0] > 0 and counts[2] > 0
    for img in (0, 2):
        cand = sc[img][sc[img] > np.float32(0.05)]
        assert 0.4 * n < cand.size < 0.75 * n
        assert (np.diff(np.sort(cand)) == 0).sum() > cand.size // 8          # scores shared within and across classes
    assert np.unique(sc[2][sc[2] > np.float32(0.05)]).size < 40


@pytest.mark.parametrize("layout", ["far_apart", "clustered"])
def test_one_class_of_21824_candidates(oracle, layout):
    """Every box a candidate of one class.  Far apart: nothing is suppressed and max_per_img keeps the best 2,000 of
    21,824.  Clustered: suppression chains run across many 64-box blocks of the sweep."""
    n = 21824
    rng = np.random.default_rng(17)
    bb = _far_apart_boxes(n) if layout == "far_apart" else _boxes(n, 23)
    sc = _sig(rng.uniform(-2.0, 4.0, (n, 1)), torch.bfloat16)[None]
    assert (sc > np.float32(0.05)).all()
    if layout == "far_apart":
        assert check_multiclass(oracle, bb[None], sc, 0.05)[0] == 2000
    else:
        k = check_multiclass(oracle, bb[None], sc, 0.05, max_per_img=n)[0]
        assert 64 * 16 < k < n // 2                                            # kept across many blocks, most suppressed


def test_signed_zero_scores_rank_as_one_score(oracle):
    """score_thr < 0: +0.0 and -0.0 are candidates of one score, ordered by box and class like every tie."""
    rng = np.random.default_rng(12)
    n, C = 6145, 3
    bb = _boxes(n, 5)
    sc = np.where(rng.random((n, C)) < 0.5, np.float32(-0.0), np.float32(0.0)).astype(np.float32)
    sc[::7, 1] = np.float32(0.25)
    sc[::11, 2] = np.float32(-0.25)
    assert (np.signbit(sc) & (sc == 0)).any() and (~np.signbit(sc) & (sc == 0)).any()
    k = check_multiclass(oracle, bb[None], sc[None], -1.0, max_per_img=n * C)[0]
    assert k > 2000


@pytest.mark.parametrize("K", [300, 6000])
def test_packed_form_equals_plain_outputs(K):
    """Two destinations, image b at slot 2 + b: rows and count rows equal the plain outputs, other slots untouched."""
    from s2anet_b200.dist import packed_views
    from s2anet_b200.nms_rotated import multiclass_nms_rotated_batched, multiclass_nms_rotated_packed
    bb, sc = _bench_density_batch(6720, torch.bfloat16, 41)
    tb, ts = torch.from_numpy(bb).to(DEV), torch.from_numpy(sc).to(DEV)
    d, l, c = multiclass_nms_rotated_batched(tb, ts, 0.05, 0.5, K)
    dst0 = torch.full((6, K + 1, 8), -1.0, device=DEV)
    dst1 = torch.full((6, K + 1, 8), -1.0, device=DEV)
    multiclass_nms_rotated_packed(tb, ts, [dst0, dst1.data_ptr()], slot0=2, score_thr=0.05, iou_thr=0.5, max_per_img=K)
    assert torch.equal(dst0, dst1)
    assert bool((dst0[:2] == -1.0).all()) and bool((dst0[5] == -1.0).all())
    pd, pl, pc = packed_views(dst0[2:5], K)
    assert pc.tolist() == c.tolist() and int(c[1]) == 0
    assert (int(c.max()) == K) == (K == 300)                                   # K below, then above the kept count
    for i in range(3):
        k = int(c[i])
        assert torch.equal(pd[i, :k], d[i, :k]) and torch.equal(pl[i, :k], l[i, :k])
    assert bool((dst0[2:5, K, 1:] == 0).all())


def test_batched_replays_in_a_cuda_graph():
    """Captured once, replayed on new inputs copied into the static buffers: the eager call's outputs."""
    from s2anet_b200.nms_rotated import multiclass_nms_rotated_batched
    bb0, sc0 = _bench_density_batch(6720, torch.bfloat16, 51)
    bb1, sc1 = _bench_density_batch(6720, torch.float16, 52)
    tb, ts = torch.from_numpy(bb0).to(DEV), torch.from_numpy(sc0).to(DEV)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        multiclass_nms_rotated_batched(tb, ts, 0.05, 0.5, 2000)
    torch.cuda.current_stream().wait_stream(s)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        out = multiclass_nms_rotated_batched(tb, ts, 0.05, 0.5, 2000)
    for bb, sc in ((bb1, sc1), (bb0, sc0)):
        tb.copy_(torch.from_numpy(bb))
        ts.copy_(torch.from_numpy(sc))
        g.replay()
        want = multiclass_nms_rotated_batched(tb, ts, 0.05, 0.5, 2000)
        torch.cuda.synchronize()
        assert torch.equal(out[2], want[2]) and int(want[2][0]) > 0
        for b in range(3):
            k = int(want[2][b])
            assert torch.equal(out[0][b, :k], want[0][b, :k]) and torch.equal(out[1][b, :k], want[1][b, :k])


def test_detect_at_1536_pixels(oracle):
    """A bf16 head on 1536^2 features, batch 2 (6,720 boxes per image after the per-level top-2000): detect() equals
    the oracle on select_and_decode's outputs, replays in a CUDA graph, and detect_packed writes the same rows."""
    from s2anet_b200.dist import packed_views
    from s2anet_b200.head import S2ANetHead
    dtype = torch.bfloat16
    head = S2ANetHead(15)
    head.init_synthetic(0)
    head = head.eval().to(DEV).to(dtype)
    g = torch.Generator().manual_seed(3)
    feats = [torch.randn(2, 256, h, w, generator=g).to(dtype).to(DEV).contiguous(memory_format=torch.channels_last)
             for h, w in synth.level_shapes(img=1536)]
    head.calibrate_scores(feats, 3000)
    with torch.no_grad():
        bb, sc = head.select_and_decode(head.forward_levels(feats))
    assert bb.shape[1] == 6720
    dets, labels, counts = head.detect(feats)
    bbn, scn = bb.cpu().numpy(), sc.cpu().numpy()
    for b in range(2):
        rd, rl = oracle.multiclass_nms_rotated(bbn[b], scn[b], head.score_thres_before_nms, head.iou_thres_nms,
                                               head.max_per_img)
        k = int(counts[b])
        assert k == rd.shape[0] and k > 0
        assert np.array_equal(bits(dets[b, :k].cpu().numpy()), bits(rd))
        assert np.array_equal(labels[b, :k].cpu().numpy(), rl)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        gout = head.detect(feats)
    graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(gout[2], counts)
    for b in range(2):
        k = int(counts[b])
        assert torch.equal(gout[0][b, :k], dets[b, :k]) and torch.equal(gout[1][b, :k], labels[b, :k])
    K = head.max_per_img
    packed = torch.zeros((2, K + 1, 8), device=DEV)
    head.detect_packed(feats, [packed])
    pd, pl, pc = packed_views(packed, K)
    assert torch.equal(pc, counts)
    for b in range(2):
        k = int(counts[b])
        assert torch.equal(pd[b, :k], dets[b, :k]) and torch.equal(pl[b, :k], labels[b, :k])


def test_workspace_one_byte_short_is_refused():
    from s2anet_b200 import _lib
    lib = _lib.load()
    n, nc, B = 6720, 15, 2
    bb, sc = (torch.zeros((B, n, w), device=DEV) for w in (5, nc))
    dets = torch.empty((B, 10, 6), device=DEV)
    labels = torch.empty((B, 10), device=DEV)
    counts = torch.full((B,), -7, dtype=torch.int32, device=DEV)
    need = lib.s2a_multiclass_nms_rotated_workspace_bytes(n, nc, B)
    ws = torch.empty((need - 1,), dtype=torch.uint8, device=DEV)
    rc = lib.s2a_multiclass_nms_rotated(_lib.ptr(bb), _lib.ptr(sc), n, nc, B, 0.05, 0.5, 10, _lib.ptr(dets),
                                        _lib.ptr(labels), _lib.ptr(counts), 10, _lib.ptr(ws), need - 1, C.c_void_p(0))
    assert rc == -3 and b"workspace too small" in lib.s2a_last_error()
    dst = torch.zeros((B, 11, 8), device=DEV)
    ptrs = (C.c_void_p * 1)(dst.data_ptr())
    rc = lib.s2a_multiclass_nms_rotated_packed(_lib.ptr(bb), _lib.ptr(sc), n, nc, B, 0.05, 0.5, 10, ptrs, 1, 0, 10,
                                               _lib.ptr(ws), need - 1, C.c_void_p(0))
    assert rc == -3 and b"workspace too small" in lib.s2a_last_error()
    torch.cuda.synchronize()
    assert counts.tolist() == [-7, -7]                                         # nothing was launched
