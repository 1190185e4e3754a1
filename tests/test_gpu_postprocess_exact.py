"""Detection post-processing, exactly: select_decode (sigmoid, per-level top-k, gather, decode) and the fused
multiclass NMS, against plain references at the tie density 16-bit inference produces.

16-bit sigmoid scores tie all the time (a bf16 score has 8 significant bits), so the output order is decided by
the tie rules, and those are what this file pins down:

  * per-level top-k: descending best class score, equal scores by ascending location (`reference_topk`);
  * multiclass NMS: descending score, then ascending box, then ascending class -- the order in which
    utils/bbox_nms_rotated.py expands (box, class) candidates, with a stable score sort.  oracle.multiclass_nms_rotated
    and the composition on the generic ml_nms_rotated kernel (`_multiclass_composed`) both define it so.

Inputs cover the head's real layout (15 and 5 channels of 32-channel channels-last buffers, whose pad channels are
poisoned here so that any read past C changes the result), boundary tie groups larger than the part that is kept,
fp16 subnormal and zero scores, +-0.0 scores, NaN scores and scores equal to the threshold.

Non-finite logits (NaN ranked first, as torch.max and torch.topk rank it) are tested in test_gpu_decode_exact.py.
"""
import numpy as np
import pytest
import torch

from conftest import bits
from s2anet_b200 import synth
from decode_reference import DeviceMath, assert_same

DEV = "cuda:0"


# ------------------------------------------------------------------------------------------------
# reference
# ------------------------------------------------------------------------------------------------
def reference_topk(scores, topk):
    """scores [n, C] of one (image, level), any float dtype -> the locations the per-level top-k keeps, in output
    order: all n in location order when topk <= 0 or n <= topk, else the topk best by max-over-classes score,
    descending, equal scores by ascending location.  As in the reference (torch.max, then torch.topk), a location with
    a NaN class has a NaN best score, and NaN ranks above every number."""
    n = scores.shape[0]
    if topk <= 0 or n <= topk:
        return np.arange(n)
    best = np.asarray(scores, np.float64).max(axis=1)
    return np.lexsort((np.arange(n), -best, ~np.isnan(best)))[:topk]


def boundary_tie(scores, keep):
    """(size of the tie group of the last kept location's best score, how many of that group are kept)"""
    best = np.asarray(scores, np.float64).max(axis=1)
    kth = best[keep[-1]]
    return int((best == kth).sum()), int((best[keep] == kth).sum())


def _nhwc(x):
    B, C, H, W = x.shape
    return x.permute(0, 2, 3, 1).reshape(B, H * W, C)


def check_select_decode(cls, reg, anchors, topk):
    """select_decode on the levels against reference_topk, with scores and gathers checked as well, and the boxes bit
    for bit against the decode model (tests/decode_reference.py).
    Returns [(image, level, n, k, tie group size, kept part of it)] for every level that selects."""
    from s2anet_b200.decode import select_decode
    B, C = cls[0].shape[:2]
    fp32 = cls[0].dtype == torch.float32
    bb, sc, idx = select_decode(cls, reg, anchors, topk, return_index=True)
    bb0, sc0 = select_decode(cls, reg, anchors, 0)
    ties = []
    off = off0 = 0
    for l, (c, r, a) in enumerate(zip(cls, reg, anchors)):
        n = c.size(2) * c.size(3)
        k = min(n, topk) if topk > 0 else n
        torch_sc = _nhwc(c).sigmoid().float()
        if fp32:       # the kernel's own scores: fp32 ties come from equal logits, independent of expf's last bit
            ref_sc = sc0[:, off0:off0 + n]
            assert float((ref_sc - torch_sc).abs().max()) <= 2e-7
        else:          # the reference's formula in the network dtype on the same GPU
            ref_sc = torch_sc
            assert torch.equal(sc0[:, off0:off0 + n], ref_sc)
        ref_np = ref_sc.cpu().numpy()
        want = np.stack([reference_topk(ref_np[b], topk) for b in range(B)])
        ii = idx[:, off:off + k].long()
        assert torch.equal(ii, torch.from_numpy(want).to(DEV)), "level %d: top-k index differs" % l
        assert torch.equal(sc[:, off:off + k], ref_sc.gather(1, ii[..., None].expand(-1, -1, C)))
        assert torch.equal(bb[:, off:off + k], bb0[:, off0:off0 + n].gather(1, ii[..., None].expand(-1, -1, 5)))
        an, dl = a.reshape(B, n, 5).cpu().numpy(), _nhwc(r).float().cpu().numpy()
        an, dl = np.stack([an[b][want[b]] for b in range(B)]), np.stack([dl[b][want[b]] for b in range(B)])
        want_b = DeviceMath(DEV).decode(an, dl, c.dtype, 16 / 1000)
        assert_same(bb[:, off:off + k].cpu().numpy(), want_b, "level %d: boxes differ from the decode model" % l)
        if n > k:
            for b in range(B):
                ties.append((b, l, n, k) + boundary_tie(ref_np[b], want[b]))
        off += k
        off0 += n
    assert off == bb.size(1) and off0 == bb0.size(1)
    return ties, (bb, sc, idx)


# ------------------------------------------------------------------------------------------------
# A. the reference has a witness of its own (CPU)
# ------------------------------------------------------------------------------------------------
def test_reference_topk_agrees_with_the_oracle(oracle, golden):
    g = golden("decode_small.npz")
    L = len(g["strides"])
    cls = [g["cls_%d" % l] for l in range(L)]
    reg = [g["reg_%d" % l] for l in range(L)]
    anc = [g["refine_%d" % l] for l in range(L)]
    topk = int(g["topk"])

    def per_level(cls, reg, anc, topk):
        _, _, oi = oracle.select_decode(cls, reg, anc, topk=topk)
        off, selecting = 0, 0
        for c in cls:
            B, C, H, W = c.shape
            k = min(H * W, topk) if topk > 0 else H * W
            for b in range(B):
                sc = oracle.sigmoid_in(np.transpose(c[b], (1, 2, 0)).reshape(H * W, C))
                want = reference_topk(sc, topk)
                assert np.array_equal(oi[b, off:off + k], want)
                if H * W > k:
                    selecting += 1
            off += k
        assert off == oi.shape[1]
        return selecting

    assert per_level(cls, reg, anc, topk) > 0
    # tie-heavy fp16: logits on a coarse grid, so the boundary of every selecting level is inside a tie group
    rng = np.random.default_rng(3)
    cls16 = [np.round(rng.normal(-3.0, 1.0, c.shape) * 2) / 2 for c in cls]
    cls16 = [c.astype(np.float16) for c in cls16]
    reg16 = [r.astype(np.float16) for r in reg]
    k16 = 40
    assert per_level(cls16, reg16, anc, k16) > 0
    for c in cls16:
        B, C, H, W = c.shape
        if H * W > k16:
            for b in range(B):
                sc = oracle.sigmoid_in(np.transpose(c[b], (1, 2, 0)).reshape(H * W, C))
                group, kept = boundary_tie(sc, reference_topk(sc, k16))
                assert group > kept


def test_reference_topk_definition():
    sc = np.array([[0.1, 0.5], [0.5, 0.2], [0.3, 0.3], [0.5, 0.5], [0.9, 0.0]], np.float16)
    assert reference_topk(sc, 3).tolist() == [4, 0, 1]         # ties at 0.5: locations 0, 1, 3 -> lowest first
    assert reference_topk(sc, 0).tolist() == [0, 1, 2, 3, 4]
    assert reference_topk(sc, 5).tolist() == [0, 1, 2, 3, 4]   # n == k: no selection, location order
    assert boundary_tie(sc, reference_topk(sc, 3)) == (3, 2)


# ------------------------------------------------------------------------------------------------
# B. select_decode matrix (GPU)
# ------------------------------------------------------------------------------------------------
# per-level top-k sizes, each with a level of exactly n == k and one of n == k + 1 locations
_EDGE = {0: ((9, 11), (13, 1)), 1: ((1, 1), (1, 2)), 2000: ((40, 50), (23, 87)), 2048: ((32, 64), (3, 683)),
         2049: ((3, 683), (41, 50)), 4096: ((64, 64), (17, 241))}


def _levels(kind, topk):
    if kind == "one":
        return [(113, 145)]
    # 16,384 locations: keys in shared memory; 16,385: keys in global memory; odd maps and 1 x 1
    return [(128, 128), (113, 145), (37, 53), (1, 1), *_EDGE[topk], (5, 7), (2, 3)]


def _logits(kind, C, H, W, g):
    n = H * W
    if kind == "random":
        return torch.randn(C, n, generator=g) * 2.0 - 3.0
    if kind == "equal":
        return torch.full((C, n), 0.25)
    if kind == "tiny":          # fp16 sigmoids of these are subnormals and exact zeros
        return -12.0 - 6.0 * torch.rand(C, n, generator=g)
    assert kind == "quantised"
    # best class score on three values (top one at half the locations), the other classes on two lower values
    x = torch.where(torch.rand(C, n, generator=g) < 0.5, -4.0, -3.0)
    u = torch.rand(n, generator=g)
    best = torch.where(u < 0.5, 1.0, torch.where(u < 0.75, 0.0, -2.0))
    x[torch.randint(0, C, (n,), generator=g), torch.arange(n)] = best
    return x


def _place(vals, layout, dtype, poison):
    """vals [B, C, H, W] fp32 (CPU) -> a CUDA view of `layout` holding vals in `dtype`; channels next to it hold
    `poison`."""
    B, C, H, W = vals.shape
    v = vals.to(dtype)
    if layout == "nchw":
        out = v.to(DEV).contiguous()
    elif layout == "cl":
        out = v.to(DEV).contiguous(memory_format=torch.channels_last)
    elif layout == "padded":    # the head's prediction convs: C channels of a 32-channel channels-last buffer
        buf = torch.full((B, 32, H, W), poison, dtype=dtype, device=DEV).contiguous(memory_format=torch.channels_last)
        out = buf[:, :C]
        out.copy_(v)
    else:                       # channels-last, one element past a 16-byte boundary: the scalar loads
        assert layout == "misaligned"
        buf = torch.full((B, H, W, C + 1), poison, dtype=dtype, device=DEV).permute(0, 3, 1, 2)
        out = buf[:, 1:]
        out.copy_(v)
        assert out.data_ptr() % 16 != 0
    assert_same(out.float().cpu().numpy(), v.float().numpy())           # (NaN == NaN)
    return out


def _inputs(dtype, layout, C, sizes, kinds, seed):
    g = torch.Generator().manual_seed(seed)
    B = len(kinds)
    cls, reg, anc = [], [], []
    for H, W in sizes:
        logit = torch.stack([_logits(k, C, H, W, g).reshape(C, H, W) for k in kinds])
        delta = torch.randn(B, 5, H, W, generator=g) * torch.tensor([0.3, 0.3, 0.6, 0.6, 0.4]).view(1, 5, 1, 1)
        a = torch.rand(B, H, W, 5, generator=g) * torch.tensor([1024.0, 1024.0, 56.0, 56.0, 3.1]) + \
            torch.tensor([0.0, 0.0, 8.0, 8.0, -0.78])
        cls.append(_place(logit, layout, dtype, 30.0))         # a poison logit would win every location
        reg.append(_place(delta, layout, dtype, 50.0))
        anc.append(a.to(DEV))
    return cls, reg, anc


_MATRIX = [
    # (layout, C, topk, levels)
    ("padded", 15, 2000, "eight"),       # the head's odm_cls / odm_reg layout and top-k
    ("padded", 9, 4096, "eight"),
    ("padded", 8, 2048, "eight"),
    ("padded", 16, 2049, "one"),
    ("padded", 17, 0, "eight"),
    ("padded", 1, 1, "eight"),
    ("cl", 15, 2049, "eight"),
    ("cl", 8, 1, "one"),
    ("nchw", 15, 2048, "eight"),
    ("nchw", 17, 4096, "one"),
    ("misaligned", 15, 2000, "eight"),
    ("misaligned", 16, 4096, "eight"),
]


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16, torch.float16], ids=["f32", "bf16", "f16"])
@pytest.mark.parametrize("layout,C,topk,levels", _MATRIX, ids=["%s-C%d-k%d-%s" % m for m in _MATRIX])
def test_select_decode_matrix(dtype, layout, C, topk, levels, monkeypatch):
    from s2anet_b200.decode import select_decode
    kinds = ["random", "equal", "quantised"] + (["tiny"] if dtype == torch.float16 else [])
    sizes = _levels(levels, topk)
    cls, reg, anc = _inputs(dtype, layout, C, sizes, kinds, seed=1000 * len(layout) + 100 * C + topk)
    monkeypatch.delenv("S2A_DEC_DEBUG", raising=False)
    ties, split = check_select_decode(cls, reg, anc, topk)
    # every boundary of the equal image, and of the quantised one on levels of 1,024 locations or more, falls inside
    # a tie group larger than its kept part; the subnormal fp16 scores tie at some boundary
    for b, l, n, k, group, kept in ties:
        if kinds[b] == "equal" or (kinds[b] == "quantised" and n >= 1024):
            assert group > kept, "image %d (%s), level %d: the top-k boundary is not inside a tie group" % (b, kinds[b], l)
    for kind in kinds[2:]:
        if topk > 0:
            assert any(kinds[b] == kind and group > kept for b, _, _, _, group, kept in ties), kind
    monkeypatch.setenv("S2A_DEC_DEBUG", "2")                   # the single-launch form
    single = select_decode(cls, reg, anc, topk, return_index=True)
    for a, b in zip(split, single):
        assert torch.equal(a, b)


@pytest.mark.gpu
def test_topk_above_4096_is_refused():
    from s2anet_b200.decode import select_decode
    cls, reg, anc = _inputs(torch.bfloat16, "padded", 15, [(113, 145)], ["random"], seed=1)
    select_decode(cls, reg, anc, 4096)
    with pytest.raises(RuntimeError):
        select_decode(cls, reg, anc, 4097)


# ------------------------------------------------------------------------------------------------
# C. fused multiclass NMS against the oracle on tied scores (GPU)
# ------------------------------------------------------------------------------------------------
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


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float16], ids=["bf16", "f16"])
@pytest.mark.parametrize("n", [150, 1024, 1025, 2048, 2049, 5344, 6144])
def test_multiclass_on_tied_16bit_scores(oracle, dtype, n):
    """Batch 3: bench-density scores (about 0.56 candidates per box, 3,000 at 5,344 boxes), no candidates, and all
    candidates at one score.  n covers the select-sort instantiations (1, 2 and 6 items per thread) and the fused
    path's maximum."""
    rng = np.random.default_rng(n)
    C = 15
    bb = np.stack([_boxes(n, 100 + n + i) for i in range(3)])
    logits = np.empty((3, n, C))
    logits[0] = rng.normal(-5.6, 1.5, (n, C))
    logits[1] = -10.0
    logits[2] = -10.0
    logits[2, :, :2] = 0.0
    sc = _sig(logits, dtype)
    counts = check_multiclass(oracle, bb, sc, 0.05)
    assert counts[1] == 0 and counts[0] > 0 and counts[2] > 0
    cand = int((sc[0] > np.float32(0.05)).sum())
    assert 0.4 * n < cand < 0.75 * n
    if n >= 1024:                                             # candidates sharing a score with another one
        assert (np.diff(np.sort(sc[0][sc[0] > np.float32(0.05)])) == 0).sum() > cand // 8


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float16], ids=["bf16", "f16"])
def test_multiclass_class_segments_cross_64_box_blocks(oracle, dtype):
    """Classes with 63, 64, 65 and 129 candidates on tied scores: the per-class sweep crosses 64-box mask blocks."""
    rng = np.random.default_rng(9)
    n, segs = 1024, (63, 64, 65, 129)
    bb = _boxes(n, 77)[None]
    logits = np.full((n, len(segs)), -10.0)
    for c, s in enumerate(segs):
        rows = rng.choice(n, s, replace=False)
        logits[rows, c] = rng.choice([0.5, 1.0, 1.5], s)
    sc = _sig(logits, dtype)[None]
    assert [(sc[0, :, c] > np.float32(0.05)).sum() for c in range(len(segs))] == list(segs)
    k = check_multiclass(oracle, bb, sc, 0.05)[0]
    assert k < sum(segs)                                      # something was suppressed


@pytest.mark.gpu
def test_multiclass_max_per_img_cuts_a_tie_group_across_classes(oracle):
    """One score shared by three classes of 20 boxes, nothing suppressed, max_per_img inside that group: the rows
    kept from it come by box, then by class."""
    n, C = 100, 5
    bb = _far_apart_boxes(n)
    sc = np.zeros((n, C), np.float32)
    sc[50:75, 0] = np.float32(0.6) + np.arange(25, dtype=np.float32) * np.float32(0.01)     # 25 distinct, above
    tie = np.float32(0.5)
    for c in (1, 2, 4):
        sc[10:30, c] = tie
    sc[80:, 3] = np.float32(0.2) + np.arange(20, dtype=np.float32) * np.float32(0.001)
    max_per_img = 25 + 31
    from s2anet_b200.nms_rotated import multiclass_nms_rotated_batched
    k = check_multiclass(oracle, bb[None], sc[None], 0.05, 0.5, max_per_img)[0]
    assert k == max_per_img
    dets, labels, _ = multiclass_nms_rotated_batched(torch.from_numpy(bb[None]).to(DEV), torch.from_numpy(sc[None]).to(DEV),
                                                     0.05, 0.5, max_per_img)
    rows = dets[0, 25:k].cpu().numpy()
    want_box = [10 + j // 3 for j in range(31)]
    want_cls = [(1, 2, 4)[j % 3] for j in range(31)]
    assert np.array_equal(rows[:, 5], np.full(31, tie))
    assert np.array_equal(rows[:, :5], bb[want_box])
    assert labels[0, 25:k].cpu().numpy().tolist() == want_cls


@pytest.mark.gpu
def test_multiclass_threshold_edge_and_nan_scores(oracle):
    """A score equal to float32(score_thr) is dropped, the next float above it is kept, NaN scores are dropped."""
    n, C = 60, 3
    bb = _far_apart_boxes(n)
    thr = np.float32(0.05)
    sc = np.zeros((n, C), np.float32)
    sc[0:10, 0] = thr
    sc[10:20, 0] = np.nextafter(thr, np.float32(1))
    sc[20:30, 1] = np.nan
    sc[30:40, 1] = np.float32(0.5)
    sc[40:50, 2] = np.nan
    sc[45:60, 2] = np.nextafter(thr, np.float32(1))
    k = check_multiclass(oracle, bb[None], sc[None], 0.05)[0]
    assert k == 10 + 10 + 15


@pytest.mark.gpu
def test_signed_zero_scores_are_one_score(oracle):
    """With score_thr < 0, +0.0 and -0.0 are candidates of equal score, ordered by box and class like any tie (the
    oracle and torch compare them equal).  The generic nms_rotated and ml_nms_rotated sort them the same way."""
    from s2anet_b200.nms_rotated import ml_nms_rotated, nms_rotated_op
    rng = np.random.default_rng(12)
    n, C = 300, 3
    far = _far_apart_boxes(n)
    near = _boxes(n, 5)
    for bb in (far, near):
        sc = np.where(rng.random((n, C)) < 0.5, np.float32(-0.0), np.float32(0.0)).astype(np.float32)
        sc[::7, 1] = np.float32(0.25)
        sc[::11, 2] = np.float32(-0.25)
        assert (np.signbit(sc) & (sc == 0)).any() and (~np.signbit(sc) & (sc == 0)).any()
        k = check_multiclass(oracle, bb[None], sc[None], -1.0)[0]
        assert k > 0
        tb = torch.from_numpy(bb).to(DEV)
        for c in range(C):
            s = np.ascontiguousarray(sc[:, c])
            got = nms_rotated_op(tb, torch.from_numpy(s).to(DEV), 0.5).cpu().numpy()
            assert np.array_equal(got, oracle.nms_rotated(bb, s, 0.5))
        flat_b = np.repeat(bb, C, 0)
        flat_s = sc.reshape(-1).copy()
        flat_l = np.tile(np.arange(C, dtype=np.float32), n)
        got = ml_nms_rotated(torch.from_numpy(flat_b).to(DEV), torch.from_numpy(flat_s).to(DEV),
                             torch.from_numpy(flat_l).to(DEV), 0.5).cpu().numpy()
        assert np.array_equal(got, oracle.nms_rotated(flat_b, flat_s, 0.5, labels=flat_l))


# ------------------------------------------------------------------------------------------------
# D. end to end: detect() at the bench's shape
# ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float16], ids=["bf16", "f16"])
def test_detect_equals_the_references_at_the_bench_shape(oracle, dtype):
    from bench import CALIBRATED_BIAS, build_head, make_feats
    from s2anet_b200.decode import select_decode
    head = build_head(torch, torch.device(DEV), dtype, seed=0, bias=CALIBRATED_BIAS[3000])
    feats = make_feats(torch, 2, 4, torch.device(DEV), dtype)
    head.calibrate_scores(feats, 3000)
    topk = head.max_before_nms_per_level
    with torch.no_grad():
        outs = head.forward_levels(feats)
    cls, reg, anc = [o[2] for o in outs], [o[3] for o in outs], [o[5] for o in outs]
    # the head's padded channels-last views: the paired key loads and the vectorised gathers
    assert cls[0].size(1) == 15 and cls[0].stride(1) == 1 and cls[0].stride(3) == 32 and reg[0].stride(3) == 32
    ties, (bb, sc, _) = check_select_decode(cls, reg, anc, topk)
    want_bb, want_sc = head.select_and_decode(outs)
    assert torch.equal(bb, want_bb) and torch.equal(sc, want_sc)
    dets, labels, counts = head.detect(feats)
    bbn, scn = bb.cpu().numpy(), sc.cpu().numpy()
    shared = 0
    for b in range(bb.size(0)):
        rd, rl = oracle.multiclass_nms_rotated(bbn[b], scn[b], head.score_thres_before_nms, head.iou_thres_nms,
                                               head.max_per_img)
        k = int(counts[b])
        assert k == rd.shape[0] and k > 0
        assert np.array_equal(bits(dets[b, :k].cpu().numpy()), bits(rd))
        assert np.array_equal(labels[b, :k].cpu().numpy(), rl)
        shared += int((np.diff(rd[:, 5]) == 0).sum())
    assert shared > 0, "no two kept detections share a score"
    assert any(l == 0 and group > kept for _, l, _, _, group, kept in ties), "no P3 top-k boundary inside a tie group"
