"""GPU parity tests (-m gpu) for box_iou_rotated, nms_rotated, ml_nms_rotated and
multiclass_nms_rotated: CUDA path (through the C ABI) vs the CPU oracle, the golden vectors
produced by the reference, and -- when oracle/_ref/ext_gpu was prebuilt -- the reference's own
CUDA kernels compiled for sm_100a and run on this box.

Bars (BASELINE.json north_star): IoU within 1e-5 absolute of the reference (here: bit-exact
against the oracle, i.e. against the reference header's device-side semantics without FMA
contraction; only a box whose fp32 sin/cos may round differently on the device than in glibc
(rbox_sets.angle_may_differ) is exempt, and no box of these sets is); NMS keep lists identical.
"""
import numpy as np
import pytest
import torch

import rbox_sets
from conftest import bits
from s2anet_b200 import synth

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def gpu_iou(b1, b2, flags=0):
    from s2anet_b200.box_iou_rotated import box_iou_rotated
    return box_iou_rotated(torch.from_numpy(np.ascontiguousarray(b1)).to(DEV),
                           torch.from_numpy(np.ascontiguousarray(b2)).to(DEV), _flags=flags).cpu().numpy()


def assert_iou_parity(mine, ref, b1, b2):
    """Bit-exact.  The one allowed exception is a pair with a box whose float64 sin/cos lies so close to an fp32
    rounding midpoint that CUDA's and glibc's (2 and 1 ulp accurate) may round it apart; such pairs must still be
    within 1e-5.  None of the synthetic sets has such a box, so it is asserted that none is flagged."""
    f1, f2 = rbox_sets.angle_may_differ(b1[:, 4]), rbox_sets.angle_may_differ(b2[:, 4])
    assert not f1.any() and not f2.any(), "a synthetic box's sin/cos sits on an fp32 rounding midpoint"
    diff = bits(mine) != bits(ref)
    assert not diff.any(), "%d pairs differ from the oracle, first %s" % (diff.sum(), np.argwhere(diff)[:5].tolist())


def test_iou_cfg1_golden_and_oracle(oracle, golden):
    g = golden("cfg1_iou_nms.npz")
    b = g["boxes"]
    mine = gpu_iou(b, b)
    assert_iou_parity(mine[:200], g["iou_rows_0_200_ref_hdr_cuda"], b[:200], b)
    assert_iou_parity(mine, oracle.box_iou_rotated(b, b), b, b)
    assert np.abs(mine[:200] - g["iou_rows_0_200_ref_ext_cpu"]).max() <= 1e-5     # reference CPU extension
    # the disjointness shortcut must not change a single bit
    np.testing.assert_array_equal(bits(mine), bits(gpu_iou(b, b, flags=1)))


def test_iou_adversarial_and_ragged(oracle, golden):
    g = golden("adversarial_iou.npz")
    mine = gpu_iou(g["boxes"], g["boxes"])
    ref = g["iou_ref_hdr_cuda"]
    ok = np.isfinite(ref)
    assert np.array_equal(np.isnan(mine), np.isnan(ref))
    assert np.abs(mine[ok] - ref[ok]).max() <= 1e-5
    # ragged tiles: sizes around the 64-wide tile edge, n != m
    rng = np.random.default_rng(5)
    for n, m in ((1, 1), (63, 65), (64, 64), (65, 1), (130, 257), (7, 500)):
        b1 = synth.clustered_boxes(n_seed=max(1, n), rep=1, seed=n)[0][:n]
        b2 = synth.clustered_boxes(n_seed=max(1, m // 2 + 1), rep=2, seed=m)[0][:m]
        assert_iou_parity(gpu_iou(b1, b2), oracle.box_iou_rotated(b1, b2), b1, b2)
    assert gpu_iou(np.zeros((0, 5), np.float32), b2).shape == (0, len(b2))
    assert gpu_iou(b2, np.zeros((0, 5), np.float32)).shape == (len(b2), 0)


def test_iou_noncontiguous_input(oracle):
    from s2anet_b200.box_iou_rotated import bbox_iou_rotated
    b, s, _ = synth.clustered_boxes(n_seed=30, rep=3, seed=2)
    d6 = torch.from_numpy(np.concatenate([b, s[:, None]], 1)).to(DEV)
    out = bbox_iou_rotated(d6, d6[:, :5]).cpu().numpy()               # 6-column + strided view
    assert_iou_parity(out, oracle.box_iou_rotated(b, b), b, b)


def test_iou_anchor_gt_golden_and_batched(oracle, golden):
    from s2anet_b200.box_iou_rotated import box_iou_rotated_batched
    g = golden("cfg4_anchor_gt_iou.npz")
    assert_iou_parity(gpu_iou(g["anchors"], g["gts"]), g["iou_ref_hdr_cuda"], g["anchors"], g["gts"])
    # batched + row-sharded form equals per-image calls
    B = 3
    an = synth.all_level_anchors(B, 3)[:, ::8]
    gt = np.stack([synth.dota_like_gt(100, 10 + i) for i in range(B)])
    ta, tg = torch.from_numpy(an).to(DEV), torch.from_numpy(gt).to(DEV)
    full = box_iou_rotated_batched(ta, tg)
    for i in range(B):
        np.testing.assert_array_equal(bits(full[i].cpu().numpy()), bits(gpu_iou(an[i], gt[i])))
    n = an.shape[1]
    out = torch.full_like(full, -7.0)
    mid = (n // 2) // 64 * 64
    box_iou_rotated_batched(ta, tg, 0, mid, out=out)
    box_iou_rotated_batched(ta, tg, mid, n, out=out)
    assert torch.equal(out, full)


def test_iou_full_size_properties():
    """BASELINE config 4 at full size for one GPU-friendly slice: 21,824 anchors x 500 GT x 8 images.
    The oracle cannot finish this in seconds, so use size-independent properties: shortcut on/off
    bit-equality, diagonal of a self-IoU == 1 within 1e-5, symmetry within 1e-5, range."""
    from s2anet_b200.box_iou_rotated import box_iou_rotated_batched
    B = 8
    an = torch.from_numpy(synth.all_level_anchors(B, 3)).to(DEV)
    gt = torch.from_numpy(np.stack([synth.dota_like_gt(500, 100 + i) for i in range(B)])).to(DEV)
    a = box_iou_rotated_batched(an, gt)
    b = box_iou_rotated_batched(an, gt, _flags=1)
    assert torch.equal(a, b)
    assert float(a.min()) >= 0.0 and float(a.max()) <= 1.0 + 1e-5
    t = box_iou_rotated_batched(gt, an)
    assert float((a - t.transpose(1, 2)).abs().max()) <= 1e-5
    s = box_iou_rotated_batched(gt, gt)
    d = torch.diagonal(s, dim1=1, dim2=2)
    assert float((d - 1).abs().max()) <= 1e-5


@pytest.mark.parametrize("world,tile_rows", [(1, 256), (2, 256), (8, 64), (3, 64), (5, 32), (2, 128)])
def test_iou_row_tiles_dealt_cyclically(world, tile_rows):
    """The multi-GPU form (s2a_box_iou_rotated_tiles): the union of the ranks' cyclically dealt row tiles, packed or
    written in place, is bit-identical to the one-call matrix; slivers, a partial last tile and partial column tiles
    included."""
    from s2anet_b200.box_iou_rotated import box_iou_rotated_batched, box_iou_rotated_tiles, tile_rows_of
    B = 2
    an = synth.all_level_anchors(B, 5)[:, ::4][:, :5021].copy()           # 5,021 rows: a partial last tile
    gt = np.stack([synth.dota_like_gt(300, 40 + i) for i in range(B)])
    gt[:, ::9, 3] = 0.7                                                   # sub-pixel slivers
    ta, tg = torch.from_numpy(an).to(DEV), torch.from_numpy(gt).to(DEV)
    full = box_iou_rotated_batched(ta, tg)
    assert torch.equal(full, box_iou_rotated_batched(ta, tg, _flags=1))   # reject tests on / off
    inplace = torch.full_like(full, -3.0)
    for r in range(world):
        rows = tile_rows_of(an.shape[1], r, world, tile_rows).to(DEV)
        packed = box_iou_rotated_tiles(ta, tg, r, world, compact=True, tile_rows=tile_rows)
        assert packed.size(1) % tile_rows == 0 and packed.size(1) >= rows.numel()
        assert torch.equal(packed[:, : rows.numel()], full[:, rows])
        box_iou_rotated_tiles(ta, tg, r, world, compact=False, out=inplace, tile_rows=tile_rows)
    assert torch.equal(inplace, full)


def test_iou_degenerate_pairs_take_the_general_clipper(oracle):
    """Pairs the register-resident hull refuses (more than eight candidate points, coincident candidates, collinear
    triples: identical boxes, shared edges and corners, axis-aligned grid anchors against themselves) fall back to
    the general 24-point routine inside the same kernel: still bit-identical to the oracle."""
    ga = np.concatenate([synth.grid_anchors(16, 16, 8).reshape(-1, 5), synth.grid_anchors(8, 8, 16).reshape(-1, 5)])
    assert_iou_parity(gpu_iou(ga, ga), oracle.box_iou_rotated(ga, ga), ga, ga)
    adv = synth.adversarial_boxes()
    assert_iou_parity(gpu_iou(adv, ga[::3]), oracle.box_iou_rotated(adv, ga[::3]), adv, ga[::3])
    rot = ga.copy()
    rot[:, 4] = np.float32(np.pi / 4)
    assert_iou_parity(gpu_iou(rot, ga), oracle.box_iou_rotated(rot, ga), rot, ga)


def gpu_nms(b, s, thr, labels=None):
    from s2anet_b200.nms_rotated import ml_nms_rotated, nms_rotated_op
    tb, ts = torch.from_numpy(b).to(DEV), torch.from_numpy(s).to(DEV)
    if labels is None:
        return nms_rotated_op(tb, ts, thr).cpu().numpy()
    return ml_nms_rotated(tb, ts, torch.from_numpy(labels).to(DEV), thr).cpu().numpy()


def test_nms_keep_lists_golden(oracle, golden):
    g = golden("cfg1_iou_nms.npz")
    b, s, l = g["boxes"], g["scores"], g["labels"]
    np.testing.assert_array_equal(gpu_nms(b, s, 0.5), g["keep_nms_thr05_cuda_semantics"])
    np.testing.assert_array_equal(gpu_nms(b, s, 0.5, l), g["keep_mlnms_thr05_cuda_semantics"])


_NMS_CASES = [(1, 1, 0.5), (13, 5, 0.1), (50, 2, 0.7), (300, 7, 0.3), (1000, 3, 0.5)]


@pytest.mark.parametrize("n_seed,rep,thr,quantise", [pytest.param(*c, None, id="%d-%d-%g" % c) for c in _NMS_CASES] +
                         [pytest.param(*c, q, id="%d-%d-%g-%s" % (c + (q,)))
                          for c in [(300, 7, 0.3), (1000, 3, 0.5)] for q in ("bf16", "f16")])
def test_nms_vs_oracle(oracle, n_seed, rep, thr, quantise):
    """quantise: scores rounded through a 16-bit type, so that many are equal; equal scores keep their input order
    (the generic path's stable sort), like the oracle's."""
    b, s, l = synth.clustered_boxes(n_seed=n_seed, rep=rep, seed=n_seed)
    if quantise:
        s = torch.from_numpy(s).to(torch.bfloat16 if quantise == "bf16" else torch.float16).float().numpy()
        assert len(np.unique(s)) < 0.9 * len(s)
    np.testing.assert_array_equal(gpu_nms(b, s, thr), oracle.nms_rotated(b, s, thr))
    np.testing.assert_array_equal(gpu_nms(b, s, thr, l), oracle.nms_rotated(b, s, thr, labels=l))


def test_nms_wrapper_and_edge_cases(oracle):
    from s2anet_b200.nms_rotated import nms_rotated
    b, s, _ = synth.clustered_boxes(n_seed=40, rep=4, seed=8)
    dets = torch.from_numpy(np.concatenate([b, s[:, None]], 1)).to(DEV)
    kept, keep = nms_rotated(dets, 0.4)                               # strided dets[:, :5] / dets[:, 5] views
    ref = oracle.nms_rotated(b, s, 0.4)
    np.testing.assert_array_equal(keep.cpu().numpy(), ref)
    assert torch.equal(kept, dets[keep])
    assert keep.dtype == torch.int64 and keep.device == dets.device
    empty = torch.zeros((0, 6), device=DEV)
    assert nms_rotated(empty, 0.5) is empty
    # identical boxes: only the best survives; negative threshold: only the best survives too
    same = np.repeat(b[:1], 70, 0)
    sc = np.linspace(0.1, 0.9, 70).astype(np.float32)
    np.testing.assert_array_equal(gpu_nms(same, sc, 0.5), [69])
    np.testing.assert_array_equal(gpu_nms(b, s, -1.0), oracle.nms_rotated(b, s, -1.0))
    # threshold 1.0 keeps everything that is not > 1
    np.testing.assert_array_equal(gpu_nms(b, s, 1.5), np.argsort(-s, kind="stable"))


def test_nms_large_idempotent():
    """N = 20,000 (the stress size of SURVEY 8d): descending scores, no kept pair above the
    threshold, idempotence."""
    from s2anet_b200.box_iou_rotated import box_iou_rotated
    from s2anet_b200.nms_rotated import nms_rotated_op
    b, s, _ = synth.clustered_boxes(n_seed=4000, rep=5, seed=21)
    tb, ts = torch.from_numpy(b).to(DEV), torch.from_numpy(s).to(DEV)
    keep = nms_rotated_op(tb, ts, 0.5)
    assert 3000 < keep.numel() < 20000
    assert bool((ts[keep][1:] <= ts[keep][:-1]).all())
    kb = tb[keep]
    again = nms_rotated_op(kb, ts[keep], 0.5)
    assert torch.equal(again, torch.arange(keep.numel(), device=DEV))
    iou = box_iou_rotated(kb[:4096], kb[:4096])
    assert int((torch.triu(iou, 1) > 0.5).sum()) == 0


def test_multiclass_vs_oracle(oracle):
    from s2anet_b200.nms_rotated import multiclass_nms_rotated, multiclass_nms_rotated_batched
    rng = np.random.default_rng(4)
    imgs = []
    for i, (n_seed, rep) in enumerate([(300, 4), (50, 3), (700, 5)]):
        b, _, _ = synth.clustered_boxes(n_seed=n_seed, rep=rep, seed=30 + i)
        sc = rng.uniform(0, 1, (b.shape[0], 15)).astype(np.float32) ** 6      # ~15 % above 0.05
        sc += (np.arange(sc.size, dtype=np.float64).reshape(sc.shape) * 1e-9).astype(np.float32)
        imgs.append((b, sc))
    for b, sc in imgs:
        dets, labels = multiclass_nms_rotated(torch.from_numpy(b).to(DEV), torch.from_numpy(sc).to(DEV), 0.05, 0.5, 2000)
        rd, rl = oracle.multiclass_nms_rotated(b, sc, 0.05, 0.5, 2000)
        np.testing.assert_array_equal(dets.cpu().numpy(), rd)
        np.testing.assert_array_equal(labels.cpu().numpy(), rl)
        assert labels.dtype == torch.float32
        d50, l50 = multiclass_nms_rotated(torch.from_numpy(b).to(DEV), torch.from_numpy(sc).to(DEV), 0.05, 0.5, 50)
        np.testing.assert_array_equal(d50.cpu().numpy(), rd[:50])
    # empty result: reference returns ([0,6], [0,1] long)
    b, sc = imgs[1]
    d, l = multiclass_nms_rotated(torch.from_numpy(b).to(DEV), torch.from_numpy(sc * 0).to(DEV))
    assert tuple(d.shape) == (0, 6) and tuple(l.shape) == (0, 1) and l.dtype == torch.int64
    # batched: pad the three images to a common n and compare per image
    n = max(b.shape[0] for b, _ in imgs)
    bb = np.zeros((3, n, 5), np.float32)
    ss = np.zeros((3, n, 15), np.float32)
    for i, (b, sc) in enumerate(imgs):
        bb[i, :len(b)], ss[i, :len(b)] = b, sc
    dets, labels, counts = multiclass_nms_rotated_batched(torch.from_numpy(bb).to(DEV), torch.from_numpy(ss).to(DEV),
                                                          0.05, 0.5, 2000)
    for i, (b, sc) in enumerate(imgs):
        rd, rl = oracle.multiclass_nms_rotated(b, sc, 0.05, 0.5, 2000)
        k = int(counts[i])
        assert k == len(rd)
        np.testing.assert_array_equal(dets[i, :k].cpu().numpy(), rd)
        np.testing.assert_array_equal(labels[i, :k].cpu().numpy(), rl)


def test_multiclass_full_size_head_shape():
    """5,344 boxes x 15 classes (the per-image maximum after the per-level top-2000): the fused
    class-segmented path equals the generic score-ordered ml_nms kernel composed like the reference."""
    from s2anet_b200.nms_rotated import _multiclass_composed, multiclass_nms_rotated
    rng = np.random.default_rng(6)
    b, _, _ = synth.clustered_boxes(n_seed=1336, rep=4, seed=44)
    sc = (rng.uniform(0, 1, (b.shape[0], 15)) ** 8).astype(np.float32)
    sc += (np.arange(sc.size, dtype=np.float64).reshape(sc.shape) * 1e-9).astype(np.float32)
    tb, ts = torch.from_numpy(b).to(DEV), torch.from_numpy(sc).to(DEV)
    d1, l1 = multiclass_nms_rotated(tb, ts, 0.05, 0.5, 2000)
    d2, l2 = _multiclass_composed(tb, ts, 0.05, 0.5, 2000)
    assert d1.shape[0] == 2000
    assert torch.equal(d1, d2) and torch.equal(l1, l2)


def _ref_gpu(name):
    from oracle import build_oracle
    mod = build_oracle.load_ref_extension(name, "gpu")
    if mod is None:
        pytest.skip("oracle/_ref/ext_gpu/%s not prebuilt" % name)
    return mod


def test_multiclass_packed_form_equals_plain_outputs():
    """The detection exchange's pack fused into the NMS finaliser (s2a_multiclass_nms_rotated_packed): rows
    (x, y, w, h, theta, score, label, 0) + the count row, into one or several destination buffers at a slot offset,
    are exactly the plain outputs."""
    from s2anet_b200.dist import packed_views
    from s2anet_b200.nms_rotated import multiclass_nms_rotated_batched, multiclass_nms_rotated_packed
    B, K = 3, 300
    rng = np.random.default_rng(5)
    bx = np.stack([synth.clustered_boxes(n_seed=150, rep=4, seed=20 + i)[0] for i in range(B)])
    sc = (rng.uniform(0, 1, (B, bx.shape[1], 15)) ** 5).astype(np.float32)
    sc[2] = 0.0                                                            # an image without detections
    tb, ts = torch.from_numpy(bx).to(DEV), torch.from_numpy(sc).to(DEV)
    d, l, c = multiclass_nms_rotated_batched(tb, ts, 0.05, 0.5, K)
    dst0 = torch.full((5, K + 1, 8), -1.0, device=DEV)
    dst1 = torch.full((5, K + 1, 8), -1.0, device=DEV)
    multiclass_nms_rotated_packed(tb, ts, [dst0, dst1.data_ptr()], slot0=2, score_thr=0.05, iou_thr=0.5, max_per_img=K)
    assert torch.equal(dst0, dst1)
    assert bool((dst0[:2] == -1.0).all())                                  # other ranks' slots untouched
    pd, pl, pc = packed_views(dst0[2:], K)
    assert pc.tolist() == c.tolist() and c[2] == 0 and int(c.max()) == K
    for i in range(B):
        k = int(c[i])
        assert torch.equal(pd[i, :k], d[i, :k]) and torch.equal(pl[i, :k], l[i, :k])
    assert bool((dst0[2:, K, 1:] == 0).all())


def test_against_reference_cuda_kernels_on_this_gpu(oracle):
    """The reference's own CUDA extensions (unmodified sources, compiled for sm_100a in the
    authoring container) run beside ours: IoU within 1e-5; keep lists identical except for pairs
    whose IoU lies within 1e-6 of the threshold (listed).

    Known, documented exception (DESIGN.md section 3): nvcc contracts the reference's parallel-edge
    determinant into an FMA, so for a box paired with an IDENTICAL box its binary returns ~1/3
    instead of 1.0.  Every pair that differs by more than 1e-5 must be such a duplicate pair, and for
    those this library must hold the float64-correct value (1.0)."""
    iou_ref = _ref_gpu("box_iou_rotated_cuda")
    nms_ref = _ref_gpu("nms_rotated_cuda")
    ml_ref = _ref_gpu("ml_nms_rotated_cuda")
    from s2anet_b200.box_iou_rotated import box_iou_rotated
    from s2anet_b200.nms_rotated import ml_nms_rotated, nms_rotated_op
    b, s, l = synth.clustered_boxes(seed=0)
    tb, ts, tl = (torch.from_numpy(x).to(DEV) for x in (b, s, l))
    mine, ref = box_iou_rotated(tb, tb), iou_ref.box_iou_rotated(tb, tb)
    bad = ((mine - ref).abs() > 1e-5).nonzero().cpu().numpy()
    print("pairs differing from the reference CUDA binary by > 1e-5:", bad.tolist())
    for i, j in bad:
        assert np.array_equal(b[i], b[j]), "non-duplicate pair (%d, %d) differs from the reference kernel" % (i, j)
        assert abs(float(mine[i, j]) - 1.0) <= 1e-5
    assert len(bad) <= 20
    for thr in (0.3, 0.5):
        near = ((ref - thr).abs() < 1e-6).nonzero().cpu().numpy()
        k1, k2 = nms_rotated_op(tb, ts, thr), nms_ref.nms_rotated(tb, ts, thr)
        m1, m2 = ml_nms_rotated(tb, ts, tl, thr), ml_ref.ml_nms_rotated(tb, ts, tl, thr)
        if len(near) == 0:
            assert torch.equal(k1, k2) and torch.equal(m1, m2)
        else:       # only pairs listed here may explain a difference
            print("pairs within 1e-6 of thr=%g:" % thr, near.tolist())
            touched = set(near.reshape(-1).tolist())
            assert set(k1.tolist()) ^ set(k2.tolist()) <= touched
            assert set(m1.tolist()) ^ set(m2.tolist()) <= touched
    an = torch.from_numpy(synth.all_level_anchors(1, 3)[0]).to(DEV)
    gt = torch.from_numpy(synth.dota_like_gt(500, 3)).to(DEV)
    assert float((box_iou_rotated(an, gt) - iou_ref.box_iou_rotated(an, gt)).abs().max()) <= 1e-5


def test_duplicate_boxes_are_the_only_keep_list_difference_to_the_reference_binary():
    """VERDICT r1 weak 1b: the one documented divergence from the reference's CUDA *binary*, listed at NMS level.

    For a box paired with an exact copy of itself the reference binary (nvcc default FMA contraction) returns IoU ~ 1/3
    instead of 1 (DESIGN.md section 3), so at thr = 0.5 it KEEPS the lower-scored copy; this library (and the
    reference's CPU build, and float64 arithmetic) suppresses it.  On a set with planted exact duplicates the two keep
    lists may differ ONLY by such copies: every index the reference keeps and we do not is an exact duplicate of a
    higher-scored box that both lists keep, and we keep nothing the reference drops."""
    nms_ref = _ref_gpu("nms_rotated_cuda")
    iou_ref = _ref_gpu("box_iou_rotated_cuda")
    from s2anet_b200.box_iou_rotated import box_iou_rotated
    from s2anet_b200.nms_rotated import nms_rotated_op
    b, s, _ = synth.clustered_boxes(n_seed=300, rep=4, seed=7)
    n0 = b.shape[0]
    dup_src = np.arange(0, n0, 5)[:120]                       # 120 planted exact copies, with lower scores
    b = np.concatenate([b, b[dup_src]])
    s = np.concatenate([s, s[dup_src] * 0.5 + np.arange(len(dup_src), dtype=np.float32) * 1e-6])
    tb, ts = torch.from_numpy(b).to(DEV), torch.from_numpy(s).to(DEV)
    thr = 0.5
    mine, ref = nms_rotated_op(tb, ts, thr), nms_ref.nms_rotated(tb, ts, thr)
    mine_set, ref_set = set(mine.tolist()), set(ref.tolist())
    assert mine_set <= ref_set, "this library keeps a box the reference binary suppresses: %s" % sorted(mine_set - ref_set)
    only_ref = sorted(ref_set - mine_set)
    listed = []
    for i in only_ref:
        assert i >= n0, "box %d (not a planted copy) is kept by the reference binary only" % i
        j = int(dup_src[i - n0])
        assert np.array_equal(b[i], b[j]) and s[j] > s[i]
        # the reference binary's IoU of the pair is the contraction artefact, ours is 1
        iou_r = float(iou_ref.box_iou_rotated(tb[i:i + 1], tb[j:j + 1]))
        iou_m = float(box_iou_rotated(tb[i:i + 1], tb[j:j + 1]))
        assert abs(iou_m - 1.0) <= 1e-5 and iou_r < thr
        listed.append((i, j, round(iou_r, 4)))
    print("duplicate pairs kept by the reference CUDA binary only (copy, original, its IoU):", listed)
    # and the common part is in the same (descending score) order
    common = [i for i in ref.tolist() if i in mine_set]
    assert common == mine.tolist()


def test_multiclass_batched_takes_more_than_6144_boxes(oracle):
    """ADVICE r1 (medium): the fused kernel stops at 6,144 candidate boxes per image (5 levels x top-2000 on inputs
    above ~1,100 px exceed it); the batched entry then composes the generic ml_nms_rotated kernel per image instead of
    raising, with the same fixed-shape outputs."""
    from s2anet_b200.nms_rotated import MC_FUSED_MAX_BOXES, multiclass_nms_rotated, multiclass_nms_rotated_batched
    n = MC_FUSED_MAX_BOXES + 200
    b, _, _ = synth.clustered_boxes(n_seed=n // 4 + 1, rep=4, seed=31)
    b = b[:n]
    rng = np.random.default_rng(8)
    sc = (rng.uniform(0, 1, (n, 3)) ** 6).astype(np.float32)
    tb, ts = torch.from_numpy(b).to(DEV), torch.from_numpy(sc).to(DEV)
    d, l, c = multiclass_nms_rotated_batched(torch.stack([tb, tb]), torch.stack([ts, ts * 0.0]), 0.05, 0.5, 500)
    rd, rl = oracle.multiclass_nms_rotated(b, sc, 0.05, 0.5, 500)
    k = int(c[0])
    assert k == rd.shape[0] and int(c[1]) == 0
    np.testing.assert_array_equal(d[0, :k].cpu().numpy(), rd)
    np.testing.assert_array_equal(l[0, :k].cpu().numpy(), rl)
    d1, l1 = multiclass_nms_rotated(tb, ts, 0.05, 0.5, 500)                # the single-image wrapper takes the same route
    np.testing.assert_array_equal(d1.cpu().numpy(), rd)


def test_torch_extension_binding_matches_the_ctypes_path_bit_for_bit(oracle):
    """csrc/torch_binding.cpp (pybind11, at::Tensor in / out) and the ctypes wrappers call the same C-ABI entries: same
    bits for the IoU matrix, same keep lists for nms / ml_nms (strided dets[:, :5] views and fp16 scores included), same
    ARF scatter; and the reference's error type for bad arguments."""
    import os
    from s2anet_b200 import _torch_ext, box_iou_rotated as biou, nms_rotated as nmsr, orn
    ext = _torch_ext.module()
    assert ext is not None, "s2anet_b200/_s2a_torch.so is not built"
    b, s, l = synth.clustered_boxes(n_seed=120, rep=5, seed=4)
    tb, ts, tl = torch.from_numpy(b).to(DEV), torch.from_numpy(s).to(DEV), torch.from_numpy(l).to(DEV)
    iou_ext = ext.box_iou_rotated(tb, tb[:77])
    os.environ["S2A_NO_TORCH_EXT"] = "1"
    saved = (_torch_ext._MOD, _torch_ext._TRIED)
    _torch_ext._MOD, _torch_ext._TRIED = None, False
    try:
        assert _torch_ext.module() is None
        iou_ct = biou.box_iou_rotated(tb, tb[:77])
        keep_ct = nmsr.nms_rotated_op(tb, ts, 0.5)
        ml_ct = nmsr.ml_nms_rotated(tb, ts, tl, 0.5)
        dets6 = torch.cat([tb, ts[:, None]], dim=1)
        strided_ct = nmsr.nms_rotated_op(dets6[:, :5], dets6[:, 5].half(), 0.3)
    finally:
        del os.environ["S2A_NO_TORCH_EXT"]
        _torch_ext._MOD, _torch_ext._TRIED = saved
    assert torch.equal(iou_ext, iou_ct)
    np.testing.assert_array_equal(iou_ext.cpu().numpy(), oracle.box_iou_rotated(b, b[:77]))
    assert torch.equal(ext.nms_rotated(tb, ts, 0.5), keep_ct)
    assert torch.equal(ext.ml_nms_rotated(tb, ts, tl, 0.5), ml_ct)
    assert torch.equal(ext.nms_rotated(dets6[:, :5], dets6[:, 5].half(), 0.3), strided_ct)
    assert ext.nms_rotated(tb[:0], ts[:0], 0.5).shape == (0,) and ext.box_iou_rotated(tb[:0], tb).shape == (0, b.shape[0])
    idx = torch.from_numpy(oracle.arf_indices(1, 8, 3)).to(DEV)
    w = torch.randn(4, 6, 1, 3, 3, device=DEV)
    rot = ext.arf_forward(w, idx)
    assert torch.equal(rot, torch.from_numpy(oracle.arf_forward(w.cpu().numpy(), oracle.arf_indices(1, 8, 3))).to(DEV))
    g = torch.randn_like(rot)
    assert torch.allclose(ext.arf_backward(idx, g), orn.arf_backward(idx, g))
    with pytest.raises(RuntimeError):
        ext.box_iou_rotated(tb[:, :4], tb)
    with pytest.raises(RuntimeError):
        ext.nms_rotated(tb, ts[:5], 0.5)
