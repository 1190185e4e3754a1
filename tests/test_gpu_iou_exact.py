"""Rotated IoU, rotated NMS and label assignment against the CPU oracle, exactly, where these kernels go wrong.

* NMS: boxes that share both long edge lines (same angle and height, one nested in the other along its axis).  The
  reference's fp32 clipper returns IoUs up to 1.0 for a true 0.49, so a kernel that skips the clip because the pair
  "cannot" reach the threshold drops suppressions the reference makes.  Also pairs whose IoU is exactly the threshold
  (the rule is IoU > thr).
* IoU: bit for bit against the oracle at the bench shape (21,824 refined anchors x 500 GTs) and on degenerate sets,
  through every kernel form (batched, row tiles, every tile height, one and two columns per thread, reject tests
  off).  The only pairs allowed to differ are those of a box whose fp32 sin/cos may round differently on the device
  (`rbox_sets.angle_may_differ`), and the synthetic sets here have none.
* assign_labels: on the oracle's own IoU matrix, with axis-aligned grid anchors where tied maxima and IoUs exactly at
  0.5, 0.4 and min_pos_iou_thr are normal, column tiles cut through the ties, a non-square image filter with anchors on
  its edges, IoUs above 1 and NaN.
"""
from multiprocessing.pool import ThreadPool

import numpy as np
import pytest
import torch

import rbox_sets
from conftest import bits
from s2anet_b200 import synth

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
F32 = np.float32


def T(x):
    return torch.from_numpy(np.ascontiguousarray(x)).to(DEV)


def assert_iou_exact(mine, ref, b1, b2):
    """Bit for bit; pairs of a box flagged by angle_may_differ are allowed 1e-5, and synthetic sets have none."""
    f1, f2 = rbox_sets.angle_may_differ(b1[:, 4]), rbox_sets.angle_may_differ(b2[:, 4])
    assert not f1.any() and not f2.any(), "a synthetic box's sin/cos sits on an fp32 rounding midpoint"
    same = (bits(mine) == bits(ref)) | (np.isnan(mine) & np.isnan(ref))
    assert same.all(), "%d of %d pairs differ from the oracle, first %s" % ((~same).sum(), same.size,
                                                                            np.argwhere(~same)[:5].tolist())


def oracle_images(pairs):
    with ThreadPool(min(len(pairs), 8)) as pool:
        return pool.map(rbox_sets.oracle_iou_image, pairs)


# ---------------------------------------------------------------------------------------------------------------------
# rotated NMS
# ---------------------------------------------------------------------------------------------------------------------
def planted_set(seed, quantise, n_pairs=1000):
    """A clustered background with n_pairs nested shared-edge pairs: boxes, scores, labels (each pair shares one),
    and the planted pair rows."""
    bg, _, bl = synth.clustered_boxes(n_seed=300, rep=4, seed=seed)
    o, i = rbox_sets.nested_pairs(n_pairs, seed + 1, shift=False)
    b = np.concatenate([bg, rbox_sets.interleave(o, i)])
    rng = np.random.default_rng(seed + 2)
    l = np.concatenate([bl, np.repeat(rng.integers(0, 15, n_pairs), 2).astype(F32)])
    perm = rng.permutation(len(b))
    b, l = b[perm], l[perm]
    s = rng.uniform(0, 1, len(b)).astype(F32)
    if quantise:
        s = torch.from_numpy(s).to(torch.bfloat16).float().numpy()
        assert len(np.unique(s)) < 0.5 * len(s)
    inv = np.argsort(perm)
    pairs = inv[len(bg):].reshape(-1, 2)
    return b, s, l, pairs


def planted_above(b, pairs, thr, oracle):
    v = np.array([oracle.single_iou(b[p], b[q]) for p, q in pairs])
    return int((v > thr).sum())


_NMS_PARAMS = [pytest.param(thr, q, id="%g-%s" % (thr, q or "f32")) for thr in (0.3, 0.5, 0.7) for q in (None, "bf16")]


@pytest.mark.parametrize("thr,quantise", _NMS_PARAMS)
def test_nms_planted_shared_edges(oracle, thr, quantise):
    from s2anet_b200.nms_rotated import ml_nms_rotated, nms_rotated_op
    b, s, l, pairs = planted_set(70, quantise)
    # the set is sharp: the reference suppresses planted pairs whose true IoU (< 0.49) is far below thr
    assert planted_above(b, pairs, thr, oracle) >= 10
    np.testing.assert_array_equal(nms_rotated_op(T(b), T(s), thr).cpu().numpy(), oracle.nms_rotated(b, s, thr))
    np.testing.assert_array_equal(ml_nms_rotated(T(b), T(s), T(l), thr).cpu().numpy(),
                                  oracle.nms_rotated(b, s, thr, labels=l))


def planted_scores(b, l, quantise, seed):
    """[n, 15] class scores: each box scores above 0.05 in its own label only (so a planted pair meets in one class)."""
    rng = np.random.default_rng(seed)
    sc = (rng.uniform(0, 1, (len(b), 15)) ** 8 * 0.05).astype(F32)
    sc[np.arange(len(b)), l.astype(int)] = rng.uniform(0.06, 1, len(b))
    if quantise:
        sc = torch.from_numpy(sc).to(torch.bfloat16).float().numpy()
    return sc


@pytest.mark.parametrize("thr,quantise", _NMS_PARAMS)
def test_multiclass_planted_shared_edges(oracle, thr, quantise):
    from s2anet_b200.dist import packed_views
    from s2anet_b200.nms_rotated import (multiclass_nms_rotated, multiclass_nms_rotated_batched,
                                         multiclass_nms_rotated_packed)
    K = 4000
    b, _, l, pairs = planted_set(80, quantise)
    sc = planted_scores(b, l, quantise, 81)
    assert planted_above(b, pairs, thr, oracle) >= 10
    rd, rl = oracle.multiclass_nms_rotated(b, sc, 0.05, thr, K)
    d, lab = multiclass_nms_rotated(T(b), T(sc), 0.05, thr, K)
    np.testing.assert_array_equal(d.cpu().numpy(), rd)
    np.testing.assert_array_equal(lab.cpu().numpy(), rl)
    # batched: image 0 is a plain clustered image, image 1 the planted one
    b0, _, l0 = synth.clustered_boxes(n_seed=400, rep=5, seed=82)
    s0 = planted_scores(b0, l0, quantise, 83)
    n = max(len(b0), len(b))
    bb, ss = np.zeros((2, n, 5), F32), np.zeros((2, n, 15), F32)
    bb[0, :len(b0)], ss[0, :len(b0)], bb[1, :len(b)], ss[1, :len(b)] = b0, s0, b, sc
    want = [oracle.multiclass_nms_rotated(b0, s0, 0.05, thr, K), (rd, rl)]
    d, lab, c = multiclass_nms_rotated_batched(T(bb), T(ss), 0.05, thr, K)
    dst = torch.full((2, K + 1, 8), -1.0, device=DEV)
    multiclass_nms_rotated_packed(T(bb), T(ss), [dst], slot0=0, score_thr=0.05, iou_thr=thr, max_per_img=K)
    pd, pl, pc = packed_views(dst, K)
    for i, (wd, wl) in enumerate(want):
        k = int(c[i])
        assert k == len(wd) and int(pc[i]) == k
        np.testing.assert_array_equal(d[i, :k].cpu().numpy(), wd)
        np.testing.assert_array_equal(lab[i, :k].cpu().numpy(), wl)
        np.testing.assert_array_equal(pd[i, :k].cpu().numpy(), wd)
        np.testing.assert_array_equal(pl[i, :k].cpu().numpy(), wl)


def test_nms_threshold_equal_pairs(oracle):
    """Axis-aligned dyadic pairs whose IoU is exactly 0.5f, 0.25f and fl(1/3): at thr == IoU the later box is kept
    (the rule is IoU > thr), one float below it is suppressed -- in every NMS entry."""
    from s2anet_b200.nms_rotated import ml_nms_rotated, multiclass_nms_rotated, nms_rotated_op
    cases = [((64, 64, 4, 4, 0), (64, 64, 4, 2, 0), 0.5),          # nested, half the area
             ((64, 64, 4, 4, 0), (64, 64, 2, 2, 0), 0.25),         # nested, a quarter
             ((64, 64, 2, 2, 0), (65, 64, 2, 2, 0), 1.0 / 3.0),    # half-shifted squares: 2 / 6
             ((96.5, 32.25, 8, 16, 0), (98.5, 32.25, 8, 16, 0), 0.6)]  # 6 x 16 / (256 - 96)
    for a, c, v in cases:
        b = np.array([a, c], F32)
        iou = oracle.box_iou_rotated(b, b)[0, 1]
        assert iou == F32(v), (a, c, iou)
        s = np.array([0.9, 0.8], F32)
        lab = np.zeros(2, F32)
        sc = np.zeros((2, 3), F32)
        sc[:, 1] = s
        for thr, keep in ((iou, [0, 1]), (np.nextafter(iou, F32(-np.inf)), [0])):
            thr = float(thr)
            np.testing.assert_array_equal(oracle.nms_rotated(b, s, thr), keep)
            np.testing.assert_array_equal(nms_rotated_op(T(b), T(s), thr).cpu().numpy(), keep)
            np.testing.assert_array_equal(ml_nms_rotated(T(b), T(s), T(lab), thr).cpu().numpy(), keep)
            d, _ = multiclass_nms_rotated(T(b), T(sc), 0.05, thr, 100)
            np.testing.assert_array_equal(d[:, 5].cpu().numpy(), s[keep])


# ---------------------------------------------------------------------------------------------------------------------
# rotated IoU kernel
# ---------------------------------------------------------------------------------------------------------------------
def test_iou_bench_shape_exact():
    """BASELINE config 4 as bench.py builds it (64 images of all-level refined anchors x 500 GTs): images 0, 1 and 63
    in full, through the batched call, the packed row tiles of world 1 and of every rank of world 8, and with the
    reject tests off."""
    from s2anet_b200 import dist
    from s2anet_b200.box_iou_rotated import box_iou_rotated_batched, box_iou_rotated_tiles, tile_rows_of
    B, imgs = 64, [0, 1, 63]
    an = synth.all_level_anchors(B, 3)
    gt = np.stack([synth.dota_like_gt(500, 100 + i) for i in range(B)])
    ta, tg = T(an), T(gt)
    ref = oracle_images([(an[i], gt[i]) for i in imgs])
    sel = torch.tensor(imgs, device=DEV)
    forms = {"batched": box_iou_rotated_batched(ta, tg)[sel], "no_reject": box_iou_rotated_batched(ta, tg, _flags=1)[sel]}
    full = torch.empty((len(imgs), an.shape[1], 500), device=DEV)
    for world in (1, 8):
        full.fill_(-7.0)
        for r in range(world):
            rows = tile_rows_of(an.shape[1], r, world, dist.TILE_ROWS).to(DEV)
            packed = box_iou_rotated_tiles(ta, tg, r, world, compact=True, tile_rows=dist.TILE_ROWS)
            full[:, rows] = packed[sel][:, : rows.numel()]
        forms["tiles_world%d" % world] = full.clone()
    for name, m in forms.items():
        m = m.cpu().numpy()
        for k, i in enumerate(imgs):
            assert_iou_exact(m[k], ref[k], an[i], gt[i])


def degenerate_sets():
    sets = dict(rbox_sets.nested_sets())
    sets["slivers"] = rbox_sets.slivers(300, 5)
    thin, fat = rbox_sets.thin_and_fat()
    sets["thin_fat"] = np.concatenate([thin, fat])
    sets["adversarial"] = np.concatenate([synth.adversarial_boxes()] * 30)
    return sets


def test_iou_degenerate_sets_exact(oracle):
    """Shared-edge nested pairs, slivers, thin/fat and adversarial boxes: bit for bit, with one column per thread
    (m = 65) and two (m = 500), every tile height, and the reject tests off."""
    from s2anet_b200.box_iou_rotated import box_iou_rotated, box_iou_rotated_tiles
    for name, x in degenerate_sets().items():
        x = x[:1200]
        for m in (65, 500):
            y = x[:m] if len(x) >= m else np.resize(x, (m, 5))
            ref = oracle.box_iou_rotated(x, y)
            tx, ty = T(x), T(y)
            assert_iou_exact(box_iou_rotated(tx, ty).cpu().numpy(), ref, x, y)
            assert_iou_exact(box_iou_rotated(tx, ty, _flags=1).cpu().numpy(), ref, x, y)
            for tr in (32, 64, 128, 256):
                got = box_iou_rotated_tiles(tx[None], ty[None], 0, 1, compact=True, tile_rows=tr)[0, : len(x)]
                assert_iou_exact(got.cpu().numpy(), ref, x, y)


# ---------------------------------------------------------------------------------------------------------------------
# assign_labels
# ---------------------------------------------------------------------------------------------------------------------
def grid_anchors_all():
    """FAM grid anchors of all five levels of a 1024^2 image (21,824, theta = 0)."""
    return np.concatenate([synth.grid_anchors(1024 // s, 1024 // s, s).reshape(-1, 5) for s in synth.STRIDES])


def p3(i, j, dx=0.0, dy=0.0, w=32.0, h=32.0):
    """A box (x, y, w, h, 0) centred dx, dy off P3 grid anchor (i, j); every coordinate is dyadic."""
    return (8 * i + 3.5 + dx, 8 * j + 3.5 + dy, w, h, 0.0)


# name -> GTs: each built around its own P3 anchor, 12 anchors (96 px) apart
TIE_GTS = {
    "two_way": [p3(10, 10, 4, 0, 24, 24)],                  # centred between two anchors
    "four_way": [p3(22, 10, 4, 4, 24, 24)],                 # between four
    "three_at_half": [p3(34, 10, 0, 0, 32, 16)],            # three anchors at exactly 0.5f, which is the GT's max
    "dup_nonbest_half": [p3(46, 10, 0, 0, 32, 40)] * 2,     # best 0.8; the anchors 8 px up and down sit at 0.5f
    "nonbest_04": [p3(58, 10, 4, 0, 24, 32)],               # best 0.75; a neighbour at exactly 0.4f
    "best_04": [p3(70, 10, 0, 0, 48, 16)],                  # 512 / 1280 = 0.4f is the GT's max
    "quarter": [p3(82, 10, 0, 0, 16, 16)],                  # max 0.25f (= min_pos_iou_thr below)
    "dup_best": [p3(94, 10, 0, 0, 32, 24)] * 2,             # duplicates: the later one takes the shared best anchor
}


def tie_gts():
    return np.array([g for v in TIE_GTS.values() for g in v], F32)


def check_tie_cases(iou):
    """The constructed cases are present in the oracle's IoU matrix (columns in TIE_GTS order)."""
    gmx = iou.max(0)
    ties = (iou == gmx[None]).sum(0)
    k = 0
    got = {}
    for name, v in TIE_GTS.items():
        got[name] = (float(gmx[k]), int(ties[k]))
        k += len(v)
    assert got["two_way"][1] == 2 and got["four_way"][1] == 4 and got["three_at_half"] == (0.5, 3)
    assert got["quarter"][0] == 0.25 and got["best_04"][0] == F32(0.4)
    rmx = iou.max(1)
    assert (rmx == 0.5).sum() >= 5 and (rmx == F32(0.4)).sum() >= 1


_ASSIGN_KW = [dict(gt_max_assign_all=a, min_pos_iou_thr=m) for a in (True, False) for m in (0.0, 0.25)]


def run_assign(anchors, gts, counts=None, **kw):
    from s2anet_b200.assign import assign_labels_batched
    c = None if counts is None else torch.tensor(counts, dtype=torch.int32, device=DEV)
    return assign_labels_batched(T(anchors), T(gts), c, **kw).cpu().numpy()


def test_assign_grid_anchor_ties(oracle):
    an = grid_anchors_all()
    g = np.concatenate([tie_gts(), synth.dota_like_gt(20, 5)])
    iou = oracle.box_iou_rotated(an, g)
    check_tie_cases(iou[:, : len(tie_gts())])
    for kw in _ASSIGN_KW:
        want = oracle.assign_labels(an, g, ious=iou, **kw)
        np.testing.assert_array_equal(run_assign(an[None], g[None], **kw)[0], want, err_msg=str(kw))
    # the cases decide labels: positives at exactly 0.5f, the 0.4f neighbour ignored, the later duplicate wins
    want = oracle.assign_labels(an, g, ious=iou)
    k = {n: sum(len(v) for v in list(TIE_GTS.values())[:i]) for i, n in enumerate(TIE_GTS)}
    assert (want == k["dup_nonbest_half"]).sum() >= 2 and (want == k["dup_nonbest_half"] + 1).sum() >= 1
    assert (want == k["dup_best"] + 1).sum() >= 1


@pytest.mark.parametrize("n", [1, 255, 256, 257, 513])
def test_assign_column_tiles_and_counts(oracle, n):
    """Ties straddling the 256-wide GT tiles (duplicates at 255 / 256), M not a multiple of 64, and a batch of three
    whose gt_counts are 0, Nmax, above Nmax and negative (the kernel clamps them to [0, Nmax])."""
    an = grid_anchors_all()[:4133]                               # P3 rows 0..32 and a partial 64-row block
    rng = np.random.default_rng(n)
    g = synth.dota_like_gt(n, 200 + n)
    g[:, 1] = rng.uniform(0, 260, n).astype(F32)
    ties = tie_gts()
    if n == 1:
        g[0] = ties[0]
    elif n < 257:
        g[n - len(ties):] = ties                                 # the last ones end at the tile edge (or one before)
    else:
        k = min(250, n - len(ties))
        g[k:k + len(ties)] = ties
        g[255] = g[256] = p3(46, 10, 0, 0, 32, 40)               # duplicates on both sides of the edge
    iou = oracle.box_iou_rotated(an, g)
    gb = np.stack([g, g, g])
    for counts in ([0, n, n + 7], [-3, n, n // 2]):
        for kw in _ASSIGN_KW[:2]:
            got = run_assign(np.stack([an] * 3), gb, counts, **kw)
            for b, c in enumerate(counts):
                c = min(max(c, 0), n)
                want = oracle.assign_labels(an, g[:c], ious=iou[:, :c] if c else None, **kw)
                np.testing.assert_array_equal(got[b], want, err_msg="%s %s image %d" % (counts, kw, b))


def test_assign_non_square_image_filter(oracle):
    """imgs_size = (800, 1333): anchors exactly on the filter's edges (x = W and y = H kept, w = W and h = H dropped,
    x one float above W dropped), and the whole P3 grid, whose rows below y = 800 only the height bound drops."""
    H, W = 800, 1333
    up = float(np.nextafter(F32(W), F32(np.inf)))
    edge = np.array([(W, 400, 32, 32, 0), (600, H, 32, 32, 0), (600, 300, W, 32, 0), (600, 500, 32, H, 0),
                     (up, 200, 32, 32, 0), (1000, 600, 32, 32, 0), (W, H, 64, 64, 0)], F32)
    an = np.concatenate([edge, synth.grid_anchors(128, 128, 8).reshape(-1, 5)])
    g = np.concatenate([edge, synth.dota_like_gt(30, 9)])
    g[2, 2], g[3, 3] = 700, 420              # GTs of the over-wide / over-tall anchors: IoU 0.525, positive if kept
    iou = oracle.box_iou_rotated(an, g)
    for kw in _ASSIGN_KW:
        want = oracle.assign_labels(an, g, imgs_size=(H, W), ious=iou, **kw)
        np.testing.assert_array_equal(run_assign(an[None], g[None], imgs_size=(H, W), **kw)[0], want, err_msg=str(kw))
    want = oracle.assign_labels(an, g, imgs_size=(H, W), ious=iou)
    assert want[0] >= 0 and want[1] >= 0 and want[5] >= 0 and want[6] >= 0
    assert want[2] == -2 and want[3] == -2 and want[4] == -2


def test_assign_iou_outside_range_and_nan(oracle):
    """Nested shared-edge pairs whose reference IoU is above 1 count as -0.5 in both; a GT with a NaN size makes
    every row maximum and its own maximum NaN (torch.max propagates NaN): those anchors are neither negative nor
    positive, unless another GT's maximum takes them; a NaN centre gives IoU 0."""
    o, i = rbox_sets.nested_pairs(3000, 41, shift=False)
    v = np.array([oracle.single_iou(a, b) for a, b in zip(o, i)])      # IoU(outer, inner): up to 1.0000081
    over = v > 1
    assert over.sum() >= 20
    an = np.concatenate([o[over], i[over], synth.grid_anchors(64, 64, 16).reshape(-1, 5)])
    g = np.concatenate([i[over], synth.dota_like_gt(40, 3)])
    iou = oracle.box_iou_rotated(an, g)
    assert (iou > 1).sum() >= 20
    for kw in _ASSIGN_KW:
        want = oracle.assign_labels(an, g, ious=iou, **kw)
        np.testing.assert_array_equal(run_assign(an[None], g[None], **kw)[0], want, err_msg=str(kw))
    for col, nan in ((2, "w"), (0, "x")):
        gn = g.copy()
        gn[5, col] = np.nan
        iou = oracle.box_iou_rotated(an, gn)
        assert np.isnan(iou[:, 5]).all() == (nan == "w")
        for kw in _ASSIGN_KW:
            want = oracle.assign_labels(an, gn, ious=iou, **kw)
            np.testing.assert_array_equal(run_assign(an[None], gn[None], **kw)[0], want, err_msg="%s %s" % (nan, kw))
        if nan == "w":
            assert (want == -2).sum() > len(an) // 2 and (want >= 0).sum() >= 1


def test_assign_bench_shape(oracle):
    """Two images of refined anchors (all levels) x 500 GTs, on the oracle's IoU."""
    B = 2
    an = synth.all_level_anchors(B, 3)
    gt = np.stack([synth.dota_like_gt(500, 100 + i) for i in range(B)])
    ious = oracle_images([(an[i], gt[i]) for i in range(B)])
    got = run_assign(an, gt)
    for b in range(B):
        np.testing.assert_array_equal(got[b], oracle.assign_labels(an[b], gt[b], ious=ious[b]))
        assert (got[b] >= 0).sum() > 100
