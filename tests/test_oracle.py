"""CPU tests (-m "not gpu"): the oracle against the golden vectors produced by the reference
itself (tests/golden/make_golden.py), against oracle/_ref when it is present, and the product's
__host__ __device__ IoU source (csrc/rbox_iou.cuh) executed on the host against the oracle."""
import ctypes as C
import hashlib
import os
import shutil
import subprocess

import numpy as np
import pytest

import rbox_sets
from conftest import ROOT, bits
from s2anet_b200 import synth


def test_iou_matches_reference_header_cuda_semantics(oracle, golden):
    g = golden("cfg1_iou_nms.npz")
    boxes = g["boxes"]
    np.testing.assert_array_equal(boxes, synth.clustered_boxes(seed=0)[0])     # generator is pinned too
    full = oracle.box_iou_rotated(boxes, boxes)
    # bit-exact against the reference header (device-side hull ordering) on the stored rows ...
    np.testing.assert_array_equal(bits(full[:200]), bits(g["iou_rows_0_200_ref_hdr_cuda"]))
    # ... and on the whole 2000x2000 matrix through its checksum
    sha = hashlib.sha256(np.ascontiguousarray(full).tobytes()).hexdigest()
    assert sha == bytes(g["iou_full_sha256_ref_hdr_cuda"]).decode()
    np.testing.assert_allclose(full.astype(np.float64).sum(1), g["iou_full_rowsum_ref_hdr_cuda"], rtol=0, atol=0)


def test_iou_vs_reference_cpu_extension(oracle, golden):
    """The reference's CPU build orders hull points with std::sort (SURVEY A.4); it may differ from
    its CUDA build in the last ulp.  north_star tolerance for IoU: 1e-5 absolute."""
    g = golden("cfg1_iou_nms.npz")
    mine = oracle.box_iou_rotated(g["boxes"][:200], g["boxes"])
    ref = g["iou_rows_0_200_ref_ext_cpu"]
    assert np.abs(mine - ref).max() <= 1e-5
    assert (bits(mine) != bits(ref)).mean() < 1e-4


def test_iou_adversarial(oracle, golden):
    g = golden("adversarial_iou.npz")
    mine = oracle.box_iou_rotated(g["boxes"], g["boxes"])
    np.testing.assert_array_equal(bits(mine), bits(g["iou_ref_hdr_cuda"]))
    assert np.nanmax(np.abs(mine - g["iou_ref_ext_cpu"])) <= 1e-5
    # the only known answer in the reference tree: unit square vs half-shifted square = 1/7
    # (DOTA_devkit/polyiou/csrc/polyiou.cpp:130-143)
    assert abs(oracle.single_iou([0, 0, 1, 1, 0], [0.5, 0.5, 1, 1, 0]) - 1.0 / 7.0) < 1e-6
    assert oracle.single_iou([0, 0, 0, 5, 0.3], [0, 0, 4, 5, 0.3]) == 0.0          # zero-area early-out


def test_iou_anchor_gt(oracle, golden):
    g = golden("cfg4_anchor_gt_iou.npz")
    np.testing.assert_array_equal(synth.all_level_anchors(1, 3)[0][::16], g["anchors"])
    mine = oracle.box_iou_rotated(g["anchors"], g["gts"])
    np.testing.assert_array_equal(bits(mine), bits(g["iou_ref_hdr_cuda"]))


def test_iou_empty(oracle):
    assert oracle.box_iou_rotated(np.zeros((0, 5)), np.zeros((3, 5))).shape == (0, 3)
    assert oracle.box_iou_rotated(np.zeros((3, 5)), np.zeros((0, 5))).shape == (3, 0)


def test_nms_keep_lists(oracle, golden):
    g = golden("cfg1_iou_nms.npz")
    b, s, l = g["boxes"], g["scores"], g["labels"]
    np.testing.assert_array_equal(oracle.nms_rotated(b, s, 0.5), g["keep_nms_thr05_cuda_semantics"])
    np.testing.assert_array_equal(oracle.nms_rotated(b, s, 0.5, labels=l), g["keep_mlnms_thr05_cuda_semantics"])
    # the reference's CPU extension (>= predicate): the oracle's ge mode reproduces its keep lists
    np.testing.assert_array_equal(oracle.nms_rotated(b, s, 0.5, ge=True), g["keep_nms_thr05_ref_ext_cpu"])
    np.testing.assert_array_equal(oracle.nms_rotated(b, s, 0.5, labels=l, ge=True), g["keep_mlnms_thr05_ref_ext_cpu"])
    assert oracle.nms_rotated(np.zeros((0, 5)), np.zeros((0,)), 0.5).shape == (0,)


def test_nms_properties(oracle):
    b, s, l = synth.clustered_boxes(n_seed=60, rep=4, seed=5)
    keep = oracle.nms_rotated(b, s, 0.3)
    assert np.all(np.diff(s[keep]) <= 0)                       # descending score
    again = oracle.nms_rotated(b[keep], s[keep], 0.3)          # idempotent
    np.testing.assert_array_equal(again, np.arange(len(keep)))
    iou = oracle.box_iou_rotated(b[keep], b[keep])
    assert (np.triu(iou, 1) > 0.3).sum() == 0                  # no kept pair above threshold
    # one class per box == class-agnostic NMS per class
    ml = oracle.nms_rotated(b, s, 0.3, labels=l)
    per_class = np.concatenate([np.nonzero(l == c)[0][oracle.nms_rotated(b[l == c], s[l == c], 0.3)]
                                for c in np.unique(l)])
    assert set(ml.tolist()) == set(per_class.tolist())


def test_multiclass_wrapper(oracle):
    rng = np.random.default_rng(2)
    b, _, _ = synth.clustered_boxes(n_seed=40, rep=3, seed=9)
    sc = rng.uniform(0, 0.2, (b.shape[0], 15)).astype(np.float32)
    dets, labels = oracle.multiclass_nms_rotated(b, sc, 0.05, 0.5, 2000)
    assert dets.shape[1] == 6 and dets.shape[0] == labels.shape[0] > 0
    assert np.all(np.diff(dets[:, 5]) <= 0)
    d2, l2 = oracle.multiclass_nms_rotated(b, sc, 0.05, 0.5, 50)
    np.testing.assert_array_equal(d2, dets[:50])
    e, el = oracle.multiclass_nms_rotated(b, sc * 0, 0.05, 0.5, 50)
    assert e.shape == (0, 6) and el.shape == (0,)


def test_arf_and_orconv(oracle, golden):
    g = golden("orconv_small.npz")
    np.testing.assert_array_equal(oracle.arf_indices(1, 8, 3), g["indices_1_8"])
    np.testing.assert_array_equal(oracle.arf_indices(8, 8, 3), g["indices_8_8"])
    np.testing.assert_array_equal(oracle.arf_forward(g["weight"], g["indices_1_8"]), g["rotated"])
    out, pooled = oracle.orconv_forward(g["x"], g["weight"], g["indices_1_8"], g["bias"], pad=1, pool_group=8)
    np.testing.assert_allclose(out, g["out"], rtol=1e-5, atol=1e-6)
    np.testing.assert_allclose(pooled, g["pooled"], rtol=1e-5, atol=1e-6)
    # ARF backward is the adjoint of forward: <ARF(w), g> == <w, ARF^T(g)>
    rng = np.random.default_rng(0)
    w = rng.normal(size=(3, 2, 8, 3, 3)).astype(np.float32)
    idx = oracle.arf_indices(8, 8, 3)
    go = rng.normal(size=(24, 16, 3, 3)).astype(np.float32)
    lhs = float((oracle.arf_forward(w, idx).astype(np.float64) * go).sum())
    rhs = float((w.astype(np.float64) * oracle.arf_backward(idx, go, 3, 2)).sum())
    assert abs(lhs - rhs) < 1e-3


def test_alignconv_and_deform_conv(oracle, golden):
    g = golden("alignconv_small.npz")
    x, anc, w, stride = g["x"], g["anchors"], g["weight"], float(g["stride"])
    B, _, H, W = x.shape
    off = np.stack([oracle.alignconv_offset(anc[i].reshape(-1, 5), H, W, stride) for i in range(B)])
    np.testing.assert_allclose(off, g["offset_ref_py"], rtol=0, atol=2e-5)      # reference get_offset (torch cos/sin)
    y = oracle.alignconv_forward(x, anc, w, stride)
    np.testing.assert_allclose(y, g["out_torchvision"], rtol=1e-4, atol=1e-4)
    y2 = oracle.deform_conv_forward(x, g["offset2"], w, stride=(2, 2), padding=(2, 2), dilation=(2, 2),
                                    deformable_groups=2)
    np.testing.assert_allclose(y2, g["out2_torchvision"], rtol=1e-4, atol=1e-4)


def test_oracle_vs_ref_shims_when_present(oracle):
    """In the authoring container oracle/_ref holds the reference header compiled in place."""
    b, _, _ = synth.clustered_boxes(n_seed=80, rep=5, seed=11)
    ref = oracle.ref_pairwise("iou", "cudasem", b, b)
    if ref is None:
        pytest.skip("oracle/_ref not built (reference not mounted)")
    np.testing.assert_array_equal(bits(oracle.box_iou_rotated(b, b)), bits(ref))


@pytest.fixture(scope="module")
def host_harness():
    if shutil.which("nvcc") is None:
        pytest.skip("nvcc not available")
    out = os.path.join(ROOT, "tests", "_build", "libhost_harness.so")
    src = os.path.join(ROOT, "tests", "host_harness.cu")
    hdr = os.path.join(ROOT, "s2anet_b200", "csrc", "rbox_iou.cuh")
    hdr2 = os.path.join(ROOT, "s2anet_b200", "csrc", "poly_iou.cuh")
    os.makedirs(os.path.dirname(out), exist_ok=True)
    if not os.path.exists(out) or os.path.getmtime(out) < max(os.path.getmtime(src), os.path.getmtime(hdr), os.path.getmtime(hdr2)):
        subprocess.check_call(["nvcc", "-O2", "-x", "cu", "-shared", "-Xcompiler", "-fPIC,-ffp-contract=off",
                               "-gencode", "arch=compute_100a,code=sm_100a", "-o", out, src])
    L = C.CDLL(out)
    f32p = np.ctypeslib.ndpointer(np.float32, flags="C")
    L.hh_pairwise.argtypes = [f32p, C.c_int64, f32p, C.c_int64, f32p, C.c_int]

    f64p = np.ctypeslib.ndpointer(np.float64, flags="C")
    L.hh_poly_iou_pairs.argtypes = [f64p, f64p, C.c_int64, f64p]
    L.hh_inter_upper_bound.argtypes = [f32p, C.c_int64, f32p, C.c_int64, f32p]
    L.hh_nms_cannot_exceed.argtypes = [f32p, C.c_int64, f32p, C.c_int64, f32p, np.ctypeslib.ndpointer(np.uint8, flags="C")]

    def run(b1, b2, mode):
        b1, b2 = np.ascontiguousarray(b1, np.float32), np.ascontiguousarray(b2, np.float32)
        out_ = np.empty((len(b1), len(b2)), np.float32)
        L.hh_pairwise(b1, len(b1), b2, len(b2), out_, mode)
        return out_

    def poly(p, q):
        p, q = np.ascontiguousarray(p, np.float64), np.ascontiguousarray(q, np.float64)
        out_ = np.empty((len(p),), np.float64)
        L.hh_poly_iou_pairs(p, q, len(p), out_)
        return out_

    def bound(b1, b2):
        b1, b2 = np.ascontiguousarray(b1, np.float32), np.ascontiguousarray(b2, np.float32)
        out_ = np.empty((len(b1), len(b2)), np.float32)
        L.hh_inter_upper_bound(b1, len(b1), b2, len(b2), out_)
        return out_
    def skip(b1, b2, thr):
        b1, b2 = np.ascontiguousarray(b1, np.float32), np.ascontiguousarray(b2, np.float32)
        thr = np.ascontiguousarray(np.broadcast_to(np.asarray(thr, np.float32), (len(b1), len(b2))))
        out_ = np.empty((len(b1), len(b2)), np.uint8)
        L.hh_nms_cannot_exceed(b1, len(b1), b2, len(b2), thr, out_)
        return out_.astype(bool)
    run.poly, run.bound, run.skip = poly, bound, skip
    return run


def test_product_iou_source_on_host(oracle, host_harness):
    """csrc/rbox_iou.cuh (classify + in-place clipper) is bit-identical to the oracle, with and
    without the disjointness shortcut, on clustered, adversarial and anchor x GT pairs."""
    sets = [(synth.clustered_boxes(n_seed=120, rep=5, seed=3)[0],) * 2,
            (synth.adversarial_boxes(),) * 2,
            (synth.all_level_anchors(1, 7)[0][::23], synth.dota_like_gt(300, 7))]
    # boxes sharing an angle and an edge line: the near-parallel guard must route them to the clipper
    base = np.array([[100, 100, 50, 20, 0.3]], np.float32)
    shifts = np.arange(0, 400, 7, dtype=np.float32)[:, None] * np.array([[np.cos(0.3), np.sin(0.3)]], np.float32)
    col = np.repeat(base, len(shifts), 0)
    col[:, :2] += shifts
    sets.append((col, col))
    # slivers (sides down to 1e-4 of the pair distance and far beyond the guard) near and far from fat boxes, at
    # generic and at shared angles: the relaxed sliver guard (rbox_iou.cuh "Sliver guard") must still only ever
    # predict an exact zero where the reference computes one
    thin, fat = rbox_sets.thin_and_fat()
    sets.append((thin, fat))
    sets.append((thin, thin))
    for b1, b2 in sets:
        ref = oracle.box_iou_rotated(b1, b2)
        # 0 / 1: the general clipper with / without the reject tests; 3 / 4: the IoU kernel's path (fast test -> full
        # classify -> register-resident hull with fall-back) with / without them
        for mode in (0, 1, 3, 4):
            np.testing.assert_array_equal(bits(host_harness(b1, b2, mode)), bits(ref))


def test_product_poly_iou_source_on_host(oracle, host_harness):
    """csrc/poly_iou.cuh (the fp64 polygon IoU of the DOTA result merging) on the CPU: bit-identical to the oracle --
    and therefore to the reference's compiled polyiou.cpp -- on the golden pairs and 5,000 random ones."""
    g = np.load(os.path.join(ROOT, "tests", "golden", "poly_small.npz"))
    with np.errstate(invalid="ignore", divide="ignore"):
        got = host_harness.poly(g["p"], g["q"])
    assert np.all((got.view(np.uint64) == g["iou"].view(np.uint64)) | (np.isnan(got) & np.isnan(g["iou"])))
    p = synth.random_quads(5000, np.random.default_rng(31))
    q = p + np.random.default_rng(32).normal(0, 6, p.shape)
    np.testing.assert_array_equal(host_harness.poly(p, q).view(np.uint64), oracle.poly_iou_pairs(p, q).view(np.uint64))


def test_nms_intersection_bound_is_an_upper_bound(oracle, host_harness):
    """rbox_inter_upper_bound (NMS kernels: skip a clip when even this bound cannot reach the threshold) never
    undercuts the intersection area the reference's IoU implies, on clustered and adversarial boxes."""
    for boxes in (synth.clustered_boxes(n_seed=150, rep=5, seed=5)[0], synth.adversarial_boxes()):
        b = boxes[(boxes[:, 2] > 0) & (boxes[:, 3] > 0)]
        iou = oracle.box_iou_rotated(b, b).astype(np.float64)
        a = (b[:, 2] * b[:, 3]).astype(np.float64)
        inter = iou * (a[:, None] + a[None, :]) / (1.0 + iou)
        ub = host_harness.bound(b, b).astype(np.float64)
        assert np.all(inter <= ub * 1.001 + 1e-6 * (a[:, None] + a[None, :])), float((inter - ub).max())
        # and it is useful: most overlapping-but-not-suppressing pairs are decided without a clip at thr = 0.5
        cand = (iou > 0) & (iou <= 0.5)
        skipped = 1.001 * ub < 0.999 * 0.5 * (a[:, None] + a[None, :] - 1.001 * ub)
        assert not np.any(skipped & (iou > 0.5))
        if cand.sum() > 1000:
            assert (skipped & cand).sum() > 0.5 * cand.sum()


def test_angle_screen():
    """rbox_sets.angle_may_differ flags an angle whose float64 sine is 2 double ulps from an fp32 rounding midpoint
    (found by a search over 10^8 random fp32 angles), not its neighbours, and almost no random angle."""
    hit = np.array([0xbef3830f], np.uint32).view(np.float32)
    assert rbox_sets.angle_may_differ(hit).all()
    assert not rbox_sets.angle_may_differ(np.nextafter(hit, np.float32(1))).any()
    t = np.random.default_rng(0).uniform(-np.pi, np.pi, 100000).astype(np.float32)
    assert rbox_sets.angle_may_differ(t).sum() <= 2


def test_nms_clip_skip_never_hides_a_suppression(oracle, host_harness):
    """rbox_nms_cannot_exceed (the NMS kernels' "no clip" decision) may only say "cannot exceed thr" for a pair whose
    oracle IoU is <= thr: at thr 0.1 ... 0.9 and just below each pair's own IoU (one ulp, 0.1 % and 1 % under).  The
    sets hold what breaks a purely geometric bound: boxes sharing both long edge lines (the reference's IoU of such a
    pair is up to 1.0 for a true 0.49), the same with the inner edges 1e-7 ... 1e-2 of the height apart, axis-aligned,
    diagonal and vertical ones, slivers down to 1e-4 px, and the existing thin/fat, clustered and adversarial sets."""
    sets = dict(rbox_sets.nested_sets())
    sets["slivers"] = rbox_sets.slivers(300, 5)
    thin, fat = rbox_sets.thin_and_fat()
    sets["thin_fat"] = (thin, fat)
    sets["thin_thin"] = thin
    sets["clustered"] = synth.clustered_boxes(n_seed=150, rep=5, seed=5)[0]
    sets["adversarial"] = synth.adversarial_boxes()
    bad = {}
    for name, s in sets.items():
        b1, b2 = s if isinstance(s, tuple) else (s, s)
        iou = oracle.box_iou_rotated(b1, b2)
        with np.errstate(invalid="ignore"):
            thrs = [np.float32(t) for t in (0.1, 0.3, 0.5, 0.7, 0.9)] + [
                np.nextafter(iou, np.float32(-np.inf)), np.float32(0.999) * iou, np.float32(0.99) * iou]
            for thr in thrs:
                wrong = host_harness.skip(b1, b2, thr) & (iou > thr)
                if wrong.any():
                    bad[name] = bad.get(name, 0) + int(wrong.sum())
    assert not bad, "pairs skipped although their IoU exceeds the threshold: %s" % bad
    # the nested sets really are the hard case: many of their pairs sit far above the true IoU
    g = sets["generic"]
    v = np.array([oracle.single_iou(g[2 * k], g[2 * k + 1]) for k in range(len(g) // 2)])
    assert (v > 0.5).sum() > 20
    # and the skip is still useful: most overlapping-but-not-suppressing clustered pairs are decided without a clip
    b = sets["clustered"]
    iou = oracle.box_iou_rotated(b, b)
    cand = (iou > 0) & (iou <= 0.5)
    assert cand.sum() > 1000
    assert (host_harness.skip(b, b, 0.5) & cand).sum() > 0.5 * cand.sum()
