"""The box decode, bit for bit: fam_decode_kernel, the FAM-decode epilogue of the plain tensor-core conv and the decode and
scores of select_decode against the op-by-op model of tests/decode_reference.py, on the clamp, wrap and overflow edges.

cosf, sinf and expf are not correctly rounded, so the model takes them from the device itself (DeviceMath, probed
through select_decode); everything around them -- the order and rounding of every fp32 operation, the T-roundings of
exp and pi*da, the clamp bound, the angle wrap -- is checked exactly.  The CPU tests pin the model's operation order to
the oracle's (oracle.delta2bbox_rotated) given numpy's transcendentals.

Non-finite logits are ranked as the reference ranks them (models/head.py:700-701: scores.max(dim=1), then topk): a
location's best score is NaN if any class is NaN, NaN ranks above every number, and equal scores -- NaN included -- go
to the ascending location.
"""
import math

import numpy as np
import pytest
import torch

from conftest import bits
from decode_reference import (CLIPS, DTYPES, F32, PI, QPI, DeviceMath, assert_same, clamp_limit, decode_model,
                              edge_angles, edge_deltas, free_landing_rows, grid_anchor_model, numpy_math, same_bits,
                              sigmoid_model, t_step, to_t)
from test_gpu_postprocess_exact import _place, reference_topk

DEV = "cuda:0"
IDS = {torch.float32: "f32", torch.bfloat16: "bf16", torch.float16: "f16"}
STRIDES5 = (8, 16, 32, 64, 128)


def tie_clip(dtype):
    """A wh_ratio_clip whose |log| lies within half a float ulp of a `dtype` rounding tie (on the side where rounding
    the double straight to `dtype` and rounding it through float disagree): returns (clip, bound through float, bound
    rounded once)."""
    lo, hi = F32(2.5), t_step(F32(2.5), dtype, np.inf)[()]          # (exp of either fits T and tells them apart)
    tie = (float(lo) + float(hi)) / 2
    even_hi = int(torch.tensor([float(hi)]).to(dtype).view(torch.int16)) % 2 == 0
    L = tie - 2.0 ** -26 if even_hi else tie + 2.0 ** -26     # float(L) == tie, which rounds to the even neighbour
    clip = math.exp(-L)
    Lr = abs(math.log(clip))
    assert F32(Lr) == F32(tie) and Lr != tie
    through_float = F32(clamp_limit(clip, dtype))
    once = float(hi) if Lr > tie else float(lo)
    assert through_float != F32(once)
    return clip, through_float, F32(once)


# ------------------------------------------------------------------------------------------------
# CPU: the model against the oracle
# ------------------------------------------------------------------------------------------------
def test_model_equals_the_oracle_on_the_golden_vectors(oracle, golden):
    g = golden("decode_small.npz")
    cos, sin, exp = numpy_math()
    for l, ((H, W), s) in enumerate(zip(g["sizes"], g["strides"])):
        a = grid_anchor_model(H, W, s, 4.0, 0.0)[None]
        assert np.array_equal(bits(a[0]), bits(oracle.grid_anchors(H, W, s)))
        d32 = np.transpose(g["fam_pred_%d" % l], (0, 2, 3, 1))
        for dt, npdt in ((torch.float32, np.float32), (torch.float16, np.float16)):
            d = d32.astype(npdt)
            want = oracle.delta2bbox_rotated(a, d, 1e-6)
            assert_same(decode_model(a, d.astype(F32), dt, 1e-6, cos, sin, exp), want, "level %d %s" % (l, dt))
    for b in range(g["cls_0"].shape[0]):
        for l in range(len(g["strides"])):
            a = g["refine_%d" % l][b].reshape(-1, 5)
            d = np.transpose(g["reg_%d" % l][b], (1, 2, 0)).reshape(-1, 5)
            assert_same(decode_model(a, d, torch.float32, 16 / 1000, cos, sin, exp), oracle.delta2bbox_rotated(a, d))
            x = g["cls_%d" % l][b]
            for dt, npdt in ((torch.float32, np.float32), (torch.float16, np.float16)):
                assert_same(sigmoid_model(x.astype(npdt).astype(F32), dt, exp), oracle.sigmoid_in(x.astype(npdt)))


@pytest.mark.parametrize("dtype", [torch.float32, torch.float16], ids=["f32", "f16"])
@pytest.mark.parametrize("clip", CLIPS)
def test_model_equals_the_oracle_on_edge_data(oracle, dtype, clip):
    rng = np.random.default_rng(7)
    cos, sin, exp = numpy_math()
    angles = edge_angles(dtype, rng)
    for theta in (F32(0.0), F32(-np.pi / 4), np.nextafter(F32(3 * np.pi / 4), F32(0))):
        d, kinds = edge_deltas(dtype, clip, theta, rng, n_random=200)
        a = np.stack([rng.uniform(0, 1024, len(d)), rng.uniform(0, 1024, len(d)), rng.uniform(8, 64, len(d)),
                      rng.uniform(8, 64, len(d)), np.full(len(d), theta)], 1).astype(F32)
        npdt = np.float16 if dtype == torch.float16 else np.float32
        assert_same(decode_model(a, d, dtype, clip, cos, sin, exp), oracle.delta2bbox_rotated(a, d.astype(npdt), clip))
        # the same deltas against anchors at every edge angle
        a2 = np.repeat(a[:1], len(angles), 0)
        a2[:, 4] = angles
        d2 = d[rng.integers(0, len(d), len(angles))]
        assert_same(decode_model(a2, d2, dtype, clip, cos, sin, exp), oracle.delta2bbox_rotated(a2, d2.astype(npdt), clip))
    for da, th in free_landing_rows(dtype, rng):
        a = np.array([[10.0, 20.0, 16.0, 16.0, th]], F32)
        d = np.array([[0.5, 0.25, 0.0, 0.0, da]], F32)
        assert_same(decode_model(a, d, dtype, clip, cos, sin, exp), oracle.delta2bbox_rotated(a, d.astype(npdt), clip))


def test_grid_anchor_model_equals_the_oracle(oracle):
    for H, W, s, scale, angle in ((1, 1, 8, 4.0, 0.0), (37, 53, 16, 4.0, 0.0), (5, 7, 128, 3.7, 0.5), (64, 64, 8, 4.5, -0.7)):
        assert np.array_equal(bits(grid_anchor_model(H, W, s, scale, angle)), bits(oracle.grid_anchors(H, W, s, scale, angle)))


def test_edge_data_hits_every_wrap_case():
    """Across the anchor angles the tests use, every dtype gets delta angles landing exactly on 0, on a multiple of pi,
    and one float below them; select_decode's free anchor angles land on all of them in every dtype."""
    rng = np.random.default_rng(1)
    for dt in DTYPES:
        seen = {"zero": 0, "multiple": 0, "below": 0}
        for th in FAM_ANGLES:
            for k, n in edge_deltas(dt, 1e-6, F32(th), rng)[1].items():
                seen[k] += n
        assert seen["zero"] > 0 and seen["multiple"] > 0, (dt, seen)
        assert len(free_landing_rows(dt, rng)) >= 4 * 4, dt


def test_clamp_bound_tie_clip_exists():
    for dt in (torch.bfloat16, torch.float16):
        tie_clip(dt)


# ------------------------------------------------------------------------------------------------
# GPU: the probe
# ------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def dm():
    return DeviceMath(DEV)


def _ulp32(v):
    v = np.abs(np.asarray(v, np.float64))
    f = np.minimum(v, np.float64(np.finfo(F32).max)).astype(F32)
    return np.maximum(np.spacing(f).astype(np.float64), 2.0 ** -149)


@pytest.mark.gpu
def test_probe_is_within_2_ulp_of_float64(dm):
    """expf / sinf / cosf without fast math are within 2 ulp (CUDA C Programming Guide, mathematical functions): a
    __expf or __cosf in the decode would not be."""
    rng = np.random.default_rng(0)
    lims = [clamp_limit(c, dt) for c in CLIPS for dt in DTYPES]
    ex = [np.linspace(-30, 30, 20001, dtype=F32), np.linspace(80, 88.7, 2001, dtype=F32),
          np.linspace(-104, -80, 2001, dtype=F32), rng.normal(0, 3, 4000).astype(F32)]
    for lim in lims:
        v = F32(lim)
        ex += [np.array([v, -v, np.nextafter(v, F32(0)), np.nextafter(v, F32(99)), np.nextafter(-v, F32(-99))], F32)]
    mx = np.nextafter(F32(np.log(np.finfo(F32).max)), F32(0))
    ex += [np.array([mx, np.nextafter(mx, F32(99)), np.nextafter(mx, F32(0))], F32)]
    ex = np.concatenate(ex)
    ang = [np.linspace(-4, 4, 20001, dtype=F32), rng.uniform(-np.pi / 4, 3 * np.pi / 4, 4000).astype(F32)]
    for c in (0.0, np.pi / 4, -np.pi / 4, np.pi / 2, -np.pi / 2, 3 * np.pi / 4):
        v = F32(c)
        ang.append(np.array([v + F32(k) * np.spacing(v) if v else F32(k) * F32(1e-30) for k in range(-8, 9)], F32))
    ang = np.concatenate(ang)
    ang = ang[ang != 0]
    dm.prefetch(angles=ang, exps=ex)
    for name, x, f in (("exp", ex, np.exp), ("cos", ang, np.cos), ("sin", ang, np.sin)):
        got = getattr(dm, name)(x).astype(np.float64)
        with np.errstate(over="ignore"):
            want = f(x.astype(np.float64))
        fin = np.isfinite(got)
        over = want > np.finfo(F32).max * (1 + 2.0 ** -24)
        assert np.all(fin | over), name
        err = np.abs(got[fin] - want[fin]) / _ulp32(want[fin])
        assert err.max() <= 2.0, "%s: %.2f ulp at %r" % (name, err.max(), x[fin][np.argmax(err)])
    # the overflow point: expf(88.7228...) is the last finite value
    assert np.isfinite(dm.exp(np.array([mx], F32)))[0]


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float16], ids=["bf16", "f16"])
def test_clamp_bound_rounds_like_torch(dm, dtype):
    """|log(clip)| within half a float ulp of a T tie: torch.clamp on a T CUDA tensor rounds its bound through float
    (to the even neighbour), not straight from the double; clamp_limit (box_decode.cuh) and the model do the same."""
    from s2anet_b200.decode import fam_decode, rboxes_decode_torch
    clip, through_float, once = tie_clip(dtype)
    big = to_t(F32(100.0), dtype)[()]
    d = torch.tensor([[0.0, 0.0, big, -big, 0.0]], dtype=dtype, device=DEV)
    a = torch.tensor([[0.0, 0.0, 1.0, 1.0, 0.0]], device=DEV)
    max_ratio = abs(math.log(clip))                          # boxes.py:115-117, as rboxes_decode_torch runs them
    got = d[0, 2:4].clamp(min=-max_ratio, max=max_ratio).float().cpu().numpy()
    assert got.tolist() == [float(through_float), -float(through_float)]
    e = dm.exp(np.array([through_float, once], F32))
    assert to_t(e[0], dtype) != to_t(e[1], dtype)
    assert_same(rboxes_decode_torch(a, d, clip).cpu().numpy(),
                dm.decode(a.cpu().numpy(), d.float().cpu().numpy(), dtype, clip))
    g = torch.zeros(1, 5, 1, 1, dtype=dtype, device=DEV)
    g[0, 2], g[0, 3] = float(big), -float(big)
    got = fam_decode([g], [8], 4.0, 0.0, clip)[0].cpu().numpy().reshape(1, 5)
    want = dm.decode(grid_anchor_model(1, 1, 8, 4.0, 0.0).reshape(1, 5), g.float().cpu().numpy().reshape(1, 5), dtype, clip)
    assert_same(got, want)


# ------------------------------------------------------------------------------------------------
# GPU: fam_decode
# ------------------------------------------------------------------------------------------------
FAM_ANGLES = (0.0, math.pi / 6, -math.pi / 4, float(np.nextafter(F32(3 * math.pi / 4), F32(0))))


def _fill(dtype, clip, theta, shape, rng):
    """[B, H, W, 5] deltas: the edge rows at random places, random ones elsewhere."""
    B, H, W = shape
    n = B * H * W
    edge, _ = edge_deltas(dtype, clip, F32(theta), rng, n_random=0)
    rand = to_t(rng.normal(0, 1, (n, 5)) * np.array([0.3, 0.3, 0.6, 0.6, 0.4]), dtype)
    rows = rand.copy()
    k = min(n, len(edge))
    rows[rng.permutation(n)[:k]] = edge[rng.permutation(len(edge))[:k]]
    return rows.reshape(B, H, W, 5)


def _fam_case(dm, dtype, layout, sizes, B, scale, theta, clip, rng):
    from s2anet_b200.decode import fam_decode
    strides = STRIDES5[:len(sizes)] if len(sizes) <= 5 else [8] * len(sizes)
    deltas = [_fill(dtype, clip, theta, (B, H, W), rng) for H, W in sizes]
    preds = [_place(torch.from_numpy(d).permute(0, 3, 1, 2).contiguous(), layout, dtype, 77.0) for d in deltas]
    out = fam_decode(preds, strides, scale, theta, clip)
    for l, ((H, W), s, d) in enumerate(zip(sizes, strides, deltas)):
        a = np.broadcast_to(grid_anchor_model(H, W, s, scale, theta)[None], d.shape)
        assert_same(out[l].cpu().numpy(), dm.decode(a, d, dtype, clip),
                    "%s %s level %d theta %r clip %r" % (IDS[dtype], layout, l, theta, clip))


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", DTYPES, ids=["f32", "bf16", "f16"])
@pytest.mark.parametrize("layout", ["nchw", "cl", "padded", "misaligned"])
def test_fam_decode_exact(dm, dtype, layout):
    rng = np.random.default_rng(100 * DTYPES.index(dtype) + len(layout))
    odd = [(1, 1), (37, 53), (5, 7)]
    clips = CLIPS + ((tie_clip(dtype)[0],) if dtype != torch.float32 else ())
    for i, theta in enumerate(FAM_ANGLES):
        for clip in clips:
            _fam_case(dm, dtype, layout, odd, 3, 4.0 if i % 2 else 3.7, theta, clip, rng)
    bench = [(1024 // s, 1024 // s) for s in STRIDES5]
    _fam_case(dm, dtype, layout, bench, 2, 4.0, 0.0, 1e-6, rng)


# ------------------------------------------------------------------------------------------------
# GPU: the FAM-decode epilogue of the plain tensor-core conv
# ------------------------------------------------------------------------------------------------
def _head(C, dtype, weight, bias):
    h = torch.nn.Conv2d(C, 5, 1).to(DEV).to(dtype)
    with torch.no_grad():
        h.weight.copy_(weight.to(dtype).view(5, C, 1, 1))
        h.bias.copy_(bias.to(dtype))
    return h


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float16], ids=["bf16", "f16"])
def test_fam_decode_epilogue_exact(dm, dtype):
    """The fused epilogue equals the model applied to the ordinary conv's T output (exact by test_gpu_tc_exact), with the
    deltas steered onto the edges through the head: identity weights pass edge rows through, zero weights with an edge
    bias make every location's deltas T(0 + bias), and sparse small integer weights exercise T(acc + bias)."""
    from s2anet_b200 import conv_tc, decode
    rng = np.random.default_rng(5 if dtype == torch.bfloat16 else 6)
    C = 64
    sizes = [(37, 53), (19, 27), (10, 14), (5, 7), (1, 1)]
    strides = STRIDES5
    B = 2
    theta, scale, clip = -math.pi / 4, 4.0, 1e-6

    def run(xs, head, what):
        with torch.no_grad():
            deltas = conv_tc.conv2d_forward_tc_multi(xs, head.weight, head.bias)
            out = conv_tc.conv2d_forward_tc_fam_decode(xs, head, strides, scale, theta, clip)
            ref = decode.fam_decode(deltas, strides, scale, theta, clip)
        for l, ((H, W), s) in enumerate(zip(sizes, strides)):
            d = deltas[l].permute(0, 2, 3, 1).float().cpu().numpy()
            a = np.broadcast_to(grid_anchor_model(H, W, s, scale, theta)[None], d.shape)
            assert_same(out[l].cpu().numpy(), dm.decode(a, d, dtype, clip), "%s level %d" % (what, l))
            assert_same(out[l].cpu().numpy(), ref[l].cpu().numpy(), "%s level %d vs fam_decode" % (what, l))

    def inputs(first5):
        xs = []
        for (H, W), f in zip(sizes, first5):
            x = torch.from_numpy(to_t(rng.integers(-3, 4, (B, C, H, W)).astype(F32), dtype))
            x[:, :5] = torch.from_numpy(np.ascontiguousarray(np.transpose(f, (0, 3, 1, 2))))
            xs.append(x.to(dtype).to(DEV).contiguous(memory_format=torch.channels_last))
        return xs

    fills = [_fill(dtype, clip, theta, (B, H, W), rng) for H, W in sizes]
    # identity on the first five channels: d = T(x + 0) = x, every edge row as it is
    eye = torch.zeros(5, C)
    eye[:, :5] = torch.eye(5)
    run(inputs(fills), _head(C, dtype, eye, torch.zeros(5)), "identity")
    # sparse small integer weights on finite edge rows and a non-zero bias: T(acc + bias)
    fin = [np.where(np.isfinite(f), f, F32(0.0)) for f in fills]
    w = torch.zeros(5, C)
    w[:, :5] = torch.diag(torch.tensor([2.0, -1.0, 1.0, -1.0, 1.0]))
    w[:, 5:] = torch.from_numpy(rng.choice([0.0, 0.0, 0.0, 1.0, -1.0], (5, C - 5)) * 2.0 ** -10)
    run(inputs(fin), _head(C, dtype, w, torch.tensor([0.3, -0.7, 0.0625, -0.0625, 0.25])), "sparse")
    # zero weights: every location decodes T(bias), the bias on the clamp and wrap edges
    lim = F32(clamp_limit(clip, dtype))
    land = edge_deltas(dtype, clip, F32(theta), rng)[0][-12:, 4]
    zero_in = inputs(fin)
    for bias in ([0.5, -0.5, lim, -lim, 0.0], [0.0, 0.0, t_step(lim, dtype, 99.0), np.inf, land[0]],
                 [1.0, 1.0, -np.inf, np.nan, -0.0], [2.0, -2.0, t_step(lim, dtype, 0.0), -lim, 0.25]):
        run(zero_in, _head(C, dtype, torch.zeros(5, C), torch.tensor(np.array(bias, F32))), "bias %r" % (bias,))


# ------------------------------------------------------------------------------------------------
# GPU: select_decode
# ------------------------------------------------------------------------------------------------
def _select_inputs(dtype, layout, sizes, C, B, rng):
    """logits, deltas (edge rows + random, T values) and refined anchors (free angles: wrap points, pi/2 and the
    landing angles of free_landing_rows), per level, as numpy [B, H, W, *] and as placed CUDA tensors."""
    free = free_landing_rows(dtype, rng, n=3)
    ang = edge_angles(dtype, rng)
    lv = []
    for i, (H, W) in enumerate(sizes):
        n = B * H * W
        d, _ = edge_deltas(dtype, 16 / 1000, F32(0.0), rng, n_random=0)
        rows = to_t(rng.normal(0, 1, (n, 5)) * np.array([0.3, 0.3, 0.6, 0.6, 0.4]), dtype)
        a = np.stack([rng.uniform(0, 1024, n), rng.uniform(0, 1024, n), rng.uniform(8, 64, n), rng.uniform(8, 64, n),
                      rng.choice(ang, n)], 1).astype(F32)
        k = min(n, len(d))
        at = rng.permutation(n)[:k]
        rows[at] = d[rng.permutation(len(d))[:k]]
        at = rng.permutation(n)[:min(n, len(free))]
        for j, p in enumerate(at):
            rows[p, 4], a[p, 4] = free[j]
        logit = to_t(rng.normal(-3.0, 2.0, (n, C)), dtype)
        lv.append((logit.reshape(B, H, W, C), rows.reshape(B, H, W, 5), a.reshape(B, H, W, 5)))
    nchw = lambda x: torch.from_numpy(np.ascontiguousarray(np.transpose(x, (0, 3, 1, 2))))      # noqa: E731
    cls = [_place(nchw(c), layout, dtype, 30.0) for c, _, _ in lv]
    reg = [_place(nchw(r), layout, dtype, 50.0) for _, r, _ in lv]
    anc = [torch.from_numpy(a).to(DEV) for _, _, a in lv]
    return lv, cls, reg, anc


def check_select_exact(dm, dtype, lv, cls, reg, anc, topk, clip=16 / 1000):
    """select_decode against reference_topk on the model's scores, the model's boxes on the gathered rows and
    sigmoid_model's scores; split and single-launch forms."""
    from s2anet_b200.decode import select_decode
    bb, sc, idx = (t.cpu().numpy() for t in select_decode(cls, reg, anc, topk, clip, return_index=True))
    B = bb.shape[0]
    dm.prefetch(angles=np.concatenate([a[..., 4].ravel() for _, _, a in lv]),
                exps=np.concatenate([np.concatenate([-x.ravel(), d[..., 2:4].ravel()]) for x, d, _ in lv]))
    off = 0
    for l, (logit, d, a) in enumerate(lv):
        _, H, W, C = logit.shape
        n = H * W
        k = min(n, topk) if topk > 0 else n
        s_all = dm.sigmoid(logit.reshape(B, n, C), dtype)
        for b in range(B):
            want = reference_topk(s_all[b], topk)
            assert np.array_equal(idx[b, off:off + k], want), "image %d level %d: top-k index differs" % (b, l)
            assert_same(sc[b, off:off + k], s_all[b][want], "scores %d/%d" % (b, l))
            assert_same(bb[b, off:off + k], dm.decode(a[b].reshape(n, 5)[want], d[b].reshape(n, 5)[want], dtype, clip),
                        "boxes %d/%d" % (b, l))
        off += k
    assert off == bb.shape[1]
    return bb, sc, idx


_SELECT = [("padded", 0), ("padded", 300), ("nchw", 300), ("misaligned", 0)]


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", DTYPES, ids=["f32", "bf16", "f16"])
@pytest.mark.parametrize("layout,topk", _SELECT, ids=["%s-k%d" % s for s in _SELECT])
def test_select_decode_exact(dm, dtype, layout, topk, monkeypatch):
    rng = np.random.default_rng(len(layout) * 1000 + topk + 7 * DTYPES.index(dtype))
    lv, cls, reg, anc = _select_inputs(dtype, layout, [(40, 50), (23, 87), (5, 7), (1, 1)], 15, 2, rng)
    monkeypatch.delenv("S2A_DEC_DEBUG", raising=False)
    split = check_select_exact(dm, dtype, lv, cls, reg, anc, topk)
    monkeypatch.setenv("S2A_DEC_DEBUG", "2")                   # the single-launch form
    single = check_select_exact(dm, dtype, lv, cls, reg, anc, topk)
    for x, y in zip(split, single):
        assert same_bits(x, y).all() if x.dtype == np.float32 else np.array_equal(x, y)


# ------------------------------------------------------------------------------------------------
# GPU: the reference's own formulation on the same GPU
# ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("dtype", DTYPES, ids=["f32", "bf16", "f16"])
def test_torch_formulation_on_the_gpu_equals_the_kernels(dm, dtype):
    """rboxes_decode_torch and select_and_decode_torch (torch's CUDA cos / sin / exp / sigmoid, no fast math either) on
    the same edge data give the kernels' bits, and torch's transcendentals give the probed values."""
    from s2anet_b200.decode import fam_decode, rboxes_decode_torch, select_and_decode_torch, select_decode
    rng = np.random.default_rng(11)
    for theta in FAM_ANGLES:
        for clip in CLIPS:
            d = _fill(dtype, clip, theta, (2, 37, 53), rng)
            g = torch.from_numpy(d).permute(0, 3, 1, 2).to(dtype).to(DEV)
            got = fam_decode([g], [16], 4.0, theta, clip)[0]
            a = torch.from_numpy(grid_anchor_model(37, 53, 16, 4.0, theta)).to(DEV)[None]
            want = rboxes_decode_torch(a.reshape(1, -1, 5), g.permute(0, 2, 3, 1).reshape(2, -1, 5), clip)
            assert_same(got.reshape(2, -1, 5).cpu().numpy(), want.cpu().numpy(), "fam theta %r clip %r" % (theta, clip))
    lv, cls, reg, anc = _select_inputs(dtype, "padded", [(40, 50), (5, 7)], 15, 2, rng)
    for topk in (0, 300):
        bb, sc = select_decode(cls, reg, anc, topk)
        tb, ts = select_and_decode_torch(cls, reg, anc, topk)
        assert_same(bb.cpu().numpy(), tb.cpu().numpy(), "select boxes k%d" % topk)
        assert_same(sc.cpu().numpy(), ts.float().cpu().numpy(), "select scores k%d" % topk)
    # the probed values are torch's
    for name, f in (("cos", torch.cos), ("sin", torch.sin), ("exp", torch.exp)):
        k = dm.keys[name].view(F32)
        assert_same(f(torch.from_numpy(k).to(DEV)).cpu().numpy(), dm.vals[name], "torch.%s" % name)


# ------------------------------------------------------------------------------------------------
# GPU: non-finite logits
# ------------------------------------------------------------------------------------------------
def _nonfinite_logits(dtype, B, C, H, W, rng, mode):
    x = to_t(rng.normal(-3.0, 2.0, (B, H, W, C)), dtype)
    n = H * W
    flat = x.reshape(B, n, C)
    for b in range(B):
        p = rng.permutation(n)
        q = np.array([np.nan, -np.nan, np.inf, -np.inf], F32)
        if mode == "single":             # one class of some locations
            for j in range(min(n, 60)):
                flat[b, p[j], rng.integers(0, C)] = q[j % 4]
        elif mode == "all":              # every class of some locations (NaN with both signs, +inf, -inf)
            for j in range(min(n, 60)):
                flat[b, p[j], :] = q[j % 4]
        else:                            # most locations NaN: the top-k boundary falls among NaNs
            flat[b, p[: (3 * n) // 4], rng.integers(0, C)] = np.where(rng.random((3 * n) // 4) < 0.5, np.nan, -np.nan)
    # -NaN with a sign bit: make sure both signs really are there
    if mode != "single":
        assert (np.signbit(flat) & np.isnan(flat)).any()
    return x


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", DTYPES, ids=["f32", "bf16", "f16"])
@pytest.mark.parametrize("mode", ["single", "all", "many"])
def test_nonfinite_logits_rank_like_the_reference(dm, dtype, mode, monkeypatch):
    """NaN ranks first, equal scores (NaN included, whatever its sign) by ascending location; torch's own
    select_and_decode selects the same set."""
    from s2anet_b200.decode import select_and_decode_torch
    rng = np.random.default_rng(DTYPES.index(dtype) * 10 + len(mode))
    sizes = [(40, 50), (23, 87), (5, 7)]
    lv, _, reg, anc = _select_inputs(dtype, "padded", sizes, 15, 2, rng)
    lv = [(_nonfinite_logits(dtype, 2, 15, H, W, rng, mode), d, a) for (H, W), (_, d, a) in zip(sizes, lv)]
    nchw = lambda x: torch.from_numpy(np.ascontiguousarray(np.transpose(x, (0, 3, 1, 2))))      # noqa: E731
    for layout in ("padded", "nchw"):
        cls = [_place(nchw(c), layout, dtype, 30.0) for c, _, _ in lv]
        for topk in (300, 1):
            monkeypatch.delenv("S2A_DEC_DEBUG", raising=False)
            _, _, idx = check_select_exact(dm, dtype, lv, cls, reg, anc, topk)
            monkeypatch.setenv("S2A_DEC_DEBUG", "2")
            check_select_exact(dm, dtype, lv, cls, reg, anc, topk)
            # the reference selects the same set per level (torch.topk leaves the order among NaNs open)
            off = 0
            for l, (c, r, a) in enumerate(zip(cls, reg, anc)):
                H, W = c.shape[2:]
                n = H * W
                k = min(n, topk)
                if n > k:
                    sc = c.permute(0, 2, 3, 1).reshape(2, n, 15).sigmoid()
                    ti = sc.max(dim=2)[0].topk(k, dim=1)[1].cpu().numpy()
                    for b in range(2):
                        assert set(ti[b].tolist()) == set(idx[b, off:off + k].tolist()), "level %d image %d" % (l, b)
                off += k
            tb, ts = select_and_decode_torch(cls, reg, anc, topk)     # the reference's ops run on NaN without error
            assert tb.shape[1] == off


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float16], ids=["bf16", "f16"])
def test_detection_with_nonfinite_logits_equals_the_oracle(oracle, dm, dtype):
    """The head's post-processing on its own outputs with NaN, +inf and -inf logits poked into the classification maps
    (one class, all classes, both NaN signs): the selection ranks them first and the multiclass NMS equals the
    oracle's on the model's boxes and scores."""
    from bench import CALIBRATED_BIAS, build_head, make_feats
    head = build_head(torch, torch.device(DEV), dtype, seed=0, bias=CALIBRATED_BIAS[3000])
    feats = make_feats(torch, 2, 4, torch.device(DEV), dtype)
    head.calibrate_scores(feats, 3000)
    with torch.no_grad():
        outs = head.forward_levels(feats)
    rng = np.random.default_rng(3)
    q = torch.tensor([float("nan"), float("inf"), float("-inf"), -float("nan")], dtype=dtype, device=DEV)
    for l in (0, 2, 4):
        c = outs[l][2]
        B, C, H, W = c.shape
        for b in range(B):
            for j, p in enumerate(rng.permutation(H * W)[:40]):
                y, x = divmod(int(p), W)
                if j % 2:
                    c[b, :, y, x] = q[j % 4]
                else:
                    c[b, int(rng.integers(0, C)), y, x] = q[j % 4]
    dets, labels, counts = head.detect_from_outs(outs)
    lv = [(o[2].permute(0, 2, 3, 1).float().cpu().numpy(), o[3].permute(0, 2, 3, 1).float().cpu().numpy(),
           o[5].reshape(o[2].size(0), o[2].size(2), o[2].size(3), 5).cpu().numpy()) for o in outs]
    bb, sc, _ = check_select_exact(dm, dtype, lv, [o[2] for o in outs], [o[3] for o in outs], [o[5] for o in outs],
                                   head.max_before_nms_per_level)
    for b in range(bb.shape[0]):
        rd, rl = oracle.multiclass_nms_rotated(bb[b], sc[b], head.score_thres_before_nms, head.iou_thres_nms,
                                               head.max_per_img)
        k = int(counts[b])
        assert k == rd.shape[0] and k > 0
        assert np.array_equal(bits(dets[b, :k].cpu().numpy()), bits(rd))
        assert np.array_equal(labels[b, :k].cpu().numpy(), rl)
