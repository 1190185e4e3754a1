"""Box-decode stages (SURVEY 8(f) rows 2-3): s2a_fam_decode / s2a_select_decode.

CPU part: the oracle's numpy restatement and the PyTorch formulation kept in s2anet_b200/decode.py
against golden vectors produced by the reference's own Python (tests/golden/make_golden_decode.py:
gen_grid_anchors, fam_bbox_decode, get_bboxes_single_img).
GPU part: the sm_100a kernels against the golden vectors, the oracle and the PyTorch formulation run
on the same GPU, at the full 1024^2 head sizes, in fp32 / bf16 / fp16 and both memory formats.

Tolerances: every decoded coordinate within 2e-6 * max(1, |value|) + 1e-6 of the witness (the only
freedom is the last bit of cosf/sinf/expf between libm implementations; an angle may differ by pi only across the
-pi/4 | 3pi/4 wrap point); sigmoid scores within 2e-7
for fp32 inputs and bit-exact after rounding through a 16-bit input dtype.
"""
import numpy as np
import pytest
import torch

STRIDES5 = (8, 16, 32, 64, 128)


def close(a, b, rel=2e-6, abs_=1e-6):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    same = a == b                                   # covers +-inf (fp16 exp overflow at the clamp limit)
    with np.errstate(invalid="ignore"):
        return np.all(same | (np.abs(a - b) <= rel * np.maximum(1.0, np.abs(b)) + abs_))


def angle_close(a, b, tol=2e-6):
    """Decoded angles lie in [-pi/4, 3pi/4).  A difference of pi is allowed only across the wrap point: one value within
    a few ulps of -pi/4 and the other within a few ulps of 3pi/4, where libm's last bit decides the side."""
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    d = np.abs(a - b)
    lo = lambda x: np.abs(x + np.pi / 4) <= 1e-6          # noqa: E731  (about 4 float ulps at 3pi/4)
    hi = lambda x: np.abs(x - 3 * np.pi / 4) <= 1e-6      # noqa: E731
    wrap = (lo(a) & hi(b)) | (hi(a) & lo(b))
    return np.all((d <= tol * 4) | (wrap & (np.abs(d - np.pi) <= tol * 4)))


def boxes_close(a, b):
    return close(a[..., :4], b[..., :4]) and angle_close(a[..., 4], b[..., 4])


# ------------------------------------------------------------------------------------------------
# CPU: oracle and torch formulation vs the reference's golden vectors
# ------------------------------------------------------------------------------------------------
def test_oracle_grid_anchors_and_fam_decode_match_reference(oracle, golden):
    g = golden("decode_small.npz")
    for l, ((H, W), s) in enumerate(zip(g["sizes"], g["strides"])):
        assert np.array_equal(oracle.grid_anchors(H, W, s).reshape(-1, 5), g["grid_anchors_%d" % l])
        r = oracle.fam_decode(g["fam_pred_%d" % l], s)
        assert boxes_close(r, g["refine_%d" % l])
        r16 = oracle.fam_decode(g["fam_pred_%d" % l].astype(np.float16), s)
        assert boxes_close(r16, g["refine_f16in_%d" % l])
    # the clamp at wh_ratio_clip=1e-6 was exercised: w = 32 * exp(13.8155)
    assert abs(g["refine_0"][0, 0, 0, 2] / (32.0 * np.exp(13.815510558)) - 1) < 1e-5


def _levels(g):
    n = len(g["strides"])
    return ([g["cls_%d" % l] for l in range(n)], [g["reg_%d" % l] for l in range(n)], [g["refine_%d" % l] for l in range(n)])


def test_oracle_select_decode_matches_reference(oracle, golden):
    g = golden("decode_small.npz")
    cls, reg, refine = _levels(g)
    bb, sc, _ = oracle.select_decode(cls, reg, refine, topk=int(g["topk"]))
    for b in range(bb.shape[0]):
        assert sc[b].shape == g["scores_%d" % b].shape
        assert np.abs(sc[b] - g["scores_%d" % b]).max() <= 2e-7       # same candidates in the same order
        assert boxes_close(bb[b], g["bboxes_%d" % b])
    # half-precision network outputs against fp32 anchors (val.py), no top-k level
    h = lambda xs: [x.astype(np.float16) for x in xs]          # noqa: E731
    bb, sc, _ = oracle.select_decode(h(cls), h(reg), refine, topk=0)
    for b in range(bb.shape[0]):
        assert np.abs(sc[b] - g["scores_f16in_%d" % b]).max() <= 1e-3 * 2 ** -10   # at most one fp16 ulp near 0
        assert boxes_close(bb[b], g["bboxes_f16in_%d" % b])


def test_torch_formulation_matches_reference(golden):
    from s2anet_b200.decode import select_and_decode_torch
    g = golden("decode_small.npz")
    cls, reg, refine = (list(map(torch.from_numpy, xs)) for xs in _levels(g))
    bb, sc = select_and_decode_torch(cls, reg, refine, topk=int(g["topk"]))
    for b in range(bb.shape[0]):
        # (torch's CPU sigmoid/exp take a vectorised or a scalar path depending on the memory layout: last-bit freedom)
        assert np.abs(sc[b].numpy() - g["scores_%d" % b]).max() <= 2e-7
        assert boxes_close(bb[b].numpy(), g["bboxes_%d" % b])


# ------------------------------------------------------------------------------------------------
# GPU
# ------------------------------------------------------------------------------------------------
DEV = "cuda:0"


@pytest.mark.gpu
def test_kernels_match_reference_golden(golden):
    from s2anet_b200.decode import fam_decode, select_decode
    g = golden("decode_small.npz")
    strides = [int(s) for s in g["strides"]]
    n = len(strides)
    fam = [torch.from_numpy(g["fam_pred_%d" % l]).to(DEV) for l in range(n)]
    refined = fam_decode(fam, strides)
    for l in range(n):
        assert boxes_close(refined[l].cpu().numpy(), g["refine_%d" % l])
    refined16 = fam_decode([f.half() for f in fam], strides)
    for l in range(n):
        assert boxes_close(refined16[l].cpu().numpy(), g["refine_f16in_%d" % l])
    cls, reg, refine = ([torch.from_numpy(x).to(DEV) for x in xs] for xs in _levels(g))
    bb, sc = select_decode(cls, reg, refine, topk=int(g["topk"]))
    for b in range(bb.size(0)):
        assert np.abs(sc[b].cpu().numpy() - g["scores_%d" % b]).max() <= 2e-7
        assert boxes_close(bb[b].cpu().numpy(), g["bboxes_%d" % b])
    bb, sc = select_decode([c.half() for c in cls], [r.half() for r in reg], refine, topk=0)
    for b in range(bb.size(0)):
        assert np.abs(sc[b].cpu().numpy() - g["scores_f16in_%d" % b]).max() <= 1e-3 * 2 ** -10
        assert boxes_close(bb[b].cpu().numpy(), g["bboxes_f16in_%d" % b])


def _head_outputs(B, img, dtype, channels_last, seed):
    g = torch.Generator().manual_seed(seed)
    fam, cls, reg = [], [], []
    scale = torch.tensor([0.3, 0.3, 0.6, 0.6, 0.4]).view(1, 5, 1, 1)
    for s in STRIDES5:
        h = img // s
        def mk(t):
            t = t.to(dtype).to(DEV)
            return t.contiguous(memory_format=torch.channels_last) if channels_last else t
        fam.append(mk(torch.randn(B, 5, h, h, generator=g) * scale))
        cls.append(mk(torch.randn(B, 15, h, h, generator=g) * 2.0 - 3.0))
        reg.append(mk(torch.randn(B, 5, h, h, generator=g) * scale))
    return fam, cls, reg


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16, torch.float16])
@pytest.mark.parametrize("channels_last", [False, True])
def test_full_size_against_torch_on_the_same_gpu(dtype, channels_last):
    """1024^2 head sizes (21,824 locations -> 5,344 candidates per image), batch 3."""
    from s2anet_b200.decode import fam_decode, rboxes_decode_torch, select_decode
    from s2anet_b200.head import S2ANetHead
    B, topk = 3, 2000
    fam, cls, reg = _head_outputs(B, 1024, dtype, channels_last, seed=11)
    head = S2ANetHead(15)
    refined = fam_decode(fam, STRIDES5)
    for f, r, s in zip(fam, refined, STRIDES5):
        H, W = f.shape[2:]
        anchors = head.grid_anchors(H, W, s, DEV)
        want = rboxes_decode_torch(anchors[None], f.permute(0, 2, 3, 1).reshape(B, H * W, 5), 1e-6).reshape(B, H, W, 5)
        assert want.dtype == torch.float32
        assert boxes_close(r.cpu().numpy(), want.cpu().numpy())
    bb, sc, idx = select_decode(cls, reg, refined, topk, return_index=True)
    assert bb.shape == (B, 5344, 5) and sc.shape == (B, 5344, 15)
    off = 0
    for c, r, a in zip(cls, reg, refined):
        H, W = c.shape[2:]
        n, k = H * W, min(H * W, topk)
        s_all = c.permute(0, 2, 3, 1).reshape(B, n, 15).sigmoid()                     # in `dtype`, like the reference
        b_all = rboxes_decode_torch(a.reshape(B, n, 5), r.permute(0, 2, 3, 1).reshape(B, n, 5))
        ii = idx[:, off:off + k].long()
        assert int(ii.min()) >= 0 and int(ii.max()) < n
        for b in range(B):
            assert ii[b].unique().numel() == k                                        # k distinct locations
        got_s = sc[:, off:off + k]
        want_s = s_all.gather(1, ii[..., None].expand(-1, -1, 15)).float()
        if dtype == torch.float32:
            assert float((got_s - want_s).abs().max()) <= 2e-7
        else:
            assert torch.equal(got_s, want_s)
        want_b = b_all.gather(1, ii[..., None].expand(-1, -1, 5))
        assert boxes_close(bb[:, off:off + k].cpu().numpy(), want_b.cpu().numpy())
        best = got_s.max(dim=2)[0]
        if n > k:
            # exactly the k best locations, in descending order, ties by ascending location
            topv = s_all.max(dim=2)[0].float().topk(k, dim=1)[0]
            if dtype == torch.float32:
                assert float((best - topv).abs().max()) <= 2e-7
            else:
                assert torch.equal(best, topv)
            d = best[:, 1:] - best[:, :-1]
            assert bool((d <= 0).all())
            tie = d == 0
            assert bool((ii[:, 1:][tie] > ii[:, :-1][tie]).all())
        else:
            assert torch.equal(ii, torch.arange(n, device=DEV)[None].expand(B, -1))
        off += k
    assert off == 5344


@pytest.mark.gpu
def test_oracle_agrees_on_a_midsize_case(oracle):
    from s2anet_b200.decode import fam_decode, select_decode
    fam, cls, reg = _head_outputs(2, 256, torch.float32, False, seed=5)
    refined = fam_decode(fam, STRIDES5)
    for f, r, s in zip(fam, refined, STRIDES5):
        assert boxes_close(r.cpu().numpy(), oracle.fam_decode(f.cpu().numpy(), s))
    bb, sc, idx = select_decode(cls, reg, refined, topk=300, return_index=True)
    ob, os_, oi = oracle.select_decode([c.cpu().numpy() for c in cls], [r.cpu().numpy() for r in reg],
                                       [r.cpu().numpy() for r in refined], topk=300)
    assert np.array_equal(idx.cpu().numpy(), oi)
    assert np.abs(sc.cpu().numpy() - os_).max() <= 2e-7
    assert boxes_close(bb.cpu().numpy(), ob)


@pytest.mark.gpu
def test_ties_and_degenerate_inputs():
    from s2anet_b200.decode import select_decode
    # all scores equal: the defined tie rule keeps the lowest locations, in order
    cls = [torch.zeros(1, 3, 64, 64, device=DEV)]
    reg = [torch.zeros(1, 5, 64, 64, device=DEV)]
    anc = [torch.rand(1, 64, 64, 5, device=DEV) + 1.0]
    bb, sc, idx = select_decode(cls, reg, anc, topk=100, return_index=True)
    assert torch.equal(idx[0], torch.arange(100, device=DEV, dtype=torch.int32))
    assert torch.equal(sc, torch.full_like(sc, 0.5))
    # zero deltas decode to the anchor itself (angle normalised)
    a = anc[0].reshape(1, -1, 5)[:, :100]
    assert float((bb[..., :4] - a[..., :4]).abs().max()) == 0.0
    # empty batch is a no-op
    e = select_decode([cls[0][:0]], [reg[0][:0]], [anc[0][:0]], topk=100)
    assert e[0].shape == (0, 100, 5)
    with pytest.raises(NotImplementedError):
        select_decode([cls[0].cpu()], [reg[0].cpu()], [anc[0].cpu()])
