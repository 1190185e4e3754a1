"""S2ANet.detect() runs only what detection reads: the FAM classification tower and head (they feed the training loss
alone) are not run.  The detections must stay bit-identical to those of the full forward pass."""
import pytest
import torch

DEV = "cuda:0"


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float16])
def test_detect_is_bit_identical_to_the_full_forward(dtype):
    from bench import CALIBRATED_BIAS, build_head, make_feats
    head = build_head(torch, torch.device(DEV), dtype, seed=0, bias=CALIBRATED_BIAS[3000])
    feats = make_feats(torch, 2, 4, torch.device(DEV), dtype)
    head.calibrate_scores(feats, 3000)
    with torch.no_grad():
        full = head.detect_from_outs(head.forward_levels(feats))
    fast = head.detect(feats)
    for a, b in zip(full, fast):
        assert torch.equal(a, b)
    assert int(fast[2].min()) > 0


def test_detect_branch_only_for_the_16bit_cuda_inference_path():
    from s2anet_b200.head import S2ANetHead
    head = S2ANetHead(15).eval()
    feats = [torch.zeros(1, 256, 8 // s, 8 // s) for s in (1, 2, 4, 8)]
    with torch.no_grad():
        assert head._forward_detect(feats) is None                        # CPU
        assert head._forward_detect([f.bfloat16() for f in feats]) is None
    assert head._forward_detect(feats) is None                            # grad enabled


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float16])
@pytest.mark.parametrize("shape", ["bench_b2", "odd_b1", "odd_b3"])
def test_fam_decode_epilogue_is_bit_identical_to_head_then_fam_decode(dtype, shape):
    from bench import build_head
    from s2anet_b200 import conv_tc, decode
    head = build_head(torch, torch.device(DEV), dtype, seed=0)
    strides = (8, 16, 32, 64, 128)
    if shape == "bench_b2":
        B, sizes = 2, [(1024 // s, 1024 // s) for s in strides]
    else:
        B, sizes = (1 if shape == "odd_b1" else 3), [(37, 53), (19, 27), (10, 14), (5, 7), (1, 1)]
    g = torch.Generator().manual_seed(11)
    feats = [torch.randn(B, 256, h, w, generator=g).to(dtype).to(DEV).contiguous(memory_format=torch.channels_last)
             for h, w in sizes]
    with torch.no_grad():
        xs = feats
        for block in head.fam_reg_ls:       # the head's real input: the ReLU'd regression tower output
            xs = conv_tc.conv2d_forward_tc_multi(xs, block[0].weight, block[0].bias, relu=True)
        deltas = conv_tc.conv2d_forward_tc_multi(xs, head.fam_reg_head.weight, head.fam_reg_head.bias)
        ref = decode.fam_decode(deltas, strides, head.anchor_scale, head.anchor_angle, 1e-6)
        out = conv_tc.conv2d_forward_tc_fam_decode(xs, head.fam_reg_head, strides, head.anchor_scale, head.anchor_angle, 1e-6)
    for a, b in zip(out, ref):
        assert a.shape == b.shape and torch.equal(a, b)


def test_fam_decode_argument_checks():
    import torch.nn as nn
    from s2anet_b200 import conv_tc
    x = [torch.zeros(1, 256, 8, 8, dtype=torch.bfloat16)]
    for bad in (nn.Conv2d(256, 15, 1), nn.Conv2d(256, 5, 3, padding=1), nn.Conv2d(256, 5, 1, bias=False),
                nn.Conv2d(256, 5, 1, stride=2)):
        with pytest.raises(ValueError):
            conv_tc.conv2d_forward_tc_fam_decode(x, bad, (8,), 4.0, 0.0)
    head = nn.Conv2d(256, 5, 1)
    with pytest.raises(ValueError):                              # input channels
        conv_tc.conv2d_forward_tc_fam_decode([torch.zeros(1, 128, 8, 8)], head, (8,), 4.0, 0.0)
    with pytest.raises(ValueError):                              # one stride per level
        conv_tc.conv2d_forward_tc_fam_decode(x, head, (8, 16), 4.0, 0.0)
    with pytest.raises(NotImplementedError):                     # CUDA only, no fallback
        conv_tc.conv2d_forward_tc_fam_decode(x, head, (8,), 4.0, 0.0)
