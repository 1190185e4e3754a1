"""Host-side caller of the hot path: the S2ANet FAM/ODM head + rotated post-processing, batched.

This is the code that sits directly above the custom ops in the reference (models/head.py:56-348
forward / forward_single, :648-725 get_bboxes / get_bboxes_single_img; models/boxes.py:82-162
delta2bbox_rotated; models/anchors.py:75-126 gen_grid_anchors; utils/general.py:925-930
norm_angle).  It is NOT one of the ops: the convolution towers stay stock PyTorch/cuDNN.  It exists
so that `bench.py` can measure "head + NMS images/s" and so that a reference checkpoint
(`head.*` parameter names are identical) can be run on the B200 ops without the reference tree.

Differences from the reference caller, all outside the ops' numerics:
  * grid anchors are built on the device once per (level, size) and cached (the reference builds
    them on the CPU and copies them every forward, head.py:315-326);
  * decode / top-k / NMS are batched over images; NMS is the fused sync-free multiclass kernel;
  * in 16-bit mode the whole head runs channels_last so AlignConv/ORConv read and write NHWC
    without layout copies.
"""
import math

import torch
import torch.nn as nn

from . import decode
from .alignconv import AlignConv
from .decode import norm_angle, rboxes_decode_torch  # noqa: F401
from .nms_rotated import multiclass_nms_rotated_batched
from .orn import ORConv2d, RotationInvariantPooling


def rboxes_decode(anchors, deltas, wh_ratio_clip=16 / 1000):
    """models/boxes.py:82-162 in PyTorch (the reference's own formulation; CPU reference arm and tests)."""
    return rboxes_decode_torch(anchors, deltas, wh_ratio_clip)


# The 16-bit multi-level path: every conv is one persistent tcgen05 launch for all FPN levels (conv_tc).
def _tc_conv(xs, m, relu=False):
    from . import conv_tc
    return conv_tc.conv2d_forward_tc_multi(xs, m.weight, m.bias, relu=relu)


def _tc_tower(seq, xs):
    for block in seq:                       # nn.Sequential(Conv2d, ReLU): one launch per layer for all levels
        xs = _tc_conv(xs, block[0], relu=True)
    return xs


def _tc_pair(xs0, m0, xs1, m1, relu=False):      # two same-shaped convs in one launch (fills the CTA pairs better)
    from . import conv_tc
    return conv_tc.conv2d_forward_tc_pair(xs0, m0.weight, m0.bias, xs1, m1.weight, m1.bias, relu=relu)


def _tc_towers(seq0, xs0, seq1, xs1):
    """Two towers layer by layer; layers of the same shape class share a launch."""
    for b0, b1 in zip(seq0, seq1):
        xs0, xs1 = _tc_pair(xs0, b0[0], xs1, b1[0], relu=True)
    return xs0, xs1


class S2ANetHead(nn.Module):
    """Same sub-module / parameter names and constructor defaults as models/head.py:56-258."""

    def __init__(self, num_classes, in_channels=256, feat_channels=256, stacked_convs=2, with_orconv=True,
                 anchor_scales=(4,), anchor_ratios=(1.0,), anchor_angles=(0,), featmap_strides=(8, 16, 32, 64, 128),
                 score_thres_before_nms=0.05, iou_thres_nms=0.5, max_before_nms_per_level=2000, max_per_img=2000):
        super().__init__()
        assert len(anchor_scales) == len(anchor_ratios) == len(anchor_angles) == 1, "one anchor per location"
        self.num_classes = num_classes
        self.in_channels = in_channels
        self.feat_channels = feat_channels
        self.stacked_convs = stacked_convs
        self.with_orconv = with_orconv
        self.anchor_scale = float(anchor_scales[0])
        self.anchor_angle = float(anchor_angles[0])
        self.featmap_strides = list(featmap_strides)
        self.score_thres_before_nms = score_thres_before_nms
        self.iou_thres_nms = iou_thres_nms
        self.max_before_nms_per_level = max_before_nms_per_level
        self.max_per_img = max_per_img

        def tower(first_in):
            layers = []
            for i in range(stacked_convs):
                cin = first_in if i == 0 else feat_channels
                layers.append(nn.Sequential(nn.Conv2d(cin, feat_channels, 3, 1, 1, bias=True), nn.ReLU(inplace=True)))
            return nn.Sequential(*layers)

        self.fam_reg_ls = tower(in_channels)
        self.fam_cls_ls = tower(in_channels)
        self.fam_reg_head = nn.Conv2d(feat_channels, 5, 1, padding=0, bias=True)
        self.fam_cls_head = nn.Conv2d(feat_channels, num_classes, 1, padding=0, bias=True)
        self.align_conv = AlignConv(feat_channels, feat_channels, kernel_size=3)
        if with_orconv:
            self.or_conv = ORConv2d(feat_channels, feat_channels // 8, kernel_size=3, padding=1, arf_config=(1, 8))
            self.or_pool = RotationInvariantPooling(feat_channels, 8)
            self.or_conv.fuse_pool = True           # the pooling comes out of the ORConv epilogue
        else:
            self.or_conv = nn.Conv2d(feat_channels, feat_channels, 3, padding=1)
        self.odm_reg_ls = tower(feat_channels)
        self.odm_cls_ls = tower(feat_channels // 8 if with_orconv else feat_channels)
        self.odm_cls_head = nn.Conv2d(feat_channels, num_classes, 3, padding=1, bias=True)
        self.odm_reg_head = nn.Conv2d(feat_channels, 5, 3, padding=1, bias=True)
        self._anchor_cache = {}
        self.init_weights()

    def init_weights(self):
        """models/head.py:232-258: N(0, 0.01) everywhere, classification biases at prior 0.01."""
        bias_cls = float(-math.log((1 - 0.01) / 0.01))
        for m in self.modules():
            if type(m) is nn.Conv2d:
                nn.init.normal_(m.weight, 0, 0.01)
                nn.init.constant_(m.bias, 0)
        nn.init.constant_(self.fam_cls_head.bias, bias_cls)
        nn.init.constant_(self.odm_cls_head.bias, bias_cls)
        self.align_conv.init_weights()
        nn.init.normal_(self.or_conv.weight, 0, 0.01)
        if self.or_conv.bias is not None:
            nn.init.constant_(self.or_conv.bias, 0)

    @torch.no_grad()
    def init_synthetic(self, seed=0):
        """Benchmark initialisation (SURVEY section 7 "benchmark realism"): with the reference's
        N(0, 0.01) init every score is ~0.01 < 0.05 and every refined anchor equals its grid anchor, so
        NMS is never reached and the gather is perfectly regular.  Here the towers get a
        variance-preserving init and the two heads are scaled so refined anchors are rotated /
        stretched like DOTA objects and class logits have spread; `calibrate_scores` then shifts the
        classification bias to a target candidate count."""
        g = torch.Generator().manual_seed(seed)
        for m in self.modules():
            if type(m) is nn.Conv2d:
                fan_in = m.weight[0].numel()
                m.weight.copy_(torch.randn(m.weight.shape, generator=g) * math.sqrt(2.0 / fan_in))
                m.bias.zero_()
        self.align_conv.deform_conv.weight.copy_(
            torch.randn(self.align_conv.deform_conv.weight.shape, generator=g) * math.sqrt(2.0 / (9 * self.feat_channels)))
        self.or_conv.weight.copy_(torch.randn(self.or_conv.weight.shape, generator=g) * math.sqrt(2.0 / (9 * self.feat_channels)))
        # deltas ~ (0.25, 0.25, 0.5, 0.5, 0.3): shifts of a quarter box, sizes x/ e^0.5, angles +-0.3*pi
        scale = torch.tensor([0.25, 0.25, 0.5, 0.5, 0.3]).view(5, 1, 1, 1)
        for head in (self.fam_reg_head, self.odm_reg_head):
            head.weight.mul_(scale / head.weight.flatten(1).norm(dim=1).view(5, 1, 1, 1).clamp_min(1e-6) * 0.7)
        self.odm_cls_head.weight.mul_(1.5 / self.odm_cls_head.weight.flatten(1).norm(dim=1).view(-1, 1, 1, 1) * 0.7)
        self.odm_cls_head.bias.fill_(-5.0)

    # ---- anchors ------------------------------------------------------------------------------
    def grid_anchors(self, H, W, stride, device):
        """models/anchors.py:75-126 for one square anchor per location: [H*W, 5] fp32 on `device`."""
        key = (H, W, stride, str(device))
        a = self._anchor_cache.get(key)
        if a is None:
            xs = torch.arange(W, dtype=torch.float32, device=device) * stride + 0.5 * (stride - 1)
            ys = torch.arange(H, dtype=torch.float32, device=device) * stride + 0.5 * (stride - 1)
            a = torch.zeros((H, W, 5), dtype=torch.float32, device=device)
            a[..., 0] = xs[None, :]
            a[..., 1] = ys[:, None]
            a[..., 2] = self.anchor_scale * stride
            a[..., 3] = self.anchor_scale * stride
            a[..., 4] = self.anchor_angle
            a = a.reshape(-1, 5)
            self._anchor_cache[key] = a
        return a

    # ---- forward ------------------------------------------------------------------------------
    @staticmethod
    def _tower(seq, x):
        """A conv+ReLU tower.  Stock PyTorch either way: on CUDA the fused cuDNN conv+bias+ReLU op is
        used (one kernel per layer instead of conv, bias-add and clamp)."""
        for block in seq:
            conv = block[0]
            if x.is_cuda and not torch.is_grad_enabled() and hasattr(torch, "cudnn_convolution_relu"):
                x = torch.cudnn_convolution_relu(x, conv.weight, conv.bias, conv.stride, conv.padding, conv.dilation,
                                                 conv.groups)
            else:
                x = torch.relu(conv(x))
        return x

    def forward_single(self, x, stride):
        """models/head.py:296-348."""
        fam_cls_pred, fam_bbox_pred, init_anchors, refine = self._fam(x, stride)
        or_feat = self.or_conv(self.align_conv(x, refine, stride))
        odm_cls_feat = self.or_pool(or_feat) if self.with_orconv else or_feat
        odm_cls_pred, odm_bbox_pred = self._odm(or_feat, odm_cls_feat)
        return fam_cls_pred, fam_bbox_pred, odm_cls_pred, odm_bbox_pred, init_anchors, refine

    def _fam_preds(self, x):
        fam_bbox_pred = self.fam_reg_head(self._tower(self.fam_reg_ls, x))
        fam_cls_pred = self.fam_cls_head(self._tower(self.fam_cls_ls, x))
        return fam_cls_pred, fam_bbox_pred

    def _fam(self, x, stride):
        fam_cls_pred, fam_bbox_pred = self._fam_preds(x)
        B, _, H, W = fam_bbox_pred.shape
        init_anchors = self.grid_anchors(H, W, stride, x.device)
        if x.is_cuda:       # fused grid-anchor generation + decode (models/head.py:27-52, models/anchors.py:75-126)
            refine = decode.fam_decode([fam_bbox_pred], [stride], self.anchor_scale, self.anchor_angle, 1e-6)[0]
        else:
            deltas = fam_bbox_pred.detach().permute(0, 2, 3, 1).reshape(B, H * W, 5)
            refine = rboxes_decode(init_anchors[None], deltas, wh_ratio_clip=1e-6).reshape(B, H, W, 5)
        return fam_cls_pred, fam_bbox_pred, init_anchors, refine

    def _odm(self, or_feat, odm_cls_feat):
        odm_cls_pred = self.odm_cls_head(self._tower(self.odm_cls_ls, odm_cls_feat))
        odm_bbox_pred = self.odm_reg_head(self._tower(self.odm_reg_ls, or_feat))
        return odm_cls_pred, odm_bbox_pred

    def forward_levels(self, feats):
        """All levels.  In 16-bit mode every layer -- the stock conv towers and prediction convs as well as
        AlignConv and ORConv2d -- runs as ONE persistent multi-level tcgen05 launch (the reference loops over
        levels in Python, head.py:265, and its convs are cuDNN calls)."""
        x0 = feats[0]
        # the fused multi-level path builds no autograd graph: training (any gradient can flow) takes forward_single,
        # whose ops are the stock differentiable ones + the DeformConv / ARF autograd Functions
        needs_grad = torch.is_grad_enabled() and (any(f.requires_grad for f in feats) or
                                                  any(p.requires_grad for p in self.parameters()))
        if needs_grad or not (x0.is_cuda and x0.dtype in (torch.bfloat16, torch.float16) and self.with_orconv):
            return [self.forward_single(x, s) for x, s in zip(feats, self.featmap_strides)]
        feats = list(feats)
        if len(self.fam_reg_ls) == len(self.fam_cls_ls):
            reg_feat, cls_feat = _tc_towers(self.fam_reg_ls, feats, self.fam_cls_ls, feats)
            fam_reg, fam_cls = _tc_pair(reg_feat, self.fam_reg_head, cls_feat, self.fam_cls_head)
        else:
            fam_reg = _tc_conv(_tc_tower(self.fam_reg_ls, feats), self.fam_reg_head)
            fam_cls = _tc_conv(_tc_tower(self.fam_cls_ls, feats), self.fam_cls_head)
        refines = decode.fam_decode(fam_reg, self.featmap_strides, self.anchor_scale, self.anchor_angle, 1e-6)
        odm_cls, odm_reg = self._odm_levels(feats, refines)
        return [(fam_cls[l], fam_reg[l], odm_cls[l], odm_reg[l],
                 self.grid_anchors(x.size(2), x.size(3), s, x.device), refines[l])
                for l, (x, s) in enumerate(zip(feats, self.featmap_strides))]

    def _odm_levels(self, feats, refines):
        """AlignConv, ORConv and the ODM towers / heads of forward_levels' 16-bit path: (odm_cls, odm_reg) per level."""
        from . import conv_tc
        aligned = conv_tc.alignconv_forward_tc_multi(feats, refines, self.align_conv.deform_conv.weight,
                                                     self.featmap_strides)
        or_feats, pooled = conv_tc.orconv_forward_tc_multi(aligned, self.or_conv.weight, self.or_conv.indices,
                                                           self.or_conv.bias, with_pool=True)
        if len(self.odm_cls_ls) == len(self.odm_reg_ls):
            # (the first layers differ in C -- 32 pooled vs 256 channels -- and fall back to two launches inside pair())
            cls_feat, reg_feat = _tc_towers(self.odm_cls_ls, pooled, self.odm_reg_ls, or_feats)
            return _tc_pair(cls_feat, self.odm_cls_head, reg_feat, self.odm_reg_head)
        return (_tc_conv(_tc_tower(self.odm_cls_ls, pooled), self.odm_cls_head),
                _tc_conv(_tc_tower(self.odm_reg_ls, or_feats), self.odm_reg_head))

    def _forward_detect(self, feats):
        """What detection reads, per level: (None, None, odm_cls, odm_reg, None, refine), or None where forward_levels
        takes forward_single.  The FAM classification tower and head only feed the training loss, so they are not run:
        two of the step's nine 256 -> 256 3x3 convs.  The regression tower layers run as single-problem launches instead
        of paired with the classification ones, and the regression head decodes in its epilogue instead of storing deltas
        for a fam_decode launch; every value is computed as forward_levels computes it, so the detections are
        bit-identical to detect_from_outs(forward_levels(feats))."""
        x0 = feats[0]
        if torch.is_grad_enabled() or not (x0.is_cuda and x0.dtype in (torch.bfloat16, torch.float16) and self.with_orconv):
            return None
        from . import conv_tc
        feats = list(feats)
        # the regression head decodes its deltas into the refined anchors in its epilogue: bit for bit
        # decode.fam_decode of its stored output, one launch and no delta tensor
        refines = conv_tc.conv2d_forward_tc_fam_decode(_tc_tower(self.fam_reg_ls, feats), self.fam_reg_head,
                                                       self.featmap_strides, self.anchor_scale, self.anchor_angle, 1e-6)
        odm_cls, odm_reg = self._odm_levels(feats, refines)
        return [(None, None, odm_cls[l], odm_reg[l], None, refines[l]) for l in range(len(feats))]

    @torch.no_grad()
    def select_and_decode(self, outs):
        """models/head.py:684-717 batched over images: sigmoid, per-level top-k by best class score,
        concatenation, final decode.  Returns (bboxes [B,n,5] fp32, scores [B,n,C] fp32)."""
        if outs[0][2].is_cuda:      # one fused launch: sigmoid + per-level top-k + gather + decode
            return decode.select_decode([o[2] for o in outs], [o[3] for o in outs], [o[5] for o in outs],
                                        self.max_before_nms_per_level)
        scores_l, deltas_l, anchors_l = [], [], []
        k = self.max_before_nms_per_level
        for (_, _, cls, reg, _, refine) in outs:
            B, C, H, W = cls.shape
            sc = cls.permute(0, 2, 3, 1).reshape(B, H * W, C).sigmoid()
            dl = reg.permute(0, 2, 3, 1).reshape(B, H * W, 5)
            an = refine.reshape(B, H * W, 5)
            if k > 0 and H * W > k:
                _, idx = sc.max(dim=2)[0].topk(k, dim=1)
                sc = sc.gather(1, idx[..., None].expand(-1, -1, C))
                dl = dl.gather(1, idx[..., None].expand(-1, -1, 5))
                an = an.gather(1, idx[..., None].expand(-1, -1, 5))
            scores_l.append(sc.float())
            deltas_l.append(dl)
            anchors_l.append(an)
        scores = torch.cat(scores_l, 1)
        bboxes = rboxes_decode(torch.cat(anchors_l, 1), torch.cat(deltas_l, 1))
        return bboxes.contiguous(), scores.contiguous()

    @torch.no_grad()
    def detect_from_outs(self, outs):
        """Post-processing of per-level head outputs (the tuples forward_levels / forward_single return, or the
        reference head's `p` regrouped per level): decode + per-level top-k + multiclass NMS, batched, sync-free."""
        bboxes, scores = self.select_and_decode(outs)
        return multiclass_nms_rotated_batched(bboxes, scores, self.score_thres_before_nms, self.iou_thres_nms,
                                              self.max_per_img)

    @torch.no_grad()
    def detect_packed(self, feats, dests, slot0=0):
        """detect() with the detection exchange fused into the NMS finaliser: rows go straight into the packed
        [slots, max_per_img + 1, 8] buffers `dests` (tensors and / or NVLink peer pointers), image b at slot slot0 + b."""
        from .nms_rotated import multiclass_nms_rotated_packed
        bboxes, scores = self.select_and_decode(self._forward_detect(feats) or self.forward_levels(feats))
        multiclass_nms_rotated_packed(bboxes, scores, dests, slot0, self.score_thres_before_nms, self.iou_thres_nms,
                                      self.max_per_img, K=self.max_per_img)

    @torch.no_grad()
    def detect(self, feats):
        """Whole hot path for a batch: head towers + AlignConv + ORConv + decode + multiclass NMS.
        Sync-free; returns (dets [B,max_per_img,6], labels [B,max_per_img], counts [B] int32)."""
        return self.detect_from_outs(self._forward_detect(feats) or self.forward_levels(feats))

    @torch.no_grad()
    def get_bboxes(self, feats):
        """Reference-shaped result (models/head.py:648-682): list of (det_bboxes [k,6], det_labels [k])."""
        return self._as_list(*self.detect(feats))

    @torch.no_grad()
    def get_bboxes_from_outs(self, outs):
        """models/head.py:648-725 `get_bboxes(p)` on already computed head outputs."""
        return self._as_list(*self.detect_from_outs(outs))

    @staticmethod
    def _as_list(dets, labels, counts):
        res = []
        for i, k in enumerate(counts.tolist()):
            if k == 0:
                res.append((dets.new_zeros((0, 6)), dets.new_zeros((0, 1), dtype=torch.long)))
            else:
                res.append((dets[i, :k], labels[i, :k]))
        return res

    @torch.no_grad()
    def calibrate_scores(self, feats, target_candidates=3000):
        """Shift odm_cls_head.bias so that about `target_candidates` (box, class) scores per image
        exceed score_thres_before_nms after the per-level top-k.  Returns the achieved mean count."""
        outs = self.forward_levels(feats)
        thr_logit = math.log(self.score_thres_before_nms / (1 - self.score_thres_before_nms))
        for _ in range(6):
            _, scores = self.select_and_decode(outs)
            logits = torch.logit(scores.clamp(1e-7, 1 - 1e-7)).flatten(1)
            kth = logits.kthvalue(max(1, logits.size(1) - target_candidates), dim=1)[0].mean()
            shift = float(thr_logit - kth)
            if abs(shift) < 1e-3:
                break
            self.odm_cls_head.bias.add_(shift)
            outs = [(a, b, c + shift, d, e, f) for (a, b, c, d, e, f) in outs]
        _, scores = self.select_and_decode(outs)
        return float((scores > self.score_thres_before_nms).sum(dim=(1, 2)).float().mean())
