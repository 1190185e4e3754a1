#!/usr/bin/env python
"""bench.py -- S2ANet head + rotated NMS images/s at 1024x1024 on B200 (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W            # this repo's sm_100a path
    python bench.py --impl reference --gpus N --steps K --warmup W   # the reference's CPU path (rank 0 only)
    python bench.py --gpus N --steps K --warmup W --dump-outputs DIR  # + the last timed step's detections as DIR/*.npy

A "step" is one pass of the hot path over one batch of synthetic input: the FAM/ODM head (conv towers, AlignConv,
ORConv2d + RotationInvariantPooling -- every layer a kernel of this library) over the five FPN levels of `--batch`
1024x1024 images per GPU, box decode, per-level top-2000 and the fused 15-class rotated NMS, and -- with more than
one GPU -- the detection exchange fused into the NMS finaliser (NVLink peer stores + one barrier).  `value` times it
with the FPN features resident in HBM; `e2e` times the same call with the features in pinned host memory (H2D inside
the timed region, double-buffered on a copy stream) and the rank's own detections read back to the host.
Prints ONE JSON line on rank 0.  Extra keys next to the contract's: `iou` (BASELINE's second metric, rotated IoU
pairs/s on configs[3], with both collective forms), `configs` (the bench legs BASELINE.md section 3 lists: config 1,
config 2 at batch 1, config 3 at batch 1, NMS at N = 2,000 / 20,000, the step at 10 k candidates), `parity` (measured
max-abs / rel-L2 of the 16-bit kernels against the reference CUDA ops).
"""
import argparse
import json
import math
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "S2ANet head+NMS images/s at 1024^2"
UNIT = "images/s"
IMG = 1024
STRIDES = (8, 16, 32, 64, 128)
NUM_CLASSES = 15
POSITIONS = sum((IMG // s) ** 2 for s in STRIDES)            # 21,824
ALIGN_FLOPS_PER_IMAGE = 2.0 * POSITIONS * 256 * 2304          # SURVEY 8d: 25.744 GFLOP
IOU_FLOP_PER_PAIR = 350.0                                      # SURVEY 8d counting convention
# odm_cls_head.bias after `calibrate_scores` on the seeded bench inputs (seed 0 weights, feature seed 4): the value
# every arm starts from, so that the CPU reference arm does not depend on a previous GPU run (round 1: it read a
# scratch file and ran 6.6x slower when the file was missing -- more candidates, quadratic CPU NMS)
CALIBRATED_BIAS = {3000: -6.21875}


def host_cores():
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            p = json.load(f)
        return {"bf16_burst": p.get("bf16_tflops"), "bf16_sustained": p.get("bf16_tflops_sustained"),
                "hbm": p.get("hbm_gbs"), "source": "MEASURED_PEAKS.json"}
    return {"bf16_burst": 1590.0, "bf16_sustained": 1400.0, "hbm": 6650.0, "source": "fallback (B200_PROFILING.md)"}


def load_json(rel):
    path = os.path.join(ROOT, rel)
    if not os.path.exists(path):
        return None
    with open(path) as f:
        return json.load(f)


def load_traffic(batch):
    """DRAM bytes per launch of the roofline kernel from the committed `ncu --set full` capture
    (profiles/roofline_traffic.json; captured at batch 8, the default): read + write, or None."""
    t = (load_json("profiles/roofline_traffic.json") or {}).get("conv_tc_kernel<ALIGN,bf16>")
    if batch != 8 or not t:
        return None
    return {"dram_bytes": t["dram_bytes_read"] + t["dram_bytes_write"], "algorithmic_bytes": t["algorithmic_bytes"],
            "source": t["source"]}


def load_parity():
    """Measured errors of the 16-bit kernels against the reference CUDA ops (tests/test_gpu_conv_tc_vs_reference.py on
    B200, committed as profiles/r2_parity_errors.json)."""
    d = load_json("profiles/r2_parity_errors.json")
    if not d:
        return None
    r = d["results"]

    def pick(k):
        return None if k not in r else {"max_abs_over_ref_max": r[k]["max_abs_rel"], "rel_l2": r[k]["rel_l2"]}
    return {"source": "profiles/r2_parity_errors.json (tests/test_gpu_conv_tc_vs_reference.py, %s)" % d.get("gpu"),
            "alignconv_bf16_P3_vs_reference_cuda_fp32": pick("alignconv_bf16_P3_vs_reference_cuda_fp32"),
            "alignconv_fp16_P3_vs_reference_cuda_fp32": pick("alignconv_fp16_P3_vs_reference_cuda_fp32"),
            "reference_cuda_fp16_P3_vs_its_own_fp32": pick("reference_cuda_fp16_P3_vs_reference_cuda_fp32"),
            "deform_conv_forward_cuda_fp16_vs_reference_cuda_fp16": pick("deform_conv_forward_cuda_fp16_L0_vs_reference_cuda_fp16"),
            "orconv_bf16_P3_vs_reference_arf_conv2d_fp32": pick("orconv_bf16_P3_vs_reference_arf_plus_conv2d_fp32")}


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self._halt = index, [], threading.Event()

    def run(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        while not self._halt.is_set():
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q,
                                      "--format=csv,noheader,nounits"], stdout=subprocess.PIPE, text=True, timeout=5).stdout
                self.rows.append([c.strip() for c in out.strip().split(",")])
            except Exception:
                pass
            self._halt.wait(0.02)

    def stop(self):
        self._halt.set()
        self.join(2)
        sm = sorted(int(r[0]) for r in self.rows if r and r[0].isdigit())
        mx = [int(r[1]) for r in self.rows if len(r) > 1 and r[1].isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({n for r in self.rows if len(r) >= 6 for n, v in zip(names, r[2:6]) if v.lower().startswith("active")})
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(self.rows)}


def make_feats(torch, batch, seed, device, dtype, pinned=False):
    g = torch.Generator().manual_seed(seed)
    feats = []
    for s in STRIDES:
        h = IMG // s
        t = torch.randn(batch, 256, h, h, generator=g).to(dtype).contiguous(memory_format=torch.channels_last)
        if pinned:
            t = t.pin_memory()
        else:
            t = t.to(device)
        feats.append(t)
    return feats


# ------------------------------------------------------------------------------------------------
# CPU reference path (the reference's own CPU kernels where it has them; see BASELINE.md section 3)
# ------------------------------------------------------------------------------------------------
class CpuReferenceHead:
    """Head + NMS on the host: stock torch CPU convs, AlignConv = the reference's get_offset formula +
    torchvision.ops.deform_conv2d (the reference has no CPU deform conv, deform_conv.py:58-59),
    ORConv2d = ARF index scatter + F.conv2d, RotationInvariantPooling, decode, and ml_nms_rotated
    through the reference's CPU extension (oracle/_ref/ext_cpu, kind "reference") or, where that
    was not prebuilt, the oracle port (kind "port")."""

    def __init__(self, head):
        import torch
        from oracle import build_oracle
        from oracle import oracle as O
        self.torch, self.O = torch, O
        self.head = head
        self.sd = {k: v.detach().float().cpu() for k, v in head.state_dict().items()}
        self.ml_ext = build_oracle.load_ref_extension("ml_nms_rotated_cuda", "cpu")
        self.kind = "reference" if self.ml_ext is not None else "port"
        w = self.sd["or_conv.weight"]
        self.w_rot = torch.from_numpy(O.arf_forward(w.numpy(), self.sd["or_conv.indices"].numpy()))

    def tower(self, x, name, n):
        F = self.torch.nn.functional
        for i in range(n):
            x = F.relu(F.conv2d(x, self.sd["%s.%d.0.weight" % (name, i)], self.sd["%s.%d.0.bias" % (name, i)], padding=1))
        return x

    def level(self, x, stride):
        import torchvision
        torch, F, h = self.torch, self.torch.nn.functional, self.head
        fam_reg = F.conv2d(self.tower(x, "fam_reg_ls", 2), self.sd["fam_reg_head.weight"], self.sd["fam_reg_head.bias"])
        _ = F.conv2d(self.tower(x, "fam_cls_ls", 2), self.sd["fam_cls_head.weight"], self.sd["fam_cls_head.bias"])
        B, _, H, W = fam_reg.shape
        from s2anet_b200.head import rboxes_decode
        anchors = h.grid_anchors(H, W, stride, "cpu")
        refine = rboxes_decode(anchors[None], fam_reg.permute(0, 2, 3, 1).reshape(B, H * W, 5), wh_ratio_clip=1e-6)
        offs = torch.stack([h.align_conv.get_offset(refine[i], (H, W), stride) for i in range(B)])
        al = F.relu(torchvision.ops.deform_conv2d(x, offs, self.sd["align_conv.deform_conv.weight"], padding=1))
        orf = F.conv2d(al, self.w_rot, self.sd["or_conv.bias"], padding=1)
        pooled = orf.view(B, -1, 8, H, W).max(dim=2)[0]
        cls = F.conv2d(self.tower(pooled, "odm_cls_ls", 2), self.sd["odm_cls_head.weight"], self.sd["odm_cls_head.bias"], padding=1)
        reg = F.conv2d(self.tower(orf, "odm_reg_ls", 2), self.sd["odm_reg_head.weight"], self.sd["odm_reg_head.bias"], padding=1)
        return (None, fam_reg, cls, reg, anchors, refine.reshape(B, H, W, 5))

    def detect(self, feats):
        torch = self.torch
        outs = [self.level(x, s) for x, s in zip(feats, STRIDES)]
        bboxes, scores = self.head.select_and_decode(outs)
        results = []
        for b in range(bboxes.size(0)):
            if self.ml_ext is not None:
                mask = scores[b] > self.head.score_thres_before_nms
                bx = bboxes[b][:, None].expand(-1, scores.size(2), 5)[mask]
                sc = scores[b][mask]
                lb = mask.nonzero(as_tuple=False)[:, 1].to(bx)
                if bx.shape[0] == 0:
                    results.append((bx.new_zeros((0, 6)), lb))
                    continue
                keep = self.ml_ext.ml_nms_rotated(bx.contiguous(), sc.contiguous(), lb.contiguous(), self.head.iou_thres_nms)
                keep = keep[: self.head.max_per_img]
                results.append((torch.cat([bx[keep], sc[keep, None]], 1), lb[keep]))
            else:
                d, l = self.O.multiclass_nms_rotated(bboxes[b].numpy(), scores[b].numpy(), self.head.score_thres_before_nms,
                                                     self.head.iou_thres_nms, self.head.max_per_img)
                results.append((torch.from_numpy(d), torch.from_numpy(l)))
        return results


def build_head(torch, device, dtype, seed=0, bias=None):
    from s2anet_b200.head import S2ANetHead
    head = S2ANetHead(NUM_CLASSES)
    head.init_synthetic(seed)
    if bias is not None:
        with torch.no_grad():
            head.odm_cls_head.bias.fill_(bias)
    head = head.eval()
    if device is not None:
        head = head.to(device)
    if dtype is not None and dtype != torch.float32:
        head = head.to(dtype)
    for m in head.modules():                      # channels_last for the stock 4-D conv weights only
        if type(m) is torch.nn.Conv2d:
            m.weight.data = m.weight.data.contiguous(memory_format=torch.channels_last)
    return head


def pin_cpu_threads():
    """Same thread count whatever launched us (torchrun exports OMP_NUM_THREADS=1 to its workers, a bare `python`
    does not): all the cores this process may run on."""
    n = host_cores()
    for k in ("OMP_NUM_THREADS", "MKL_NUM_THREADS"):
        os.environ[k] = str(n)
    return n


def run_reference(args, rank, world):
    """Reference arm: the CPU path, rank 0 only, a bounded sample (1 image per step).  Self-contained: the
    classification bias is the committed calibration, the inputs are seeded, the thread count is pinned."""
    if rank != 0:
        return
    ncores = pin_cpu_threads()
    import torch
    torch.set_num_threads(ncores)
    head = build_head(torch, None, torch.float32, seed=0, bias=CALIBRATED_BIAS[3000])
    ref = CpuReferenceHead(head)
    feats = make_feats(torch, 1, 4, "cpu", torch.float32)
    feats = [f.contiguous() for f in feats]
    for _ in range(args.warmup):
        res = ref.detect(feats)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        res = ref.detect(feats)
    dt = time.perf_counter() - t0
    value = args.steps / dt
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": dt / max(1, args.steps) * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic", "impl": "reference",
        "config": {"workload": "S2ANet R-50-FPN head + 15-class rotated NMS, 1024x1024 (CPU reference path)",
                   "batch_per_step": 1, "detections_img0": int(res[0][0].shape[0]),
                   "odm_cls_bias": CALIBRATED_BIAS[3000]},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": torch.get_num_threads(), "kind": ref.kind,
                         "sample": "1 image per step, all 5 FPN levels, torch CPU convs + torchvision deform_conv2d "
                                   "(all threads) + reference ml_nms_rotated CPU kernel (1 thread)"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))


def cuda_time(torch, fn, reps, warm=3):
    """Average ms of fn() over `reps` calls, CUDA events on the current stream."""
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps


DUMP_MAX_BYTES = 64 << 20


def dump_outputs(path, dets, labels, counts, odm_cls_bias):
    """Write what one step returned to its caller as path/<name>.npy, so that two builds run with the same arguments
    (hence the same seeded inputs) can be compared output for output: dets [n,K,6] and labels [n,K] float32, counts [n]
    float64, rows at or past an image's count zeroed (the NMS leaves them unspecified).  n is every image of the step,
    or a fixed seeded sample of them where all would exceed DUMP_MAX_BYTES; image_index [n] float64 names them.
    odm_cls_bias [C] float64 is the classification bias the step ran with: calibrate_scores sets it from this build's
    own forward pass, so outputs of two builds are comparable as they stand only where their biases are equal."""
    import numpy as np
    bias = odm_cls_bias.detach().double().cpu().numpy()
    dets, labels = dets.float().cpu().numpy(), labels.float().cpu().numpy()
    counts = counts.cpu().numpy().astype(np.float64)
    n, K = labels.shape
    keep = np.arange(n)
    per_image = dets[0].nbytes + labels[0].nbytes + 16
    budget = DUMP_MAX_BYTES - bias.nbytes
    if n * per_image > budget:
        keep = np.sort(np.random.default_rng(0).choice(n, budget // per_image, replace=False))
    dets, labels, counts = dets[keep], labels[keep], counts[keep]
    unused = np.arange(K)[None, :] >= counts[:, None]
    dets[unused] = 0
    labels[unused] = 0
    os.makedirs(path, exist_ok=True)
    for name, a in (("dets", dets), ("labels", labels), ("counts", counts), ("image_index", keep.astype(np.float64)),
                    ("odm_cls_bias", bias)):
        np.save(os.path.join(path, name + ".npy"), a)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=8, help="images per GPU per step")
    ap.add_argument("--dtype", default="bf16", choices=["bf16", "fp16", "fp32"])
    ap.add_argument("--candidates", type=int, default=3000, help="target (box, class) candidates per image")
    ap.add_argument("--exchange", default="push", choices=["push", "nccl"],
                    help="detection exchange at N > 1: NVLink peer stores fused into the NMS finaliser, or NCCL all-gather")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip the extra bench legs (configs 1-3, NMS sizes, 10k candidates)")
    ap.add_argument("--no-graph", action="store_true", help="launch eagerly instead of replaying CUDA graphs")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the detections of the last timed step to DIR/<name>.npy (see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs applies to --impl b200")
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        return run_reference(args, rank, world)

    if world == 1:
        pin_cpu_threads()
    import numpy as np
    import torch
    import torch.distributed as dist
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; this repository has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    torch.backends.cudnn.benchmark = True
    from s2anet_b200 import _lib
    from s2anet_b200 import dist as sdist
    from s2anet_b200.alignconv import alignconv_forward
    dtype = {"bf16": torch.bfloat16, "fp16": torch.float16, "fp32": torch.float32}[args.dtype]
    B = args.batch
    head = build_head(torch, dev, dtype, seed=0, bias=CALIBRATED_BIAS.get(args.candidates))
    K = head.max_per_img
    # two rotating input sets (> L2 together with the ~GBs of activations each step writes)
    feat_sets = [make_feats(torch, B, 4 + rank + 100 * i, dev, dtype) for i in range(2)]
    ncand = head.calibrate_scores(feat_sets[0], args.candidates)
    calibrated_bias = float(head.odm_cls_head.bias.detach().float().mean())

    # ---- detection exchange (N > 1) -------------------------------------------------------------------------
    exch, exch_mode, exch_note = None, "none", None
    if world > 1:
        exch_mode = args.exchange
        if exch_mode == "push":
            try:
                exch = sdist.DetectionExchange(B, K, dev, nbuf=2)
            except Exception as e:                   # symmetric memory not available on this box: say so, use NCCL
                exch_mode, exch_note = "nccl", "symmetric memory unavailable (%s)" % (str(e).splitlines()[0][:120],)
        ok = torch.tensor([1 if exch_mode == "push" else 0], device=dev)
        dist.all_reduce(ok, op=dist.ReduceOp.MIN)
        if int(ok.item()) == 0:
            exch_mode, exch = "nccl", None
    send_bufs = [torch.zeros((B, K + 1, 8), dtype=torch.float32, device=dev) for _ in range(2)]
    recv_bufs = [torch.zeros((world * B, K + 1, 8), dtype=torch.float32, device=dev) for _ in range(2)] if world > 1 else None

    graphs = {}
    in_graph = {"barrier": True, "allgather": True}

    def run_head(feats, i):
        """The capturable part of a step for buffer set i; returns the packed buffer holding the result."""
        if world == 1:
            return head.detect(feats)
        if exch_mode == "push":
            ptrs, slot0 = exch.targets(i)
            head.detect_packed(feats, ptrs, slot0)
            if in_graph["barrier"]:
                exch.handles[i].barrier(channel=0)
            return exch.bufs[i]
        head.detect_packed(feats, [send_bufs[i]], 0)
        if in_graph["allgather"]:
            dist.all_gather_into_tensor(recv_bufs[i], send_bufs[i])
        return recv_bufs[i]

    def capture(feats, i):
        for _ in range(2):                   # warm every lazy path (weight packing, workspace allocation)
            run_head(feats, i)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        g = torch.cuda.CUDAGraph()
        before = _lib.launches
        with torch.cuda.graph(g):
            out_ = run_head(feats, i)
        return g, out_, _lib.launches - before

    def step(feats, i):
        """One pass of the hot path.  The sync-free head + NMS (+ exchange) is captured once per buffer set into a
        CUDA graph and replayed."""
        if args.no_graph:
            out_ = run_head(feats, i)
        else:
            if i not in graphs or graphs[i][3] is not feats:
                ok = 1
                try:
                    g, out_, n_mine = capture(feats, i)
                except Exception:
                    ok = 0
                if world > 1:                        # every rank takes the same decision
                    flag = torch.tensor([ok], device=dev)
                    torch.cuda.synchronize()
                    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
                    ok = int(flag.item())
                if not ok:
                    # the collective / barrier refused stream capture somewhere: keep it outside the graph everywhere
                    torch.cuda.synchronize()
                    in_graph["barrier"] = in_graph["allgather"] = False
                    g, out_, n_mine = capture(feats, i)
                graphs[i] = (g, out_, n_mine, feats)
            g, out_, n_mine, _ = graphs[i]
            g.replay()
            _lib.launches += n_mine
        if world > 1:
            if exch_mode == "push" and not in_graph["barrier"]:
                exch.handles[i].barrier(channel=0)
            elif exch_mode == "nccl" and not in_graph["allgather"]:
                dist.all_gather_into_tensor(recv_bufs[i], send_bufs[i])
            return sdist.packed_views(out_, K)
        return out_

    def sync_all():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed_steps(nsteps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        sync_all()
        e0.record()
        for i in range(nsteps):
            out_ = step(feat_sets[i % 2], i % 2)
        e1.record()
        sync_all()
        t = torch.tensor([e0.elapsed_time(e1)], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item()), out_

    for i in range(args.warmup):
        out = step(feat_sets[i % 2], i % 2)
    sync_all()
    sampler = ClockSampler(local_rank)
    sampler.start()
    l0 = _lib.launches
    ms, out = timed_steps(args.steps)
    launches = _lib.launches - l0
    clocks = sampler.stop()
    if args.dump_outputs and rank == 0:              # before the legs below replay the graphs into the same buffers
        dump_outputs(args.dump_outputs, *out, head.odm_cls_head.bias)
    value = world * B * args.steps / (ms / 1e3)
    own = slice(rank * B, (rank + 1) * B) if world > 1 else slice(0, B)
    ndet = int(out[2][own].float().mean().item())
    exchange = None
    rank_ms = None
    if world > 1:
        # the residual of the scaling curve, named: every rank's own step WITHOUT the exchange (same graph-replayed head +
        # NMS, no peer stores, no barrier).  The exchanged step runs at the pace of the slowest GPU of the box (each step
        # ends with all ranks' detections on every rank), so max(rank_ms) is its floor whatever the exchange costs.
        for _ in range(2):
            head.detect(feat_sets[0])
        torch.cuda.synchronize()
        g_local = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g_local):
            head.detect(feat_sets[0])
        sync_all()
        mine_ms = torch.tensor([cuda_time(torch, g_local.replay, min(args.steps, 50))], device=dev, dtype=torch.float64)
        all_ms = [torch.zeros_like(mine_ms) for _ in range(world)]
        dist.all_gather(all_ms, mine_ms)
        rank_ms = [float(t_.item()) for t_ in all_ms]
        del g_local
    if world > 1:
        # every rank's images must have arrived on every rank: image counts of all slots are plausible
        assert int((out[2] >= 0).sum().item()) == world * B
        exchange = {"mode": exch_mode, "inside_cuda_graph": in_graph["barrier"] if exch_mode == "push" else in_graph["allgather"],
                    "bytes_per_rank_per_step": B * (K + 1) * 8 * 4, "note": exch_note,
                    "ms_per_step_without_exchange_by_rank": rank_ms,
                    "exchange_cost_ms": ms / args.steps - max(rank_ms),
                    "what": "push: mc_emit_kernel stores each kept detection into the packed buffer of every rank over NVLink "
                            "peer pointers (torch symmetric memory) + one signal-pad barrier; nccl: the same kernel packs "
                            "locally, then all_gather_into_tensor"}

    # ---- e2e: host (pinned) features in, the rank's OWN detections back on the host, copies inside the timed region
    host_sets = [make_feats(torch, B, 4 + rank + 100 * i, dev, dtype, pinned=True) for i in range(2)]
    copy_stream = torch.cuda.Stream(device=dev)
    h2d_bytes = sum(t_.numel() * t_.element_size() for t_ in host_sets[0])
    host_out = (torch.empty((B, K, 6), dtype=torch.float32).pin_memory(), torch.empty((B, K), dtype=torch.float32).pin_memory(),
                torch.empty((B,), dtype=torch.int32).pin_memory())
    d2h_bytes = sum(t_.numel() * t_.element_size() for t_ in host_out)
    dev_bufs = [[torch.empty_like(f, device=dev) for f in host_sets[0]] for _ in range(2)]
    ready = [torch.cuda.Event() for _ in range(2)]
    freed = [torch.cuda.Event() for _ in range(2)]

    def upload(i):
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(freed[i % 2])
            for d, h in zip(dev_bufs[i % 2], host_sets[i % 2]):
                d.copy_(h, non_blocking=True)
            ready[i % 2].record(copy_stream)

    def e2e_loop(n):
        cur = torch.cuda.current_stream(dev)
        for j in range(2):
            freed[j].record(cur)
        upload(0)
        for i in range(n):
            if i + 1 < n:
                upload(i + 1)
            cur.wait_event(ready[i % 2])
            dets, labels, counts = step(dev_bufs[i % 2], i % 2)
            freed[i % 2].record(cur)
            host_out[0].copy_(dets[own], non_blocking=True)
            host_out[1].copy_(labels[own], non_blocking=True)
            host_out[2].copy_(counts[own], non_blocking=True)
        cur.synchronize()

    e2e_loop(min(3, args.warmup))
    sync_all()
    t0 = time.perf_counter()
    e2e_loop(args.steps)
    sync_all()
    e2e_s = time.perf_counter() - t0
    te = torch.tensor([e2e_s], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e_value = world * B * args.steps / float(te.item())
    del host_sets, dev_bufs

    # ---- second headline metric: rotated IoU pairs/s on BASELINE configs[3] ------------------------------------
    # 21,824 anchors x 500 GTs x 64 images; anchor rows dealt out to the ranks in 32-row tiles, cyclically; every
    # rank allocates only its own rows.  Three forms (SURVEY 8e): compute only, compute + per-GT column maxima +
    # one [B,M] MAX all-reduce (what label assignment consumes), compute + literal all-gather of the row tiles.
    from s2anet_b200 import synth
    from s2anet_b200.box_iou_rotated import box_iou_rotated_tiles
    IB, IM = 64, 500
    an = torch.from_numpy(synth.all_level_anchors(IB, 3)).to(dev)
    gt = torch.from_numpy(np.stack([synth.dota_like_gt(IM, 100 + i) for i in range(IB)])).to(dev)
    N_an = an.size(1)
    pairs = IB * N_an * IM
    tiles_mine, rows_mine = sdist.shard_tiles(N_an, rank, world)
    local_iou = torch.empty((IB, len(tiles_mine) * sdist.TILE_ROWS, IM), dtype=torch.float32, device=dev)

    def iou_compute():
        box_iou_rotated_tiles(an, gt, rank, world, compact=True, out=local_iou, tile_rows=sdist.TILE_ROWS)

    def iou_max_allreduce():
        iou_compute()
        gmax = local_iou[:, : rows_mine.numel()].amax(dim=1)
        if world > 1:
            dist.all_reduce(gmax, op=dist.ReduceOp.MAX)
        return gmax

    def timed_max(fn, reps):
        sync_all()
        t_ = torch.tensor([cuda_time(torch, fn, reps)], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t_, op=dist.ReduceOp.MAX)
        return float(t_.item())

    iou_ms = timed_max(iou_compute, 5)
    iou_ar_ms = timed_max(iou_max_allreduce, 5)
    iou_ag_ms = None
    if world > 1:
        def iou_all_gather():
            return sdist.sharded_box_iou(an, gt, gather=True)
        iou_ag_ms = timed_max(iou_all_gather, 2)
    iou_bytes = 4.0 * pairs + 20.0 * IB * (N_an + IM)
    peaks0 = load_peaks()
    fma = None
    if rank == 0:
        import ctypes
        v = ctypes.c_double(0.0)
        with torch.cuda.device(dev):
            rc = _lib.load().s2a_measure_fp32_fma_tflops(ctypes.byref(v), 3, _lib.stream_ptr(dev))
        fma = float(v.value) if rc == 0 else None
    iou_metric = {"metric": "rotated IoU pairs/s", "value": pairs / (iou_ms / 1e3), "unit": "pairs/s", "ms": iou_ms,
                  "config": "21,824 anchors x 500 GTs x 64 images (BASELINE configs[3]); anchor rows dealt to %d GPU(s) in "
                            "%d-row tiles, cyclically; value = compute form, max over ranks" % (world, sdist.TILE_ROWS),
                  "forms": {"compute_only_ms": iou_ms,
                            "max_allreduce_ms": iou_ar_ms, "max_allreduce_pairs_per_s": pairs / (iou_ar_ms / 1e3),
                            "all_gather_ms": iou_ag_ms,
                            "all_gather_pairs_per_s": None if iou_ag_ms is None else pairs / (iou_ag_ms / 1e3),
                            "note": "max_allreduce = kernel + per-GT column maxima of the local rows (one more read of the "
                                    "local matrix) + one [64,500] MAX all-reduce over NCCL; all_gather = kernel + "
                                    "all_gather_into_tensor of the packed tiles (2.8 GB on every rank) + the copy that undoes "
                                    "the cyclic deal"},
                  "roofline": {"bound": "hbm", "achieved": iou_bytes / (iou_ms / 1e3) / 1e9 / world, "peak": peaks0["hbm"],
                               "unit": "GB/s", "frac": iou_bytes / (iou_ms / 1e3) / 1e9 / world / peaks0["hbm"],
                               "note": "algorithmic bytes 4*N*M + 20*(N+M) per image; per-GPU figure"},
                  "fp32": None if not fma else {
                      "fma_tflops_measured": fma, "flop_per_pair": IOU_FLOP_PER_PAIR,
                      "pairs_per_s_fp32_bound": fma * 1e12 / IOU_FLOP_PER_PAIR,
                      "frac_of_fp32_bound": pairs / (iou_ms / 1e3) / world / (fma * 1e12 / IOU_FLOP_PER_PAIR),
                      "note": "SURVEY 8d convention: 350 FP32 flop per pair (the reference's no-intersection case) against the "
                              "FMA throughput measured in this run (s2a_measure_fp32_fma_tflops); per-GPU figure.  The kernel "
                              "decides ~95 % of the pairs with a ~20-flop test, so the fraction can exceed 1."}}
    del local_iou, an, gt

    if rank != 0:
        return shutdown(torch, dist, world, graphs)

    # ---- roofline of the dominant kernel of this library: the AlignConv tcgen05 implicit GEMM,
    # timed alone with CUDA events on its launch stream over all five levels of the batch
    peaks = load_peaks()
    roof = None
    refines = None
    if dtype != torch.float32:
        w = head.align_conv.deform_conv.weight
        outs = head.forward_levels(feat_sets[0])
        refines = [o[5] for o in outs]
        del outs
        from s2anet_b200.conv_tc import alignconv_forward_tc_multi
        t_align = cuda_time(torch, lambda: alignconv_forward_tc_multi(feat_sets[0], refines, w, STRIDES), 10) / 1e3
        p3 = feat_sets[0][0]
        t_p3 = cuda_time(torch, lambda: alignconv_forward(p3, refines[0], w, 8), 10) / 1e3
        flops_p3 = 2.0 * B * 128 * 128 * 256 * 2304
        ach = flops_p3 / t_p3 / 1e12
        roof = {"bound": "tensor", "kernel": "conv_tc_kernel<ALIGN,bf16> (AlignConv, P3 level of the batch, one launch)",
                "achieved": ach, "peak": peaks["bf16_burst"], "unit": "TFLOP/s", "frac": ach / peaks["bf16_burst"],
                "peak_source": peaks["source"] + " bf16_tflops (burst: kernel timed alone)", "traffic": load_traffic(B),
                "all_levels_tflops": ALIGN_FLOPS_PER_IMAGE * B / t_align / 1e12,
                "alignconv_share_of_step": t_align / (ms / 1e3 / args.steps)}

    # ---- the other bench legs of BASELINE.md section 3 (rank 0, one GPU's worth of work each) ---------------------
    extra = None
    if not args.no_extra and world == 1:
        extra = extra_legs(torch, np, dev, dtype, head, feat_sets, refines, peaks, args)

    cpu = None
    if not args.no_cpu_baseline and world == 1:
        torch.set_num_threads(host_cores())
        cpu_head = build_head(torch, None, torch.float32, seed=0)
        cpu_head.odm_cls_head.bias.data.copy_(head.odm_cls_head.bias.detach().float().cpu())
        ref = CpuReferenceHead(cpu_head)
        cf = [f[:1].float().cpu().contiguous() for f in feat_sets[0]]
        t0 = time.perf_counter()
        r = ref.detect(cf)
        dt = time.perf_counter() - t0
        cpu = {"value": 1.0 / dt, "unit": UNIT, "cores": torch.get_num_threads(), "kind": ref.kind,
               "sample": "1 of the %d images of one step (all 5 FPN levels, %d candidates -> %d detections), fp32, "
                         "timed once: %.1f s" % (B, int(ncand), int(r[0][0].shape[0]), dt)}
        if extra is not None:
            extra["cpu"] = cpu_legs(torch, np, args)

    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": args.dtype, "data": "synthetic",
        "config": {"workload": "S2ANet R-50-FPN head + 15-class rotated NMS at 1024x1024, batch %d per GPU "
                               "(BASELINE configs[4] per-GPU shard; configs[2] is the same at batch 1)" % B,
                   "global_batch": world * B, "positions_per_image": POSITIONS, "nms_candidates_per_image": int(ncand),
                   "odm_cls_bias": calibrated_bias,
                   "detections_per_image": ndet, "parallelism": "dp%d (image-sharded, detection exchange: %s)" % (world, exch_mode),
                   "l2": "two rotating feature sets (2 x %.0f MB) plus >1 GB of activations per step: working set > 126 MB L2"
                         % (h2d_bytes / 1e6)},
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d_bytes, "d2h_bytes_per_step": d2h_bytes},
        "gpu_launches": launches, "clocks": clocks, "roofline": roof, "cpu_baseline": cpu, "iou": iou_metric,
        "exchange": exchange, "configs": extra, "parity": load_parity(),
    }
    print(json.dumps(line), flush=True)
    shutdown(torch, dist, world, graphs)


def shutdown(torch, dist, world, graphs):
    """Leave cleanly and in bounded time: CUDA graphs that captured collectives / peer barriers must die before the
    communicator does (destroying the process group first hung a 2-GPU run for the whole gpurun limit), and a watchdog
    ends the process if the teardown still stalls."""
    if world <= 1:
        return
    import gc
    wd = threading.Timer(30.0, lambda: os._exit(0))
    wd.daemon = True
    wd.start()
    graphs.clear()
    gc.collect()
    torch.cuda.synchronize()
    try:
        dist.destroy_process_group()
    except Exception:
        pass
    sys.stdout.flush()
    os._exit(0)


def extra_legs(torch, np, dev, dtype, head, feat_sets, refines, peaks, args):
    """BASELINE.md section 3 legs that are not the headline: config 1 (2,000 boxes), config 2 (one AlignConv + ORConv2d
    layer at P3, batch 1), config 3 (the head + NMS at batch 1), NMS at N = 2,000 / 20,000, the step at 10 k candidates."""
    from s2anet_b200 import synth
    from s2anet_b200.box_iou_rotated import box_iou_rotated
    from s2anet_b200.nms_rotated import ml_nms_rotated, nms_rotated_op
    out = {}
    # config 1: IoU 2000 x 2000 and NMS on the clustered set
    b, s, l = synth.clustered_boxes(n_seed=400, rep=5, seed=0)
    tb, ts, tl = torch.from_numpy(b).to(dev), torch.from_numpy(s).to(dev), torch.from_numpy(l).to(dev)
    iou_us = cuda_time(torch, lambda: box_iou_rotated(tb, tb), 20) * 1e3
    nms_us = cuda_time(torch, lambda: nms_rotated_op(tb, ts, 0.5), 20) * 1e3
    ml_us = cuda_time(torch, lambda: ml_nms_rotated(tb, ts, tl, 0.5), 20) * 1e3
    out["config1_2000_boxes"] = {"box_iou_rotated_2000x2000_us": iou_us, "iou_pairs_per_s": 4e6 / (iou_us * 1e-6),
                                 "nms_rotated_us": nms_us, "ml_nms_rotated_us": ml_us,
                                 "kept": int(nms_rotated_op(tb, ts, 0.5).numel()),
                                 "note": "NMS times include the 4-byte host read of the result length"}
    # NMS at N = 20,000 (the stress point of SURVEY 8d): upper-triangle pairs per second
    b2, s2, _ = synth.clustered_boxes(n_seed=4000, rep=5, seed=1)
    tb2, ts2 = torch.from_numpy(b2).to(dev), torch.from_numpy(s2).to(dev)
    n2 = b2.shape[0]
    nms20_ms = cuda_time(torch, lambda: nms_rotated_op(tb2, ts2, 0.5), 5)
    out["nms_rotated_20000"] = {"ms": nms20_ms, "pairs_per_s": n2 * (n2 - 1) / 2 / (nms20_ms / 1e3)}
    # per-call host cost of the eager drop-in path (ctypes binding + argument checks + launch), on inputs so small that
    # the kernels are empty: wall clock per call over 200 back-to-back calls, one synchronize at the end
    def call_us(fn, n=200):
        for _ in range(10):
            fn()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(n):
            fn()
        torch.cuda.synchronize()
        return (time.perf_counter() - t0) / n * 1e6
    tiny = tb[:4].contiguous()
    xs_ = torch.randn(1, 64, 8, 8, device=dev).to(torch.bfloat16).contiguous(memory_format=torch.channels_last)
    an_ = torch.from_numpy(synth.refined_anchors(1, 8, 8, 8, seed=1)).to(dev)
    w_ = (torch.randn(64, 64, 3, 3, device=dev) * 0.05).to(torch.bfloat16)
    from s2anet_b200.alignconv import alignconv_forward as _af
    from s2anet_b200 import _torch_ext
    ext_on = _torch_ext.module() is not None
    over = {
        "binding": "torch extension (_s2a_torch.so: at::Tensor in, one C-ABI call, at::Tensor out)" if ext_on else "ctypes",
        "box_iou_rotated_4x4": call_us(lambda: box_iou_rotated(tiny, tiny)),
        "alignconv_forward_bf16_8x8": call_us(lambda: _af(xs_, an_, w_, 8)),
        "nms_rotated_4_boxes_incl_4_byte_readback": call_us(lambda: nms_rotated_op(tiny, ts[:4].contiguous(), 0.5), 50),
        "note": "wrapper + binding + kernel launch per call (alignconv always goes through ctypes: its packed-weight cache lives "
                "in Python); the bench step itself replays a CUDA graph and pays none of it"}
    if ext_on:                                            # the same two calls through the ctypes wrappers, for comparison
        saved = (_torch_ext._MOD, _torch_ext._TRIED)
        _torch_ext._MOD, _torch_ext._TRIED = None, True
        try:
            over["ctypes_box_iou_rotated_4x4"] = call_us(lambda: box_iou_rotated(tiny, tiny))
            over["ctypes_nms_rotated_4_boxes_incl_4_byte_readback"] = call_us(lambda: nms_rotated_op(tiny, ts[:4].contiguous(), 0.5), 50)
        finally:
            _torch_ext._MOD, _torch_ext._TRIED = saved
    out["dropin_call_overhead_us"] = over
    if dtype != torch.float32 and refines is not None:
        from s2anet_b200.alignconv import alignconv_forward
        from s2anet_b200.orn import orconv_forward
        # config 2: single AlignConv + ORConv2d layer, P3, batch 1
        x1 = feat_sets[0][0][:1].contiguous(memory_format=torch.channels_last)
        a1 = refines[0][:1].contiguous()
        w = head.align_conv.deform_conv.weight
        oc = head.or_conv
        y1 = alignconv_forward(x1, a1, w, 8)
        t_al = cuda_time(torch, lambda: alignconv_forward(x1, a1, w, 8), 30) / 1e3
        t_or = cuda_time(torch, lambda: orconv_forward(y1, oc.weight, oc.indices, oc.bias, with_pool=True), 30) / 1e3
        fl = 2.0 * 128 * 128 * 256 * 2304
        out["config2_p3_batch1"] = {
            "alignconv_us": t_al * 1e6, "alignconv_tflops": fl / t_al / 1e12, "alignconv_frac_of_peak": fl / t_al / 1e12 / peaks["bf16_burst"],
            "orconv_pool_us": t_or * 1e6, "orconv_tflops": fl / t_or / 1e12, "orconv_frac_of_peak": fl / t_or / 1e12 / peaks["bf16_burst"],
            "note": "128 tiles on 148 SMs: a batch-1 P3 launch cannot fill the GPU (86 % at best); eager calls incl. launch overhead"}
        # config 2 with fp32 tensors (the dtype the reference's training runs the op in): 3 x TF32 on tcgen05, the SIMT
        # kernel beside it; BASELINE.md quotes the reference binary at 0.59 ms for this layer on this GPU
        from s2anet_b200 import alignconv as _ac
        x32, w32 = x1.float(), w.float()
        t_tf = cuda_time(torch, lambda: alignconv_forward(x32, a1, w32, 8), 20) / 1e3
        _ac.set_fp32_path("simt")
        try:
            t_simt = cuda_time(torch, lambda: alignconv_forward(x32, a1, w32, 8), 5) / 1e3
        finally:
            _ac.set_fp32_path("tf32x3")
        out["config2_p3_batch1_fp32"] = {
            "alignconv_tf32x3_us": t_tf * 1e6, "alignconv_tf32x3_tflops": fl / t_tf / 1e12, "alignconv_simt_us": t_simt * 1e6,
            "note": "fp32 in / fp32 NCHW out; tf32x3 = three tcgen05.mma.kind::tf32 per K step on hi / lo splits (rel-L2 5.5e-6 "
                    "of fp64, profiles/r2_parity_errors.json); simt = individually rounded FMAs (set_fp32_path('simt'))"}
        del x32, w32
        # config 3: head + NMS at batch 1 (CUDA graph replay latency)
        f1 = [f[:1].contiguous(memory_format=torch.channels_last) for f in feat_sets[0]]
        for _ in range(2):
            head.detect(f1)
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            head.detect(f1)
        lat = cuda_time(torch, g.replay, 50)
        out["config3_batch1"] = {"ms_per_image": lat, "images_per_s": 1e3 / lat,
                                 "note": "head + NMS only (the ResNet-50/FPN backbone stays stock PyTorch and is not timed)"}
        # SURVEY 8(f) row 1: the deformable-conv backward of AlignConv at P3, batch 8, on tcgen05 (16-bit training route)
        from s2anet_b200.conv_tc import deform_conv_dgrad_tc, deform_conv_wgrad_tc
        xb = feat_sets[0][0]
        gyb = torch.randn_like(xb)
        offb = torch.randn(xb.size(0), 18, xb.size(2), xb.size(3), device=dev) * 1.2
        t_dg = cuda_time(torch, lambda: deform_conv_dgrad_tc(gyb, offb, w), 3, warm=1)
        t_wg = cuda_time(torch, lambda: deform_conv_wgrad_tc(xb, offb, gyb), 3, warm=1)
        flb = 2.0 * xb.size(0) * 128 * 128 * 256 * 2304
        out["backward_p3_batch%d" % xb.size(0)] = {
            "dgrad_ms": t_dg, "dgrad_tflops": flb / t_dg / 1e9, "wgrad_ms": t_wg, "wgrad_tflops": flb / t_wg / 1e9,
            "note": "dgrad = nine 1x1 implicit GEMMs with a bilinear scatter epilogue (bound by 4.8 GB of L2 reductions, issued as full 128-byte segments); wgrad = "
                    "MN-major operands, accumulator in tensor memory (bound by the nine-fold re-gather from L2); no column buffer"}
        del gyb, offb
        # the step at ~10 k candidates per image (SURVEY 8d: 2-10 k)
        bias0 = head.odm_cls_head.bias.detach().clone()
        n10 = head.calibrate_scores(feat_sets[0], 10000)
        for _ in range(2):
            head.detect(feat_sets[0])
        torch.cuda.synchronize()
        g2 = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g2):
            head.detect(feat_sets[0])
        ms10 = cuda_time(torch, g2.replay, 20)
        B = feat_sets[0][0].size(0)
        out["step_at_10k_candidates"] = {"candidates_per_image": int(n10), "ms_per_step": ms10, "images_per_s": B * 1e3 / ms10}
        with torch.no_grad():
            head.odm_cls_head.bias.copy_(bias0)
    return out


def cpu_legs(torch, np, args):
    """The reference's CPU kernels on bounded samples of configs 1 and 4 (1 core: they are strictly serial)."""
    from oracle import build_oracle
    from s2anet_b200 import synth
    out = {"cores": "1 of %d" % host_cores()}
    iou = build_oracle.load_ref_extension("box_iou_rotated_cuda", "cpu")
    nms = build_oracle.load_ref_extension("nms_rotated_cuda", "cpu")
    b, s, _ = synth.clustered_boxes(n_seed=400, rep=5, seed=0)
    tb, ts = torch.from_numpy(b), torch.from_numpy(s)
    if iou is not None:
        t0 = time.perf_counter()
        iou.box_iou_rotated(tb[:250].contiguous(), tb)
        dt = time.perf_counter() - t0
        out["config1_box_iou_rotated_cpu"] = {"sample": "250 of the 2,000 rows (500,000 pairs)", "seconds": dt,
                                               "pairs_per_s": 5e5 / dt, "extrapolated_2000x2000_s": dt * 8}
        an = torch.from_numpy(synth.all_level_anchors(1, 3)[0][::22][:992].copy())
        gt = torch.from_numpy(synth.dota_like_gt(500, 100))
        t0 = time.perf_counter()
        iou.box_iou_rotated(an, gt)
        dt = time.perf_counter() - t0
        npairs = an.size(0) * gt.size(0)
        out["config4_box_iou_rotated_cpu"] = {"sample": "%d anchors (every 22nd) x 500 GTs of one image (%d pairs)" % (an.size(0), npairs),
                                               "seconds": dt, "pairs_per_s": npairs / dt,
                                               "extrapolated_698368000_pairs_s": dt * 698368000.0 / npairs}
    if nms is not None:
        t0 = time.perf_counter()
        keep = nms.nms_rotated(tb[:1000].contiguous(), ts[:1000].contiguous(), 0.5)
        dt = time.perf_counter() - t0
        out["config1_nms_rotated_cpu"] = {"sample": "the first 1,000 of the 2,000 boxes", "seconds": dt, "kept": int(keep.numel()),
                                           "extrapolated_2000_boxes_s": dt * 4}
    return out


if __name__ == "__main__":
    main()
