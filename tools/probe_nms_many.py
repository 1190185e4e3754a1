"""Time the fused multiclass NMS at 5,344 to 21,824 boxes per image (batch 8, 15 classes), against the composed per-image
path it replaces above 6,144 boxes.

    python tools/probe_nms_many.py [--reps 200] [--json out.json]

Scores are bench-density: sigmoid of N(-5.6, 1.5) logits rounded to bf16, about 0.56 (box, class) candidates per box
(3,000 per image at 5,344 boxes, the bench's calibration); boxes are synth.clustered_boxes.  For each n:

  * fused: multiclass_nms_rotated_batched captured in a CUDA graph, CUDA events around `reps` replays after warm-up;
    the CTA selection runs up to MC_FUSED_MAX_BOXES boxes per image, the segmented sort above;
  * composed: the per-image composition on the generic ml_nms_rotated kernel (_multiclass_composed), eager, one host
    read per image -- what the batched entry ran above 6,144 boxes before the segmented route existed.

At 5,344 the segmented route is timed too, on the same images padded with 801 boxes that are no candidate of any class
(6,145 boxes per image, same detections): an upper bound of that route at the bench's size, since its key kernel reads
15 % more scores.  The two routes alternate over `--rounds` rounds to show the spread, and one profiled eager pass per
route gives the selection kernels' own time.  Prints the card name and power limit with the numbers.
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from s2anet_b200 import synth  # noqa: E402
from s2anet_b200.nms_rotated import (MC_FUSED_MAX_BOXES, _multiclass_composed,  # noqa: E402
                                     multiclass_nms_rotated_batched)

B, C, THR, IOU, MAXK = 8, 15, 0.05, 0.5, 2000


def card():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = "unknown"
    return name, q


def inputs(n, dev, seed):
    rng = np.random.default_rng(seed)
    bb = np.stack([synth.clustered_boxes(n_seed=n // 4 + 1, rep=4, seed=seed + i)[0][:n] for i in range(B)])
    logits = torch.from_numpy(rng.normal(-5.6, 1.5, (B, n, C)).astype(np.float32))
    sc = torch.sigmoid(logits.bfloat16()).float()
    return torch.from_numpy(bb).to(dev), sc.to(dev)


def padded(bb, sc, n_to):
    """The same images with boxes appended that are no candidate of any class."""
    extra = n_to - bb.size(1)
    return (torch.cat([bb, bb[:, :1].expand(-1, extra, -1)], 1).contiguous(),
            torch.cat([sc, sc.new_zeros((B, extra, C))], 1).contiguous())


def graph_of(bb, sc):
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        for _ in range(3):
            multiclass_nms_rotated_batched(bb, sc, THR, IOU, MAXK)
    torch.cuda.current_stream().wait_stream(s)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        out = multiclass_nms_rotated_batched(bb, sc, THR, IOU, MAXK)
    g.replay()                                                    # (capture alone leaves the outputs unwritten)
    torch.cuda.synchronize()
    return g, out


def time_replays(g, reps):
    for _ in range(10):
        g.replay()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        g.replay()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps * 1e3


def time_composed(bb, sc, reps):
    def run():
        return [_multiclass_composed(bb[i], sc[i], THR, IOU, MAXK) for i in range(B)]
    run()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        out = run()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps * 1e3, out


def same(fused, composed):
    dets, labels, counts = fused
    for i, (d, l) in enumerate(composed):
        k = int(counts[i])
        if k != d.size(0) or (k and not (torch.equal(dets[i, :k], d) and torch.equal(labels[i, :k], l.reshape(-1)))):
            return False
    return True


def selection_us(bb, sc, reps=20):
    """Per call, device time of the selection kernels (CTA select, or memset + key + segmented sort + gather) and of
    all kernels of the call, from one profiled eager pass."""
    from torch.profiler import ProfilerActivity, profile
    multiclass_nms_rotated_batched(bb, sc, THR, IOU, MAXK)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            multiclass_nms_rotated_batched(bb, sc, THR, IOU, MAXK)
        torch.cuda.synchronize()
    sel = tot = 0.0
    for e in prof.key_averages():
        t = getattr(e, "device_time_total", None)
        if t is None:
            t = e.cuda_time_total
        name = e.key
        if not any(k in name for k in ("mc_", "SegmentedRadixSort", "Memset", "memset")):
            continue
        tot += t
        if any(k in name for k in ("mc_select_sort", "mc_key", "mc_gather", "SegmentedRadixSort", "Memset", "memset")):
            sel += t
    return sel / reps, tot / reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=200)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--json", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("probe_nms_many: needs a CUDA device")
    dev = torch.device("cuda", 0)
    name, power = card()
    print("card: %s | power.limit, clocks.max.sm: %s" % (name, power))
    res = {"card": name, "power_limit_max_sm_clock": power, "batch": B, "classes": C, "reps": args.reps, "sizes": []}
    for n in (5344, 6720, 7280, 21824):
        bb, sc = inputs(n, dev, n)
        cand = float((sc > THR).sum(dim=(1, 2)).float().mean())
        g, out = graph_of(bb, sc)
        comp_us, comp = time_composed(bb, sc, 5)
        row = {"n": n, "route": "cta" if n <= MC_FUSED_MAX_BOXES else "segmented", "candidates_per_image": cand,
               "largest_class_segment": int((sc > THR).sum(dim=1).max()), "composed_eager_us": comp_us,
               "same_as_composed": same(out, comp)}
        if n <= MC_FUSED_MAX_BOXES:
            pb, ps = padded(bb, sc, MC_FUSED_MAX_BOXES + 1)
            gp, outp = graph_of(pb, ps)
            row["padded_same"] = same(outp, [(out[0][i, :int(out[2][i])], out[1][i, :int(out[2][i])]) for i in range(B)])
            cta, seg = [], []
            for _ in range(args.rounds):                          # alternate the two routes
                cta.append(time_replays(g, args.reps))
                seg.append(time_replays(gp, args.reps))
            row["fused_graph_us_rounds"] = cta
            row["segmented_padded_graph_us_rounds"] = seg
            row["selection_us_cta"], row["call_kernels_us_cta"] = selection_us(bb, sc)
            row["selection_us_segmented_padded"], row["call_kernels_us_segmented_padded"] = selection_us(pb, ps)
            del gp, outp
        else:
            row["fused_graph_us_rounds"] = [time_replays(g, args.reps) for _ in range(args.rounds)]
            row["selection_us_segmented"], row["call_kernels_us_segmented"] = selection_us(bb, sc)
        del g, out
        torch.cuda.empty_cache()
        res["sizes"].append(row)
        print(json.dumps(row))
    print("\n%-7s %-10s %-8s %-28s %-28s %s" % ("n", "route", "cand/img", "fused graph replay us", "selection us",
                                                "composed eager us"))
    for r in res["sizes"]:
        f = r["fused_graph_us_rounds"]
        sel = r.get("selection_us_cta", r.get("selection_us_segmented"))
        print("%-7d %-10s %-8.0f %-28s %-28s %.0f" % (r["n"], r["route"], r["candidates_per_image"],
                                                     "%.1f (%.1f-%.1f)" % (float(np.median(f)), min(f), max(f)),
                                                     "%.1f" % sel, r["composed_eager_us"]))
        if "segmented_padded_graph_us_rounds" in r:
            s = r["segmented_padded_graph_us_rounds"]
            print("%-7s %-10s %-8s %-28s %-28s" % ("", "segmented*", "",
                                                   "%.1f (%.1f-%.1f)" % (float(np.median(s)), min(s), max(s)),
                                                   "%.1f" % r["selection_us_segmented_padded"]))
    print("(* padded to %d boxes with non-candidates; card %s, %s)" % (MC_FUSED_MAX_BOXES + 1, name, power))
    if args.json:
        os.makedirs(os.path.dirname(os.path.abspath(args.json)), exist_ok=True)
        with open(args.json, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
