#!/usr/bin/env python
"""A/B of the FAM branch of the detection step, built like bench.py (build_head, make_feats seeds 4 / 104, the committed
classification bias re-calibrated to 3,000 candidates, batch 8, bf16):

  A  the full forward: detect_from_outs(forward_levels(f))   (FAM classification + regression towers)
  B  detect(f): the FAM regression branch only (S2ANetHead._forward_detect)

Each path is captured as one CUDA graph per feature set; the graphs are replayed interleaved (A B A B ...), ROUNDS
rounds of STEPS steps on the two rotating feature sets.  Then, in a separate pass, torch.profiler lists every launch of
one step per path, and the outputs are compared (they must be torch.equal).

    python tools/ab_fam_branch.py [--batch 8] [--dtype bf16] [--rounds 5] [--steps 100] [--bench-dump DIR --bench-steps K]

--bench-dump: also compare A's detections with `bench.py --steps K --dump-outputs DIR` (same seeds and arguments; its
last timed step ran on feature set (K - 1) % 2).
"""
import argparse
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_info(index):
    q = "name,power.limit,clocks.max.sm"
    try:
        out = subprocess.run(["nvidia-smi", "-i", str(index), "--query-gpu=" + q, "--format=csv,noheader"],
                             stdout=subprocess.PIPE, text=True, timeout=10).stdout.strip()
    except Exception as e:                          # the numbers below are still valid, only unlabeled
        out = "nvidia-smi unavailable (%s)" % e
    return out


def match(dets0, dets1, tag):
    """bench-style matcher: counts within max(3, 2 %), top 100 matched by label, score (1e-3) and box (0.05 px)."""
    d0, l0, c0 = dets0
    d1, l1, c1 = dets1
    ok, worst_s, worst_b = True, 0.0, 0.0
    for b in range(d0.size(0)):
        n0, n1 = int(c0[b]), int(c1[b])
        ok &= abs(n0 - n1) <= max(3, int(0.02 * n0))
        for i in range(min(100, n0, n1)):
            cand = ((d0[b, :n0, 5] - d1[b, i, 5]).abs() <= 1e-3) & (l0[b, :n0] == l1[b, i])
            if not bool(cand.any()):
                ok = False
                continue
            err = float((d0[b, :n0][cand, :4] - d1[b, i, :4]).abs().max(dim=1)[0].min())
            worst_b = max(worst_b, err)
            worst_s = max(worst_s, float((d0[b, :n0][cand, 5] - d1[b, i, 5]).abs().min()))
            ok &= err <= 0.05
    print("%s: matcher %s (worst score diff %.2e, worst box diff %.3f px; counts %s vs %s)" %
          (tag, "holds" if ok else "FAILS", worst_s, worst_b, c0.tolist(), c1.tolist()))
    return ok


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=8)
    ap.add_argument("--dtype", default="bf16", choices=["bf16", "fp16"])
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--bench-dump", default=None)
    ap.add_argument("--bench-steps", type=int, default=None)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("ab_fam_branch.py: no CUDA device; this measurement needs a B200")
    from bench import CALIBRATED_BIAS, ClockSampler, build_head, make_feats
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    dtype = {"bf16": torch.bfloat16, "fp16": torch.float16}[args.dtype]
    B = args.batch
    head = build_head(torch, dev, dtype, seed=0, bias=CALIBRATED_BIAS[3000])
    feat_sets = [make_feats(torch, B, 4 + 100 * i, dev, dtype) for i in range(2)]
    ncand = head.calibrate_scores(feat_sets[0], 3000)
    print("GPU: %s | batch %d %s, %.0f NMS candidates per image" % (gpu_info(0), B, args.dtype, ncand))

    paths = {
        "A": lambda f: head.detect_from_outs(head.forward_levels(f)),
        "B": lambda f: head.detect(f),
    }
    graphs = {}
    with torch.no_grad():
        for name, fn in paths.items():
            for i, f in enumerate(feat_sets):
                for _ in range(2):
                    fn(f)
                torch.cuda.synchronize()
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g):
                    out = fn(f)
                graphs[name, i] = (g, out)
    torch.cuda.synchronize()

    # ---- interleaved timing ----
    ms = {k: [] for k in paths}
    sampler = ClockSampler(0)
    sampler.start()
    for name in paths:                               # warm-up round
        for s in range(10):
            graphs[name, s % 2][0].replay()
    for r in range(args.rounds):
        for name in paths:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            e0.record()
            for s in range(args.steps):
                graphs[name, s % 2][0].replay()
            e1.record()
            torch.cuda.synchronize()
            ms[name].append(e0.elapsed_time(e1) / args.steps)
    clocks = sampler.stop()
    print("SM clock sampled during the rounds: median %s MHz (max %s MHz), reasons %s, %d samples" %
          (clocks["sm_mhz"], clocks["sm_max_mhz"], clocks["reasons"], clocks["samples"]))
    for name in paths:
        v = sorted(ms[name])
        med = v[len(v) // 2]
        print("%s: median %.4f ms/step (min %.4f, max %.4f; spread %.4f) = %.0f images/s | rounds %s" %
              (name, med, v[0], v[-1], v[-1] - v[0], B / med * 1e3, " ".join("%.4f" % x for x in ms[name])))
    gain = [a / b - 1.0 for a, b in zip(ms["A"], ms["B"])]
    print("B vs A images/s per round: %s (min %+.1f %%)" % (" ".join("%+.1f%%" % (100 * x) for x in gain), 100 * min(gain)))

    # ---- per-launch list (separate pass, eager, profiler on) ----
    from torch.profiler import ProfilerActivity, profile
    nprof = 5
    with torch.no_grad():
        for name, fn in paths.items():
            fn(feat_sets[0])
            torch.cuda.synchronize()
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                for s in range(nprof):
                    fn(feat_sets[s % 2])
                torch.cuda.synchronize()
            ev = sorted([e for e in prof.events() if e.device_type.name == "CUDA" and "emcpy" not in e.name and
                         "emset" not in e.name], key=lambda e: e.time_range.start)
            n = len(ev) // nprof
            rows = []
            for j in range(n):
                ts = [ev[s * n + j].time_range.elapsed_us() for s in range(nprof)]
                rows.append((ev[j].name, sorted(ts)[nprof // 2]))
            print("\n%s: %d launches per step, %.1f us summed (median of %d eager steps per launch)" %
                  (name, n, sum(t for _, t in rows), nprof))
            for j, (k, t) in enumerate(rows):
                print("  %2d %9.1f us  %s" % (j, t, k[:110]))

    # ---- outputs ----
    with torch.no_grad():
        outs = {}
        for name in paths:
            graphs[name, 0][0].replay()
            torch.cuda.synchronize()
            outs[name] = [t.clone() for t in graphs[name, 0][1]]
    eq = all(torch.equal(a, b) for a, b in zip(outs["A"], outs["B"]))
    print("\nA vs B outputs torch.equal: %s" % eq)
    if args.bench_dump:
        import numpy as np
        i = (args.bench_steps - 1) % 2
        with torch.no_grad():
            graphs["A", i][0].replay()
            torch.cuda.synchronize()
        ref = [t.cpu() for t in graphs["A", i][1]]
        keep = torch.from_numpy(np.load(os.path.join(args.bench_dump, "image_index.npy"))).long()
        dump = [torch.from_numpy(np.load(os.path.join(args.bench_dump, n + ".npy"))) for n in ("dets", "labels", "counts")]
        bias = np.load(os.path.join(args.bench_dump, "odm_cls_bias.npy"))
        print("bench dump bias %.6f vs this run %.6f" % (float(bias.mean()), float(head.odm_cls_head.bias.float().mean())))
        match((ref[0][keep], ref[1][keep].float(), ref[2][keep]), (dump[0], dump[1], dump[2].int()),
              "A (feature set %d) vs bench.py --dump-outputs" % i)

if __name__ == "__main__":
    main()
