"""Per-boundary gaps of one replayed benchmark step (torch.profiler, CUDA activities).

    python profiles/capture_gaps.py [--batch 128] [--steps 3] [--out FILE]

Builds bench.Workload from the tree this script lives in, captures its three graphs, replays `--steps` steps under
torch.profiler and, for the last step, lists the device kernels in start order.  For each of the step's launch
boundaries it records gap = start(next) - end(previous) and advance = end(next) - end(previous), in microseconds.
Under programmatic dependent launch the gap is negative: the next grid's CTAs are resident (waiting, or with its
loads issued above griddepcontrol.wait) before its predecessor ends.  The advances add up to the step's span, so
they are what a boundary costs.  Prints one JSON
summary line and writes the per-boundary table to --out when given.  Run it separately from timing runs: tracing
slows the host."""
import argparse
import json
import os
import statistics
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=128)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    from torch.profiler import ProfilerActivity, profile

    import bench
    wl = bench.Workload(args.batch, torch.device("cuda"), 2333)
    wl.capture()
    for _ in range(3):
        wl.g_fwd.replay(); wl.g_bwd.replay(); wl.g_wt.replay()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(args.steps):
            wl.g_fwd.replay(); wl.g_bwd.replay(); wl.g_wt.replay()
        torch.cuda.synchronize()
    kernels = sorted((e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA
                      and e.name not in ("Memcpy", "Memset")), key=lambda e: e.time_range.start)
    per_step = wl.launches_per_step
    if len(kernels) < per_step * args.steps:
        raise SystemExit(f"expected {per_step * args.steps} kernels in the trace, found {len(kernels)}")
    step = kernels[-per_step:]
    rows, gaps, adv = [], {"fwd": [], "bwd": [], "other": []}, {"fwd": [], "bwd": [], "other": []}
    for a, b in zip(step, step[1:]):
        gap = b.time_range.start - a.time_range.end
        kind = ("fwd" if "fq_fwd_flat" in a.name and "fq_fwd_flat" in b.name else
                "bwd" if "fq_bwd_flat" in a.name and "fq_bwd_flat" in b.name else "other")
        advance = b.time_range.end - a.time_range.end
        gaps[kind].append(gap)
        adv[kind].append(advance)
        rows.append({"prev": a.name.split("(")[0][:60], "next": b.name.split("(")[0][:60], "gap_us": round(gap, 2),
                     "advance_us": round(advance, 2),
                     "prev_us": round(a.time_range.end - a.time_range.start, 2)})
    span = step[-1].time_range.end - step[0].time_range.start
    busy = sum(k.time_range.end - k.time_range.start for k in step)
    summary = {"batch": args.batch, "kernels_per_step": per_step,
               "gpu": torch.cuda.get_device_name(), "step_span_us": round(span, 1),
               "kernel_time_us": round(busy, 1), "span_minus_kernel_time_us": round(span - busy, 1)}
    for kind, v in gaps.items():
        if v:
            summary[kind] = {"boundaries": len(v), "gap_sum_us": round(sum(v), 1),
                             "gap_median_us": round(statistics.median(v), 2), "advance_sum_us": round(sum(adv[kind]), 1)}
    print(json.dumps(summary), flush=True)
    if args.out:
        with open(args.out, "w") as f:
            json.dump({"summary": summary, "boundaries": rows}, f, indent=1)


if __name__ == "__main__":
    main()
