"""One step of the bench.py workload (configs[1]: 50 x 1 Mbp, k = 31, compute_device) under torch.profiler with CUDA activities.

Prints the kernels of the last of a few profiled steps in stream order with their durations and the idle gap before each, then the
sum of kernel time and the sum of the gaps between the step's first kernel start and its last kernel end.  The gaps are where the
GPU waits for the host: launches issued one at a time and synchronising read-backs.  The profiler adds its own overhead per launch,
so the step time of bench.py (no profiler) is the number to compare; the kernel list and the gap sum are what this script is for.

    python profiles/step_timeline.py [--out FILE.json]
"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="also write the table as JSON here")
    ap.add_argument("--steps", type=int, default=5)
    args = ap.parse_args()
    import torch
    from torch.profiler import ProfilerActivity, profile
    import kmercamel_b200 as kb
    from kmercamel_b200 import synth

    seq = synth.frame_records(synth.random_genome_records(50, 1_000_000, 12345))[0]
    d = torch.from_numpy(seq).cuda()
    ctx = kb.Context(0, torch.cuda.current_stream().cuda_stream)
    for _ in range(5):
        ctx.compute_device(d.data_ptr(), d.numel(), k=31)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        for i in range(args.steps):
            with torch.profiler.record_function(f"step{i}"):
                ctx.compute_device(d.data_ptr(), d.numel(), k=31)
            torch.cuda.synchronize()
    events = prof.events()
    kern = sorted([e for e in events if e.device_type == torch.autograd.DeviceType.CUDA and "memcpy" not in e.name.lower()
                   and "memset" not in e.name.lower()], key=lambda e: e.time_range.start)
    steps = sorted([e for e in events if e.name.startswith("step")], key=lambda e: e.time_range.start)
    # the device work of the last step: kernels that start after the host entered it
    last = steps[-1]
    mine = [e for e in kern if e.time_range.start >= last.time_range.start]
    ops = sorted([e for e in events if e.device_type == torch.autograd.DeviceType.CUDA and e.time_range.start >= last.time_range.start
                  and not e.name.startswith("step")],  # the step annotation's own device range spans everything
                 key=lambda e: e.time_range.start)
    rows = []
    prev_end = None
    for e in ops:
        gap = 0.0 if prev_end is None else max(0.0, e.time_range.start - prev_end)
        rows.append({"name": e.name[:90], "us": round(e.time_range.end - e.time_range.start, 2), "gap_before_us": round(gap, 2)})
        prev_end = max(prev_end or 0, e.time_range.end)
    busy = sum(r["us"] for r in rows)
    gaps = sum(r["gap_before_us"] for r in rows)
    span = ops[-1].time_range.end - ops[0].time_range.start if ops else 0.0
    print(f"{'kernel / copy':92s} {'us':>8s} {'gap before':>10s}")
    for r in rows:
        print(f"{r['name']:92s} {r['us']:8.2f} {r['gap_before_us']:10.2f}")
    summary = {"gpu": torch.cuda.get_device_name(0), "kernels": len(mine), "device_ops": len(rows), "busy_us": round(busy, 1),
               "idle_gaps_us": round(gaps, 1), "span_us": round(span, 1), "read_backs_per_step": None}
    try:  # a build without the counter leaves it None
        r0 = ctx.stat("read_backs")
        ctx.compute_device(d.data_ptr(), d.numel(), k=31)
        summary["read_backs_per_step"] = ctx.stat("read_backs") - r0
    except kb.KcError:
        pass
    print(json.dumps(summary))
    if args.out:
        json.dump({"summary": summary, "ops": rows}, open(args.out, "w"), indent=1)


if __name__ == "__main__":
    main()
