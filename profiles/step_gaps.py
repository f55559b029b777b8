"""Where the idle time of the bench.py step goes (configs[1]: 50 x 1 Mbp, k = 31, compute_device), under torch.profiler with CUDA
activities, in a run of its own (the profiler slows the host; bench.py's step time is the number to compare).

Per profiled step it reports:
  ops               every device operation (kernel, memset, copy) of the call, its duration and the idle time before it
  busy_us           the sum of their durations
  idle_in_span_us   the step's device span (first op start -> last op end) minus busy time
  idle_between_us   from the end of the previous call's last device op (its status read-back) to this call's first op
  host_us           the host time of one kc_compute_device call, split into
                      prologue    call entry -> the first launch API call
                      enqueue     first launch API call -> the first synchronise call
                      synchronise the synchronise calls (the host waits for the device)
                      epilogue    after the last synchronise call, back to Python
With programmatic dependent launches a kernel may start before its predecessor ends and wait for it, so busy_us can count the same
time twice and idle_in_span_us can come out negative; span_us is the number that holds.
The calls run back to back as in bench.py, so idle_between_us is the GPU's wait for the host between steps.

    python profiles/step_gaps.py [--root DIR] [--steps N] [--out FILE.json]

--root imports kmercamel_b200 from another tree (e.g. a build of the parent commit).
"""
import argparse
import json
import os
import sys

LAUNCH_APIS = ("cudaLaunchKernel", "cudaLaunchKernelExC", "cudaLaunchKernelEx", "cudaGraphLaunch", "cudaMemsetAsync", "cudaMemcpyAsync")
SYNC_APIS = ("cudaStreamSynchronize",)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--root", default=os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    sys.path.insert(0, os.path.abspath(args.root))
    import torch
    from torch.profiler import ProfilerActivity, profile
    import kmercamel_b200 as kb
    from kmercamel_b200 import synth

    seq = synth.frame_records(synth.random_genome_records(50, 1_000_000, 12345))[0]
    d0 = torch.from_numpy(seq).cuda()
    bufs = [d0] + [d0.clone() for _ in range(3)]  # rotated as in bench.py
    ctx = kb.Context(0, torch.cuda.current_stream().cuda_stream)
    for i in range(8):
        ctx.compute_device(bufs[i % 4].data_ptr(), d0.numel(), k=31)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        for i in range(args.steps):
            with torch.profiler.record_function(f"kcstep{i}"):
                ctx.compute_device(bufs[i % 4].data_ptr(), d0.numel(), k=31)
    torch.cuda.synchronize()
    ev = prof.events()
    steps = sorted([e for e in ev if e.name.startswith("kcstep") and e.device_type == torch.autograd.DeviceType.CPU],
                   key=lambda e: e.time_range.start)
    dev = sorted([e for e in ev if e.device_type == torch.autograd.DeviceType.CUDA and not e.name.startswith("kcstep")],
                 key=lambda e: e.time_range.start)
    apis = sorted([e for e in ev if e.device_type == torch.autograd.DeviceType.CPU and e.name in LAUNCH_APIS + SYNC_APIS],
                  key=lambda e: e.time_range.start)

    rows = []
    prev_end = None
    for i, s in enumerate(steps):
        lo, hi = s.time_range.start, s.time_range.end
        # the ops that start after the host entered the step and before it entered the next one
        mine = [e for e in dev if lo <= e.time_range.start and (i + 1 == len(steps) or e.time_range.start < steps[i + 1].time_range.start)]
        ops = []
        last = None
        for e in mine:
            gap = 0.0 if last is None else max(0.0, e.time_range.start - last)
            ops.append({"name": e.name[:90], "us": round(e.time_range.end - e.time_range.start, 2), "gap_before_us": round(gap, 2)})
            last = e.time_range.end if last is None else max(last, e.time_range.end)
        busy = sum(o["us"] for o in ops)
        span = (mine[-1].time_range.end - mine[0].time_range.start) if mine else 0.0
        between = (mine[0].time_range.start - prev_end) if mine and prev_end is not None else None
        prev_end = max(e.time_range.end for e in mine) if mine else prev_end
        host_apis = [a for a in apis if lo <= a.time_range.start <= hi]
        launches = [a for a in host_apis if a.name in LAUNCH_APIS]
        syncs = [a for a in host_apis if a.name in SYNC_APIS]
        first_launch = launches[0].time_range.start if launches else hi
        sync_start = syncs[0].time_range.start if syncs else hi
        sync_end = syncs[-1].time_range.end if syncs else hi
        host = {"total": round(hi - lo, 1), "prologue": round(first_launch - lo, 1),
                "enqueue": round(sync_start - first_launch, 1),
                "synchronise": round(sum(a.time_range.end - a.time_range.start for a in syncs), 1),
                "epilogue": round(hi - sync_end, 1),
                "api_calls": {n: sum(1 for a in host_apis if a.name == n) for n in sorted({a.name for a in host_apis})}}
        rows.append({"step": i, "device_ops": len(ops), "busy_us": round(busy, 1), "span_us": round(span, 1),
                     "idle_in_span_us": round(span - busy, 1), "idle_between_us": None if between is None else round(between, 1),
                     "host_us": host, "ops": ops})
    body = rows[1:]  # the first profiled step has no predecessor inside the trace

    def med(key, sub=None):
        v = sorted((r[key] if sub is None else r[key][sub]) for r in body if (r[key] if sub is None else r[key][sub]) is not None)
        return v[len(v) // 2] if v else None

    summary = {"gpu": torch.cuda.get_device_name(0), "root": os.path.abspath(args.root), "steps": len(body),
               "median": {"device_ops": med("device_ops"), "busy_us": med("busy_us"), "span_us": med("span_us"),
                          "idle_in_span_us": med("idle_in_span_us"), "idle_between_us": med("idle_between_us"),
                          "host_total_us": med("host_us", "total"), "host_prologue_us": med("host_us", "prologue"),
                          "host_enqueue_us": med("host_us", "enqueue"), "host_synchronise_us": med("host_us", "synchronise"),
                          "host_epilogue_us": med("host_us", "epilogue")}}
    last = body[-1]
    print(f"{'device op (last step)':92s} {'us':>8s} {'gap before':>10s}")
    for o in last["ops"]:
        print(f"{o['name']:92s} {o['us']:8.2f} {o['gap_before_us']:10.2f}")
    print("host API calls of the last step:", last["host_us"]["api_calls"])
    print(json.dumps(summary))
    if args.out:
        json.dump({"summary": summary, "steps": rows}, open(args.out, "w"), indent=1)


if __name__ == "__main__":
    main()
