#!/usr/bin/env python3
"""bench.py — `kmercamel compute` hot path on B200 (driver contract, see DESIGN.md "Measurement").

  python bench.py [--gpus N] [--steps K] [--warmup W] [--dump-outputs DIR]   our CUDA path
  python bench.py --impl reference [--gpus N] [--steps K] [--warmup W]   the reference's own CPU path (oracle/_ref)

A step = one pass of the whole hot path (extract -> count -> overlap levels -> emission) over one synthetic input.
Workload = BASELINE.json configs[1]: 50 x 1,000,000 bp uniform random multi-FASTA (seed 12345), k = 31, canonical.
  value  = distinct k-mers represented per second, device-timed, input already resident in HBM;
  e2e    = the same through kc_compute with pinned HOST buffers (H2D of the input and D2H of the superstring
           inside the timed region).
N > 1 (torchrun): ONE job over a genome of N x 50 Mbp (rank r contributes the 50 records of seed 12345 + r), hash-range
sharded as the north star asks: every rank extracts the k-mers of its slice, the (k-mer, position) items go to their
owner rank over NVLink (the level-0 scatter kernel stores straight into the owner's heap through peer pointers, so the
partition pass is the all-to-all; ranks synchronise with device-side signal words, nothing goes through NCCL on the data path), every
rank resolves its hash range and clears the duplicates' bits on every rank, every rank repeats the (sequential, deterministic) greedy
merge and emits — and in the end-to-end arm copies back — its own 16-byte-aligned slice of the superstring.  After the warm-up the
concatenated slices are compared (md5) with the single-GPU result of the same sequence: "parity_n".  Per-GPU counting work is fixed as N grows (weak
scaling); value = distinct k-mers of the whole job / max-over-ranks time.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

K = 31
N_RECORDS = 50
RECORD_LEN = 1_000_000
SEED = 12345
METRIC = "distinct k-mers/sec for `compute` (k=31, canonical, device-timed)"
UNIT = "k-mers/s"


def measured_peak_gbs():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region."""

    def __init__(self, index: int):
        self.index = index
        self.rows = []
        self.proc = None

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={q}", "--format=csv,noheader,nounits",
                                          "-lms", "50"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx.append(float(r[1]))
                for n, v in zip(names, r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            except Exception:
                continue
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def make_workload(rank: int):
    from kmercamel_b200 import synth
    recs = synth.random_genome_records(N_RECORDS, RECORD_LEN, SEED + rank)
    return recs, synth.frame_records(recs)


DUMP_SAMPLE = 1 << 22   # superstring bytes written by --dump-outputs: 16 MB of float32 values + 32 MB of float64 positions


def dump_outputs(out_dir: str, ms: bytes, n_kmers: int):
    """Writes what one `compute` returned, so that two builds can be compared output for output:
      result.npy                        float64 [superstring length, distinct k-mers]
      superstring_sample_positions.npy  float64 positions in the masked superstring: one per equal stratum, drawn with a fixed seed
                                        (every position when the superstring has at most DUMP_SAMPLE bytes)
      superstring_sample.npy            float32 byte values of the superstring at those positions"""
    n = len(ms)
    if n <= DUMP_SAMPLE:
        pos = np.arange(n, dtype=np.int64)
    else:
        edges = np.arange(DUMP_SAMPLE + 1, dtype=np.int64) * n // DUMP_SAMPLE
        pos = edges[:-1] + np.random.default_rng(SEED).integers(0, np.diff(edges))
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "result.npy"), np.array([n, n_kmers], dtype=np.float64))
    np.save(os.path.join(out_dir, "superstring_sample.npy"), np.frombuffer(ms, dtype=np.uint8)[pos].astype(np.float32))
    np.save(os.path.join(out_dir, "superstring_sample_positions.npy"), pos.astype(np.float64))


def ref_binary():
    p = os.path.join(ROOT, "oracle", "_ref", "kmercamel")
    return p if os.path.exists(p) else None


def time_reference(records, n_sample_records: int):
    """The reference's CPU `compute` (oracle/_ref/kmercamel, unmodified sources) on the first n_sample_records records.
    -> (k-mers/s, distinct k-mers, seconds, kind)"""
    from kmercamel_b200 import synth
    sample = records[:n_sample_records]
    exe = ref_binary()
    with tempfile.TemporaryDirectory() as td:
        fa = os.path.join(td, "sample.fa")
        with open(fa, "wb") as f:
            f.write(synth.fasta_bytes(sample))
        if exe:
            t0 = time.perf_counter()
            p = subprocess.run([exe, "compute", "-k", str(K), "-o", os.path.join(td, "out.msfa"), fa], capture_output=True, text=True)
            dt = time.perf_counter() - t0
            if p.returncode == 0:
                n = None
                for ln in p.stderr.splitlines():
                    if "Finished collecting k-mers:" in ln:
                        n = int(ln.split("k-mers:")[1].split()[0])
                return n / dt, n, dt, "reference"
    # oracle/_ref not built (no /root/reference at build time): time the oracle port of stage 1 instead
    from oracle import orc
    seq, off, ln = synth.frame_records(sample)
    t0 = time.perf_counter()
    keys, _ = orc.count_kmers(seq, off, ln, K, True)
    dt = time.perf_counter() - t0
    return len(keys) / dt, len(keys), dt, "port"


def run_reference_arm(args, rank, world):
    if rank != 0:
        return
    records, _ = make_workload(0)
    n_sample = 5  # 5 Mbp per step: ~4 s of single-thread CPU work
    for _ in range(args.warmup if args.warmup < 1 else 1):
        time_reference(records, 1)
    vals, secs, n_k, kind = [], [], 0, "reference"
    for _ in range(args.steps):
        v, n_k, dt, kind = time_reference(records, n_sample)
        vals.append(v)
        secs.append(dt)
    value = n_k * len(secs) / sum(secs)
    sample = f"first {n_sample} of the {N_RECORDS} records ({n_sample * RECORD_LEN / 1e6:.0f} Mbp, {n_k} distinct k-mers) per step; " \
             f"wall clock of `kmercamel compute -k 31` incl. file read and output write"
    ref_cfg = workload_config(world)
    ref_cfg["workload"] += (f" -- REFERENCE ARM SAMPLE: the first {n_sample} of the {N_RECORDS} records ({n_sample} Mbp) per step, the whole `kmercamel compute` "
                            "process incl. file read and output write.  The reference's hash tables slow down with the set size (BASELINE.md: 1.82 M k-mers/s at "
                            "10 Mbp, 1.23 M/s at 50 Mbp), so this sampled rate OVER-states what it reaches on the full 50 Mbp workload: ratios against it are "
                            "conservative.  Like-for-like wall clocks (both CLIs, same file, same box) are in profiles/ (r02_cli_wallclock.json, r02_northstar/)")
    ref_cfg["reference_sample_records"] = n_sample
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1000 * sum(secs) / len(secs), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u64", "data": "synthetic",
        "config": ref_cfg,
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": 1, "kind": kind, "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "host_cores_available": os.cpu_count(),
        "note": "the reference is single-threaded (no threads/OpenMP in its sources): cores = 1 is all it can use",
    }
    print(json.dumps(line), flush=True)


def workload_config(world):
    return {"workload": "BASELINE configs[1]: synthetic 50 Mbp random multi-FASTA (50 x 1 Mbp, default_rng(12345)), "
                        "k=31 canonical, min-one mask, u64 word path" + (f"; x{world}: one genome of {world} x 50 Mbp" if world > 1 else ""),
            "k": K, "bases_per_gpu": N_RECORDS * RECORD_LEN, "records_per_gpu": N_RECORDS,
            "sharding": ("k-mer set construction sharded by hash range of the k-mer SIGNATURE (kmerset_sig.cuh): every rank scans its slice, "
                         "stages super-k-mer records (8 bytes per ~5 windows) per bucket and ships them to the bucket's owner (bucket % N) "
                         "as one dense stream per owner over NVLink (CUDA IPC peer pointers); 2-bit code words and valid-window words of "
                         "the slice go to every rank; ranks synchronise through device-side signal words (no collective and no host round "
                         "trip on the data path), duplicates clear their first-occurrence bit on every rank; every rank repeats the greedy "
                         "merge and emits its own slice of the superstring") if world > 1 else "single GPU",
            "l2": ("inputs larger than L2: the timed steps rotate over 4 device copies of the 50 MB sequence (200 MB) and every step streams "
                   "another ~200 MB of intermediates and output (record rows 141 MB, code words, flags, 50 MB superstring), so a step's input "
                   "was last touched > 500 MB of traffic ago (L2 = 126 MB); no explicit flush") if world == 1 else
                  (f"inputs larger than L2: the job's sequence is {world} x 50 MB on every GPU, and every step streams the staged / shipped / "
                   "gathered records (~3 x 78 MB per GPU), code words, flags and its superstring slice on top; no explicit flush")}


def run_sharded_arm(args, rank, local_rank, world, ctx, part):
    """N > 1: one hash-range sharded job over the concatenation of every rank's 50 Mbp (see the module docstring)."""
    import hashlib
    import torch
    import torch.distributed as dist
    import kmercamel_b200 as kb
    from kmercamel_b200 import sharded

    dev = torch.device("cuda", local_rank)
    stream = torch.cuda.current_stream()
    part_len = int(part.size)                       # identical on every rank (same record count and lengths)
    pinned = torch.from_numpy(part).pin_memory()
    full = torch.empty(world * part_len, dtype=torch.uint8, device=dev)
    own = torch.empty(part_len, dtype=torch.uint8, device=dev)

    def barrier():
        dist.barrier()
        torch.cuda.synchronize()

    def load():                                      # H2D of the rank's own part + all-gather of the parts over NVLink
        own.copy_(pinned, non_blocking=True)
        dist.all_gather_into_tensor(full, own)

    # set-up (not timed): every rank allocates its heap, the 64-byte IPC handles are all-gathered, the heaps are mapped
    sharded.attach(ctx, rank, world, k=K, n_bytes_cap=full.numel(), device=dev)

    def step():  # no collective inside: peer stores over NVLink + device-side signals; every rank emits its own slice of the superstring
        return sharded.sharded_compute(ctx, full.data_ptr(), full.numel(), k=K)

    load()
    for _ in range(max(args.warmup, 3)):
        r = step()
    # ---- parity at N ranks: the concatenated slices against kc_compute_device of the same sequence on ONE GPU (rank 0) ----------
    pad = (r.length // world + 4096 + 15) // 16 * 16
    mine = torch.zeros(pad, dtype=torch.uint8, device=dev)
    assert r.slice_len <= pad
    ctx._check(ctx._lib.kc_copy_to_host(ctx._h, pinned_scratch(pad).data_ptr(), r.ms_ptr, r.slice_len))
    mine[:r.slice_len] = pinned_scratch(pad)[:r.slice_len].to(dev)
    allp = torch.empty(world * pad, dtype=torch.uint8, device=dev)
    dist.all_gather_into_tensor(allp, mine)
    meta = torch.tensor([r.slice_begin, r.slice_len], dtype=torch.int64, device=dev)
    metas = torch.empty(world * 2, dtype=torch.int64, device=dev)
    dist.all_gather_into_tensor(metas, meta)
    parity = None
    if rank == 0:
        metas = metas.cpu().numpy().reshape(world, 2)
        host = allp.cpu().numpy().reshape(world, pad)
        h = hashlib.md5()
        at = 0
        tiles = True
        for i in range(world):
            tiles &= int(metas[i, 0]) == at
            h.update(host[i, :int(metas[i, 1])].tobytes())
            at += int(metas[i, 1])
        single = kb.Context(local_rank)
        want = single.compute_device(full.data_ptr(), full.numel(), k=K)
        want_ms = single.copy_to_host(want.ms_ptr, want.length)
        parity = bool(tiles and at == want.length == r.length and r.n_kmers == want.n_kmers and h.hexdigest() == hashlib.md5(want_ms).hexdigest())
        single.close()
        del want_ms
    del allp, mine
    barrier()

    # headline region without the kernel-class timers, then the same K steps with them (see the single-GPU arm)
    sampler = ClockSampler(local_rank)
    barrier()
    sampler.start()
    launches0 = ctx.total_launches()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(args.steps):
        r = step()
    e1.record(stream)
    barrier()
    dev_ms = e0.elapsed_time(e1)
    launches = ctx.total_launches() - launches0
    ctx.profile_enable(True)
    ctx.profile_reset()
    barrier()
    p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    p0.record(stream)
    for _ in range(args.steps):
        r = step()
    p1.record(stream)
    barrier()
    prof_ms = p0.elapsed_time(p1)
    prof = ctx.profile()
    ctx.profile_enable(False)

    # end to end: pinned host part -> device -> all-gather -> sharded job -> every rank's slice of the superstring back on its host
    host_out = torch.empty(part_len + (1 << 20), dtype=torch.uint8).pin_memory()
    d2h = 0
    for timed in (False, True):
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.steps if timed else 2):
            load()
            r = step()
            assert r.slice_len <= host_out.numel()
            ctx._check(ctx._lib.kc_copy_to_host(ctx._h, host_out.data_ptr(), r.ms_ptr, r.slice_len))
            d2h = r.slice_len
        torch.cuda.synchronize()
        e2e_s = time.perf_counter() - t0
    barrier()
    # the slices must tile the superstring: lengths add up, and each rank's slice carries the mask bits of its own range
    ones = int((host_out[:d2h] <= 90).sum())
    chk = torch.tensor([float(d2h), float(ones)], dtype=torch.float64, device=dev)
    dist.all_reduce(chk, op=dist.ReduceOp.SUM)
    assert int(chk[0]) == r.length and int(chk[1]) == r.n_kmers, (chk.tolist(), r.length, r.n_kmers)
    clocks = sampler.stop()
    fast_runs, fallbacks = ctx.stat("fast_runs"), ctx.stat("fast_fallbacks")

    t = torch.tensor([dev_ms, e2e_s * 1000.0, float(launches), prof_ms], dtype=torch.float64, device=dev)
    tmax = t.clone()
    dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
    tsum = t.clone()
    dist.all_reduce(tsum, op=dist.ReduceOp.SUM)
    ctx.group_close()
    if rank != 0:
        return
    dev_ms, e2e_ms, launches, prof_ms = float(tmax[0]), float(tmax[1]), int(tsum[2]), float(tmax[3])
    n_kmers = r.n_kmers
    value = n_kmers * args.steps / (dev_ms / 1000.0)
    e2e_value = n_kmers * args.steps / (e2e_ms / 1000.0)
    peak, peak_src = measured_peak_gbs()
    dom = max(prof.items(), key=lambda kv: kv[1]["ms"])
    dname, d = dom
    ach = d["bytes"] / (d["ms"] / 1000.0) / 1e9 if d["ms"] > 0 else 0.0
    kernels = {n: {"ms_per_step": v["ms"] / args.steps, "launches_per_step": v["launches"] / args.steps,
                   "gbs": (v["bytes"] / (v["ms"] / 1000.0) / 1e9) if v["ms"] > 0 and v["bytes"] else None}
               for n, v in prof.items() if v["launches"]}
    sig_runs, sig_fb = ctx.stat("sig_runs"), ctx.stat("sig_fallbacks")
    sig_path = sig_runs > 0 and sig_fb == 0
    # what a rank stores into OTHER ranks' heaps per job: signature path = its records (8 bytes per ~5.16 windows) to the owners, plus the
    # 2-bit code words (1/4 byte per base) and flag words (1/8) of its slice to every other rank; fixed-slot path = 12-byte items
    part_windows = r.n_occurrences / world
    if sig_path:
        sent_bytes = part_windows / 5.16 * 8 * (world - 1) / world + part_windows * (0.25 + 0.125) * (world - 1)
    else:
        sent_bytes = part_windows * (world - 1) / world * 12
    s0 = (kernels.get("ks_scatter0", {}).get("ms_per_step") or 0) + ((kernels.get("sort_misc", {}).get("ms_per_step") or 0) if sig_path else 0)
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
        "ms_per_step": dev_ms / args.steps, "ms_per_step_with_kernel_timers": prof_ms / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "u64", "data": "synthetic", "config": workload_config(world),
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": part_len * world, "d2h_bytes_per_step": int(r.length),
                "ms_per_step": e2e_ms / args.steps,
                "timer": "host perf_counter around H2D + all-gather + sharded job + D2H of every rank's superstring slice, max over ranks"},
        "gpu_launches": launches, "clocks": clocks,
        "parity_n": parity,
        "parity_n_check": "md5 of the concatenated per-rank superstring slices == md5 of kc_compute_device of the same sequence on one GPU "
                          "(rank 0), slices tile [0, length), same k-mer count; taken after the warm-up steps",
        "roofline": {"bound": "hbm", "kernel": dname + " (rank 0)", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                     "traffic": None, "peak_source": peak_src, "share_of_step": d["ms"] / prof_ms},
        "cpu_baseline": None, "kernel_classes_rank0": kernels,
        "exchange": {"construction": "signature buckets: records + code words + flag words" if sig_path else "fixed slots: (k-mer, position) items",
                     "nvlink_store_bytes_per_rank_per_step": int(sent_bytes),
                     "nvlink_gbs_during_scan_and_ship_rank0": (sent_bytes / (s0 / 1000.0) / 1e9) if s0 else None,
                     "nvlink_peak_gbs_per_direction": 900.0,
                     "collectives_on_the_data_path": 0, "sig_runs_rank0": sig_runs, "sig_fallbacks_rank0": sig_fb,
                     "fast_runs_rank0": fast_runs, "fast_fallbacks_rank0": fallbacks},
        "result": {"distinct_kmers": int(n_kmers), "superstring_length": int(r.length), "nodes": int(r.n_nodes)},
    }
    _REAL_STDOUT.write(json.dumps(line) + "\n")
    _REAL_STDOUT.flush()


_REAL_STDOUT = sys.stdout
_SCRATCH = {}


def pinned_scratch(n):
    import torch
    if _SCRATCH.get("n", 0) < n:
        _SCRATCH["t"] = torch.empty(n, dtype=torch.uint8).pin_memory()
        _SCRATCH["n"] = n
    return _SCRATCH["t"]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)  # 50 x ~1.5 ms device + 50 x ~3 ms end to end: long enough for the clock sampler
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one returned as DIR/*.npy (see dump_outputs; one GPU only)")
    args = ap.parse_args()
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.dump_outputs and (world > 1 or args.impl != "ours"):
        raise SystemExit("--dump-outputs: only for our path on one GPU")

    if args.impl == "reference":
        run_reference_arm(args, rank, world)
        return

    import torch
    import torch.distributed as dist
    import kmercamel_b200 as kb

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product has no CPU path")
    torch.cuda.set_device(local_rank)
    if world > 1:
        # stdout carries exactly one JSON line.  NCCL writes its version banner (and, with NCCL_DEBUG=INFO, its whole log) to file
        # descriptor 1 from C: point fd 1 at stderr for the lifetime of the process and keep the real stdout for the final line.
        global _REAL_STDOUT
        sys.stdout.flush()
        _REAL_STDOUT = os.fdopen(os.dup(1), "w")
        os.dup2(2, 1)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    records, (seq, off, ln) = make_workload(rank)
    stream = torch.cuda.current_stream()
    ctx = kb.Context(local_rank, stream.cuda_stream)
    if world > 1:
        run_sharded_arm(args, rank, local_rank, world, ctx, seq)
        dist.destroy_process_group()
        return
    d_seq = torch.from_numpy(seq).cuda()
    pinned = torch.from_numpy(seq).pin_memory()
    pinned_np = pinned.numpy()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- device-timed arm (input resident in HBM) ---------------------------------------------------------------
    res = None
    d_seqs = [d_seq] + [d_seq.clone() for _ in range(3)]   # rotated, so that a step never finds its input in L2 (see config.l2)
    for i in range(max(args.warmup, 3)):
        res = ctx.compute_device(d_seqs[i % 4].data_ptr(), d_seq.numel(), k=K)
    # The headline region runs WITHOUT the library's kernel-class timers: they bracket every launch with two event records, which costs
    # ~0.07 ms per step (profiles/prof_overhead.py: 0.85 ms without, 0.93 ms with).  The per-kernel durations the roofline needs are
    # measured by the same CUDA events in a second region of the same K steps, reported as ms_per_step_with_kernel_timers.
    sampler = ClockSampler(local_rank)
    barrier()
    sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sig_runs0 = ctx.stat("sig_runs")
    e0.record(stream)
    launches = 0
    for i in range(args.steps):
        res = ctx.compute_device(d_seqs[i % 4].data_ptr(), d_seq.numel(), k=K)
        launches += res.n_launches
    e1.record(stream)
    barrier()
    dev_ms = e0.elapsed_time(e1)
    if args.dump_outputs:   # the next call reuses the result buffer of the last timed step
        last_ms, last_n_kmers = ctx.copy_to_host(res.ms_ptr, res.length), res.n_kmers
    ctx.profile_enable(True)
    ctx.profile_reset()
    barrier()
    p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    p0.record(stream)
    for i in range(args.steps):
        res = ctx.compute_device(d_seqs[i % 4].data_ptr(), d_seq.numel(), k=K)
    p1.record(stream)
    barrier()
    prof_ms = p0.elapsed_time(p1)
    prof = ctx.profile()
    stage_ms = res.times_ms
    ctx.profile_enable(False)
    sig_path = ctx.stat("sig_runs") - sig_runs0 == 2 * args.steps   # every timed step took the signature-bucket construction
    del d_seqs

    # ---- end-to-end arm (pinned host buffers in, host superstring out) ----------------------------------------
    for _ in range(2):
        r2 = ctx.compute(pinned_np, k=K, copy=False)
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        t1 = time.perf_counter()
        r2 = ctx.compute(pinned_np, k=K, copy=False)
        if os.environ.get("KC_BENCH_DEBUG"):
            print(f"[debug] e2e step {time.perf_counter() - t1:.4f}s stages {r2.times_ms}", file=sys.stderr)
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    barrier()
    clocks = sampler.stop()  # sampled through both timed regions; stopping it earlier stalls the next CUDA calls

    n_kmers = res.n_kmers
    t = torch.tensor([dev_ms, e2e_s * 1000.0, float(n_kmers)], dtype=torch.float64, device="cuda")
    if world > 1:
        tmax = t.clone()
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        tsum = t.clone()
        dist.all_reduce(tsum, op=dist.ReduceOp.SUM)
        dev_ms, e2e_ms, total_kmers = float(tmax[0]), float(tmax[1]), float(tsum[2])
    else:
        dev_ms, e2e_ms, total_kmers = float(t[0]), float(t[1]), float(t[2])

    if rank == 0:
        value = total_kmers * args.steps / (dev_ms / 1000.0)
        e2e_value = total_kmers * args.steps / (e2e_ms / 1000.0)
        peak, peak_src = measured_peak_gbs()
        # dominant kernel class = largest share of device time in the timed region
        dom = max(prof.items(), key=lambda kv: kv[1]["ms"])
        dname, d = dom
        B, M, U, W = float(seq.size), float(res.n_occurrences), float(n_kmers), 8.0
        # ALGORITHMIC bytes per launch = SURVEY.md 8(d)'s per-unit figure x the units one launch processes.  The two kernels of the
        # signature-bucket construction do the work of SURVEY's pack + emit_canonical (scan) and sort / dedup / count (resolve):
        #   scan:    F + B/4 + B/8  +  B/4 + B/8 + M W        resolve:  M W + U (W + 1)   (all radix passes charged as ONE read + ONE write)
        # Other kernel classes keep the bytes the library declares at launch (inputs read once + outputs written once).
        alg_8d = {"ks_scatter0": (B + B / 4 + B / 8) + (B / 4 + B / 8 + M * W), "ks_resolve": M * W + U * (W + 1)} if sig_path else {}
        def alg_bytes(name, v):
            return alg_8d.get(name, v["bytes"] / max(v["launches"], 1))
        ach = alg_bytes(dname, d) / (d["ms"] / max(d["launches"], 1) / 1000.0) / 1e9 if d["ms"] > 0 else 0.0
        traffic, tj = None, {}
        tpath = os.path.join(ROOT, "profiles", "traffic.json")
        if os.path.exists(tpath):
            try:
                tj = json.load(open(tpath))
                tj = tj.get("signature_buckets", {}) if sig_path else tj
                traffic = tj.get(dname)
            except Exception:
                traffic, tj = None, {}
        roofline = {"bound": "hbm", "kernel": dname + (" = kc_sig_resolve_kernel" if sig_path and dname == "ks_resolve" else
                                                        " = kc_sig_scan_kernel" if sig_path and dname == "ks_scatter0" else ""),
                    "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                    "traffic": traffic, "peak_source": peak_src,
                    "launches_per_step": d["launches"] / args.steps, "ms_per_launch": d["ms"] / max(d["launches"], 1),
                    "algorithmic_bytes_per_launch": alg_bytes(dname, d),
                    "algorithmic_bytes_are": "SURVEY 8(d): sort/dedup/count = M W + U (W + 1) per launch" if sig_path and dname == "ks_resolve" else
                                             "SURVEY 8(d): pack + emit_canonical = F + B/2 + B/4 + M W per launch" if sig_path and dname == "ks_scatter0" else
                                             "inputs read once + outputs written once, declared by the library at launch",
                    "share_of_step": d["ms"] / prof_ms,
                    "limiter": ("instruction issue, not HBM: the kernel re-creates the k-mers from 2-bit code words instead of moving them "
                                "(ncu profiles/r02z_final_ncu.md: DRAM 5-9 % of peak, SM throughput 53-54 %); `traffic` = measured DRAM bytes per launch")
                               if sig_path else None}
        if sig_path:
            roofline["per_kernel_8d"] = {c: {"algorithmic_bytes": alg_8d[c], "ms": prof[c]["ms"] / max(prof[c]["launches"], 1),
                                             "frac": alg_8d[c] / (prof[c]["ms"] / max(prof[c]["launches"], 1) / 1000.0) / 1e9 / peak,
                                             "dram_bytes_ncu": tj.get(c)}
                                         for c in ("ks_scatter0", "ks_resolve") if c in prof and prof[c]["ms"] > 0}
        # SURVEY.md §8(d) accounting next to the per-pass one: the k-mer set stage (pack + emit_canonical + sort / dedup / count) is charged
        # F + B/4 + B/8  +  B/4 + B/8 + M W  +  M W + U (W + 1) bytes — every radix pass together as ONE read + ONE write — over the time of
        # the three kernels that do that work here (level-0 partition, level-1 partition, leaf resolve); and the whole step is charged
        # SURVEY's ~60 B per distinct k-mer.  The per-kernel fractions by measured DRAM bytes come from the ncu capture (profiles/traffic.json).
        set_ms = sum(prof[c]["ms"] for c in ("ks_scatter0", "sort_scatter", "ks_resolve") if c in prof) / args.steps
        bytes_8d = (B + B / 4 + B / 8) + (B / 4 + B / 8 + M * W) + (M * W + U * (W + 1))
        roofline["stage_8d"] = {"stage": "k-mer set (pack + emit_canonical + sort/dedup/count of SURVEY 8d = ks_scatter0 + sort_scatter + ks_resolve here)",
                                "algorithmic_bytes": bytes_8d, "ms": set_ms, "achieved": bytes_8d / (set_ms / 1000.0) / 1e9 if set_ms else None,
                                "frac": bytes_8d / (set_ms / 1000.0) / 1e9 / peak if set_ms else None}
        roofline["step_8d"] = {"algorithmic_bytes": 60.0 * U, "ms": dev_ms / args.steps, "frac": 60.0 * U / (dev_ms / args.steps / 1000.0) / 1e9 / peak}
        try:
            roofline["frac_by_dram_bytes"] = {c: (tj[c] / (prof[c]["ms"] / max(prof[c]["launches"], 1) / 1000.0) / 1e9 / peak)
                                              for c in ("ks_scatter0", "sort_scatter", "ks_resolve") if c in tj and c in prof and prof[c]["ms"] > 0}
        except Exception:
            pass
        kernels = {n: {"ms_per_step": v["ms"] / args.steps, "launches_per_step": v["launches"] / args.steps,
                       "gbs": (v["bytes"] / (v["ms"] / 1000.0) / 1e9) if v["ms"] > 0 and v["bytes"] else None}
                   for n, v in prof.items() if v["launches"]}
        cpu = None
        if not args.no_cpu_baseline and world == 1:
            v, n_k, dt, kind = time_reference(records, 10)
            cpu = {"value": v, "unit": UNIT, "cores": 1, "kind": kind,
                   "sample": f"first 10 of the 50 records (10 Mbp, {n_k} distinct k-mers): `kmercamel compute -k 31` wall "
                             f"clock {dt:.1f} s on one host core (the reference is single-threaded; {os.cpu_count()} cores present)"}
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": dev_ms / args.steps, "ms_per_step_with_kernel_timers": prof_ms / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "u64", "data": "synthetic", "config": workload_config(world),
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(seq.size), "d2h_bytes_per_step": int(r2.length),
                    "ms_per_step": e2e_ms / args.steps, "timer": "host perf_counter around kc_compute (stream-synchronous), max over ranks"},
            "gpu_launches": int(launches), "clocks": clocks, "roofline": roofline, "cpu_baseline": cpu,
            "stage_ms_last_step": stage_ms, "kernel_classes": kernels,
            "result": {"distinct_kmers_per_gpu": int(n_kmers), "superstring_length": int(res.length), "nodes": int(res.n_nodes),
                       "kmer_set_construction": "signature buckets (kmerset_sig.cuh)" if sig_path else "fixed slots / exact (kmerset_fast.cuh, kmerset.cuh)",
                       "sig_fallbacks": int(ctx.stat("sig_fallbacks"))},
        }
        print(json.dumps(line), flush=True)
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, last_ms, last_n_kmers)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
