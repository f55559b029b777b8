"""One line of device time and arena bytes for `compute` on 4.4 Gbases (k = 63, 44 x 100 Mbp uniform random records, seed 44;
the input of tests/test_gpu_positions64.py::test_4_4_gbases_genome_by_additive_digests), on one GPU: window positions past 2^32.

    python profiles/big_positions64.py [repeats]  ->  one JSON line on stdout
"""
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

import kmercamel_b200 as kb  # noqa: E402


def main():
    repeats = int(sys.argv[1]) if len(sys.argv) > 1 else 3
    k, n_rec, rec_len = 63, 44, 100_000_000
    g = torch.Generator(device="cuda")
    g.manual_seed(44)
    lut = torch.tensor(list(b"ACGT"), dtype=torch.uint8, device="cuda")
    seq = torch.empty(n_rec * (rec_len + 1), dtype=torch.uint8, device="cuda")
    for i in range(n_rec):
        o = i * (rec_len + 1)
        seq[o:o + rec_len] = lut[torch.randint(0, 4, (rec_len,), dtype=torch.uint8, device="cuda", generator=g).long()]
        seq[o + rec_len] = ord("\n")
    torch.cuda.synchronize()
    ctx = kb.Context(0)
    runs = []
    for _ in range(repeats + 1):  # the first call also reserves the arena
        t0 = time.perf_counter()
        r = ctx.compute_device(seq.data_ptr(), seq.numel(), k=k)
        runs.append(dict(wall_ms=(time.perf_counter() - t0) * 1e3, **{s: round(v, 3) for s, v in r.times_ms.items()}))
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    out = dict(workload=f"compute_device, k={k}, canonical, {n_rec} x {rec_len} bp uniform random records (torch seed 44)",
               n_bytes=seq.numel(), n_kmers=r.n_kmers, length=r.length, n_nodes=r.n_nodes, sig_runs=ctx.stat("sig_runs"),
               arena_reserved_bytes=ctx.stat("arena_bytes"), arena_high_bytes=ctx.stat("arena_high"),
               first_call=runs[0], timed=runs[1:], device_total_ms_min=min(x["total"] for x in runs[1:]),
               gpu=smi[0] if smi else "unknown")
    ctx.close()
    print(json.dumps(out))


if __name__ == "__main__":
    main()
