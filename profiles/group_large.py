"""Inputs of 2^32 bytes or more on one GPU and on groups: `kc_compute` against `kc_group_compute` on 1, 2, 4 and 8 distinct devices
(as many as are visible), k = 31, canonical.

Input (generated on the device from a seed): two haplotypes of a uniform random genome, 24 records of human-like relative lengths
per haplotype, the second a copy of the first with 0.1 % i.i.d. substitutions; 2 x 2.25 Gbp = 4.5 GB framed.  Every group result
is compared byte for byte with the one-GPU result.

    python profiles/group_large.py [--out FILE] [--repeats N]   ->  JSON (default profiles/group_large.json) and one line on stdout
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

import kmercamel_b200 as kb  # noqa: E402

K = 31
HAPLOTYPE = 2_250_000_000
# relative lengths of the 24 human chromosomes (1..22, X, Y), as in synth.human_like_genome
CHROM = [248956422, 242193529, 198295559, 190214555, 181538259, 170805979, 159345973, 145138636, 138394717, 133797422, 135086622,
         133275309, 114364328, 107043718, 101991189, 90338345, 83257441, 80373285, 58617616, 64444167, 46709983, 50818468, 156040895,
         57227415]


def make_input(seed=4500):
    g = torch.Generator(device="cuda")
    g.manual_seed(seed)
    lut = torch.tensor(list(b"ACGT"), dtype=torch.uint8, device="cuda")
    lens = [int(HAPLOTYPE * c / sum(CHROM)) for c in CHROM]
    lens[-1] += HAPLOTYPE - sum(lens)
    hap_a = lut[torch.randint(0, 4, (HAPLOTYPE,), dtype=torch.uint8, device="cuda", generator=g).long()]
    hap_b = hap_a.clone()
    n_sub = HAPLOTYPE // 1000
    at = torch.randint(0, HAPLOTYPE, (n_sub,), device="cuda", generator=g)
    shift = torch.randint(1, 4, (n_sub,), dtype=torch.uint8, device="cuda", generator=g)
    code = torch.zeros(256, dtype=torch.uint8, device="cuda")
    for i, c in enumerate(b"ACGT"):
        code[c] = i
    hap_b[at] = lut[((code[hap_b[at].long()] + shift) % 4).long()]
    del at, shift
    seq = torch.empty(2 * (HAPLOTYPE + len(lens)), dtype=torch.uint8, device="cuda")
    o = 0
    for hap in (hap_a, hap_b):
        s = 0
        for ln in lens:
            seq[o:o + ln] = hap[s:s + ln]
            seq[o + ln] = ord("\n")
            o += ln + 1
            s += ln
    assert o == seq.numel() and seq.numel() >= 2**32
    host = seq.cpu().numpy()
    del seq, hap_a, hap_b
    torch.cuda.empty_cache()
    return host


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=index,name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return [line.strip() for line in q.stdout.strip().splitlines()]


def timed(call, repeats):
    runs, res = [], None
    for _ in range(repeats + 1):  # the first call also reserves arenas and heaps
        t0 = time.perf_counter()
        res = call()
        runs.append(dict(wall_ms=round((time.perf_counter() - t0) * 1e3, 1), **{s: round(v, 3) for s, v in res.times_ms.items()}))
    return res, runs


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "group_large.json"))
    ap.add_argument("--repeats", type=int, default=2)
    a = ap.parse_args()
    n_dev = torch.cuda.device_count()
    seq = make_input()
    rows = []
    ctx = kb.Context(0)
    one, runs = timed(lambda: ctx.compute(seq, k=K), a.repeats)
    rows.append(dict(what="kc_compute", devices=[0], first_call=runs[0], timed=runs[1:], sig_runs=[ctx.stat("sig_runs")],
                     sig_fallbacks=[ctx.stat("sig_fallbacks")]))
    ctx.close()
    for n in (1, 2, 4, 8):
        if n > n_dev:
            rows.append(dict(what="kc_group_compute", n_ranks=n, devices=None, note=f"not measured: {n_dev} device(s) visible"))
            continue
        grp = kb.Group(list(range(n)))
        got, runs = timed(lambda: grp.compute(seq, k=K), a.repeats)
        rows.append(dict(what="kc_group_compute", n_ranks=n, devices=list(range(n)), first_call=runs[0], timed=runs[1:],
                         sig_runs=grp.stat("sig_runs"), sig_fallbacks=grp.stat("sig_fallbacks"),
                         identical=got.ms == one.ms and got.n_kmers == one.n_kmers and got.length == one.length))
        grp.close()
    out = dict(workload=f"k={K}, canonical, two haplotypes of a uniform random genome (24 records each, 0.1 % substitutions), "
                        f"{seq.size} bytes framed, torch seed 4500", n_bytes=int(seq.size), n_kmers=int(one.n_kmers), length=int(one.length),
               gpus=card(), rows=rows)
    with open(a.out, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps(dict(gpus=out["gpus"], rows=[{k: r.get(k) for k in ("what", "n_ranks", "identical", "note")} |
                                                   ({"wall_ms_min": min(x["wall_ms"] for x in r["timed"])} if "timed" in r else {}) for r in rows])))


if __name__ == "__main__":
    main()
