"""Wall time of the neighbours of `compute` through the signature construction, on one GPU:
  * at 4.4 Gbases (k = 63, 44 x 100 Mbp uniform random records, seed 44, the input of profiles/big_positions64.py): kc_kmer_digest of
    the input, kc_kmer_digest (masked) of its superstring, kc_lower_bound and kc_streaming;
  * at 50 Mbp (the same generator, 5 x 10 Mbp): kc_kmer_digest with option sig_set = 1 against sig_set = 0, alternating.
Every call goes through host buffers (what the CLI does), so the times include the host -> device copy.  The card name and power limit
are read in the same run.

    python profiles/large_neighbours.py [repeats]  ->  one JSON line on stdout
"""
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


def genome(n_rec, rec_len, seed):
    g = torch.Generator(device="cuda")
    g.manual_seed(seed)
    lut = torch.tensor(list(b"ACGT"), dtype=torch.uint8, device="cuda")
    seq = torch.empty(n_rec * (rec_len + 1), dtype=torch.uint8, device="cuda")
    for i in range(n_rec):
        o = i * (rec_len + 1)
        seq[o:o + rec_len] = lut[torch.randint(0, 4, (rec_len,), dtype=torch.uint8, device="cuda", generator=g).long()]
        seq[o + rec_len] = ord("\n")
    host = seq.cpu().numpy()
    del seq
    torch.cuda.empty_cache()
    return host


def timed(f, repeats):
    out = []
    for _ in range(repeats):
        t0 = time.perf_counter()
        v = f()
        out.append(round((time.perf_counter() - t0) * 1e3, 2))
    return v, out


def main():
    repeats = int(sys.argv[1]) if len(sys.argv) > 1 else 3
    ctx = kb.Context(0)
    res = {}
    # 50 Mbp: digest by signature route (1) and by sorted keys (0), alternating, after one warm-up call of each
    small = genome(5, 10_000_000, 50)
    ctx.set_option("sig_set", 1)
    ctx.kmer_digest(small, k=31)
    ctx.set_option("sig_set", 0)
    ctx.kmer_digest(small, k=31)
    t = {1: [], 0: []}
    for _ in range(repeats):
        for s in (1, 0):
            ctx.set_option("sig_set", s)
            d, ms = timed(lambda: ctx.kmer_digest(small, k=31), 1)
            t[s] += ms
    ctx.set_option("sig_set", 1)
    res["digest_50mbp_k31_ms"] = {"sig_set_1": t[1], "sig_set_0": t[0]}
    del small
    # 4.4 Gbases, k = 63
    k = 63
    big = genome(44, 100_000_000, 44)
    r = ctx.compute(big, k=k)
    ms = np.frombuffer(r.ms, dtype=np.uint8).copy()
    d_in, res["digest_4g4_ms"] = timed(lambda: ctx.kmer_digest(big, k=k), repeats)
    d_out, res["digest_masked_4g4_ms"] = timed(lambda: ctx.kmer_digest(ms, k=k, masked=True), repeats)
    (lb, _), res["lowerbound_4g4_ms"] = timed(lambda: ctx.lower_bound(big, k=k), repeats)
    st, res["streaming_4g4_ms"] = timed(lambda: ctx.streaming(big, k=k, copy=False), repeats)
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    res.update(workload_4g4=f"k={k}, canonical, 44 x 100 Mbp uniform random records (torch seed 44), host buffers",
               workload_50mbp="k=31, canonical, 5 x 10 Mbp uniform random records (torch seed 50), host buffers",
               n_bytes=int(big.size), n_kmers=r.n_kmers, superstring_length=r.length, digest_matches=d_in == d_out,
               digest_n=d_in[0], lower_bound=lb, streaming_length=st.length, sig_runs=ctx.stat("sig_runs"),
               sig_fallbacks=ctx.stat("sig_fallbacks"), arena_high_bytes=ctx.stat("arena_high"), gpu=smi[0] if smi else "unknown")
    ctx.close()
    print(json.dumps(res))


if __name__ == "__main__":
    main()
