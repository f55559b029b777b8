#!/usr/bin/env python3
"""Per-call parity of the C ABI: one seeded input per entry point and route, and what each call leaves behind.

For every case it records the hash of the output bytes, n_launches, the change of the context's statistics (read-backs, launches,
construction runs and fallbacks, speculative tail, arena retries and high-water mark, overlap stage), the return code and the error
text without its " (file:line)" suffix.  A change that only moves host code must leave the JSON file as it was: run this once per
build and diff the two files.

    python profiles/call_parity.py OUT.json [--root TREE]    # TREE: the checkout whose kmercamel_b200 is loaded (default: this one)

Needs one GPU with ~120 GB free for the group's refusal of an input of 2^32 bytes or more (two ranks share device 0); with less, that
case is recorded as skipped.
"""
import argparse
import hashlib
import json
import os
import re
import sys

import numpy as np

STATS = ["read_backs", "total_launches", "sig_runs", "sig_fallbacks", "fast_runs", "fast_fallbacks", "tail_spec_runs",
         "tail_spec_fallbacks", "arena_retries", "arena_high", "path_levels", "path_ban_rounds", "path_bans"]
ACGT = np.frombuffer(b"ACGT", dtype=np.uint8)


def h(*parts):
    d = hashlib.sha256()
    for p in parts:
        d.update(b"-" if p is None else (p if isinstance(p, bytes) else np.ascontiguousarray(p).tobytes()))
    return d.hexdigest()[:32]


def frame(records):
    seq = b"".join(r + b"\n" for r in records)
    off, o = [], 0
    for r in records:
        off.append(o)
        o += len(r) + 1
    return (np.frombuffer(seq, dtype=np.uint8).copy(), np.array(off, dtype=np.uint64),
            np.array([len(r) for r in records], dtype=np.uint64))


def random_bases(rng, n):
    return ACGT[rng.integers(0, 4, n)].tobytes()


def mutate(rng, s, rate):
    a = np.frombuffer(s, dtype=np.uint8).copy()
    at = rng.random(a.size) < rate
    a[at] = ACGT[rng.integers(0, 4, int(at.sum()))]
    return a.tobytes()


def inputs():
    rng = np.random.default_rng(20261022)
    genome = [random_bases(rng, 50_000) for _ in range(4)]
    genome.append(genome[0][1000:3000])
    reads = []
    for _ in range(3000):  # ~4x coverage of the first record, 1 % errors: repeated k-mers for -z, many runs for the fixed slots
        s = int(rng.integers(0, 50_000 - 150))
        reads.append(mutate(rng, genome[0][s:s + 150], 0.01))
    simplitigs = [g[:200] for g in genome[:4]] + [genome[1][150:420]]
    return dict(genome=frame(genome), reads=frame(genome + reads), simplitigs=frame(simplitigs),
                big=frame([random_bases(rng, 12 << 20)]), empty=frame([b"N" * 100]), bad_s=frame([b"ACGTNACGT" * 10]))


def strip_site(msg):
    return re.sub(r" \([^()]*:\d+\)$", "", msg)


def run_case(ctx_or_group, fn):
    is_group = not hasattr(ctx_or_group, "_h")
    stat = ctx_or_group.stat
    s0 = {n: stat(n) for n in STATS}
    rec = {}
    try:
        rec.update(fn())
        rec["code"] = 0
    except kb.KcError as e:
        rec["code"] = e.code
        rec["error"] = strip_site(str(e))
    s1 = {n: stat(n) for n in STATS}
    if is_group:
        rec["stats"] = {n: [b - a for a, b in zip(s0[n], s1[n])] for n in STATS}
    else:
        rec["stats"] = {n: s1[n] - s0[n] for n in STATS}
    return rec


def result(r):
    return dict(out=h(r.ms, r.maxone), length=r.length, n_kmers=r.n_kmers, n_occ=r.n_occurrences, n_nodes=r.n_nodes,
                n_simplitigs=r.n_simplitigs, n_launches=r.n_launches)


def single_cases(d, torch):
    g_seq = d["genome"][0]
    r_seq = d["reads"][0]
    s_seq, s_off, s_len = d["simplitigs"]
    cases = {}

    def compute(seq, opts=None, *a, **kw):
        return (opts or {}), lambda c: result(c.compute(seq, *a, **kw))

    sig = dict(sig_min_items=0)
    cases["compute_sig_tail"] = compute(g_seq, sig, k=31)
    cases["compute_sig_no_tail"] = compute(g_seq, dict(sig, tail_spec=0), k=31)
    cases["compute_sig_overflow_fast"] = compute(r_seq, dict(sig, sig_load_pct=400, fast_min_items=0, fast_heuristics=0), k=31)
    cases["compute_fast_overflow_exact"] = compute(r_seq, dict(sig_set=0, fast_min_items=0, fast_leaf_target=16, fast_sigmas=0,
                                                               fast_heuristics=0), k=31)
    cases["compute_fast"] = compute(r_seq, dict(sig_set=0, fast_min_items=0, fast_heuristics=0), k=31)
    cases["compute_M"] = compute(r_seq, {}, k=31, want_maxone=True)
    cases["compute_S"] = compute(s_seq, {}, s_off, s_len, k=31, assume_simplitigs=True)
    cases["compute_S_M"] = compute(s_seq, {}, s_off, s_len, k=31, assume_simplitigs=True, want_maxone=True)
    cases["compute_z2"] = compute(r_seq, {}, k=31, min_frequency=2)
    cases["compute_k21"] = compute(r_seq, {}, k=21)
    cases["compute_k63_u"] = compute(r_seq, {}, k=63, complements=False)
    cases["compute_k127"] = compute(g_seq, sig, k=127)
    cases["compute_arena_retry"] = compute(r_seq, dict(arena_estimate_ppm=1_000, tail_spec=0), k=31)
    cases["compute_chunked_upload"] = compute(d["big"][0], {}, k=31)
    cases["compute_empty"] = compute(d["empty"][0], {}, k=31)
    cases["compute_S_bad_seq"] = compute(d["bad_s"][0], {}, d["bad_s"][1], d["bad_s"][2], k=31, assume_simplitigs=True)

    def compute_device(c):
        t = torch.from_numpy(r_seq).cuda()
        r = c.compute_device(t.data_ptr(), t.numel(), k=31)
        out = result(r)
        out["out"] = h(c.copy_to_host(r.ms_ptr, r.length))
        return out
    cases["compute_device"] = ({}, compute_device)

    def lower_bound(*a, **kw):
        def f(c):
            lb, st = c.lower_bound(*a, **kw)
            return dict(lb=int(lb), n_kmers=st.n_kmers, n_nodes=st.n_nodes, n_simplitigs=st.n_simplitigs, n_launches=st.n_launches,
                        length=st.length)
        return {}, f
    cases["lowerbound"] = lower_bound(r_seq, k=31)
    cases["lowerbound_S"] = lower_bound(s_seq, s_off, s_len, k=31, assume_simplitigs=True)
    for z in (1, 3):
        cases[f"streaming_z{z}"] = ({}, lambda c, z=z: result(c.streaming(r_seq, k=31, min_frequency=z)))

    def maskopt(minimize):
        def f(c):
            ms = c.compute(r_seq, k=31).ms
            return result(c.maskopt(ms, k=31, minimize=minimize))
        return {}, f
    cases["maskopt_min"] = maskopt(True)
    cases["maskopt_max"] = maskopt(False)

    def count(c):
        keys, vals = c.count_kmers(r_seq, k=31)
        return dict(out=h(keys, vals), n=int(len(vals)))
    cases["count_kmers"] = ({}, count)

    def digest(masked=False, z=1):
        def f(c):
            seq = np.frombuffer(c.compute(r_seq, k=31).ms, dtype=np.uint8) if masked else r_seq
            return dict(digest=[int(x) for x in c.kmer_digest(seq, k=31, min_frequency=z, masked=masked)])
        return {}, f
    cases["digest"] = digest()
    cases["digest_masked"] = digest(masked=True)
    cases["digest_z2"] = digest(z=2)

    rng = np.random.default_rng(7)
    first = rng.integers(0, 1 << 62, (2000, 1), dtype=np.uint64)
    last = first.copy()
    last[:1000] = first[1000:]  # overlaps to find

    def overlap(c):
        ef, ov = c.overlap_path(first, last, k=31)
        return dict(out=h(ef, ov))
    cases["overlap_path"] = ({}, overlap)
    kmers = rng.integers(0, 1 << 62, (5000, 1), dtype=np.uint64)
    cases["partial_presort"] = ({}, lambda c: dict(out=h(c.partial_presort(kmers, k=31))))
    words = rng.integers(0, 1 << 62, (5000, 2), dtype=np.uint64)
    words[:, 1] &= (1 << 36) - 1

    def debug_sort(c):
        out, st = c.debug_sort(words, 100)
        return dict(out=h(out), sort_stats=st)
    cases["debug_sort"] = ({}, debug_sort)
    return cases


def big_input(overflow):
    """As in tests/test_gpu_group_positions64.py: A, N up to 4 Mbp before byte 2^32, B, newline (A and B random, 8 Mbp each); with
    `overflow` a repeat-rich stretch after A (300 copies of 2 kbp) overflows the signature buckets."""
    part = 8 << 20
    rng = np.random.default_rng(20261020)
    a = np.frombuffer(random_bases(rng, part), dtype=np.uint8)
    b = np.frombuffer(random_bases(rng, part), dtype=np.uint8)
    gap = 2**32 - (4 << 20) - part
    big = np.full(part + gap + part + 1, ord("N"), dtype=np.uint8)
    big[:part] = a
    big[part + gap:part + gap + part] = b
    big[-1] = ord("\n")
    if overflow:
        rep = np.tile(np.concatenate([a[:2000], np.array([ord("N")], dtype=np.uint8)]), 300)
        big[part + 16:part + 16 + rep.size] = rep
    return big


def group_cases(d, torch):
    r_seq = d["reads"][0]
    cases = [("group_sig", dict(sig_min_items=0), lambda g: result(g.compute(r_seq, k=31))),
             ("group_fast", dict(sig_set=0, fast_min_items=0), lambda g: result(g.compute(r_seq, k=31))),
             ("group_exact", dict(sig_set=0, fast_set=0), lambda g: result(g.compute(r_seq, k=31))),
             ("group_empty", {}, lambda g: result(g.compute(d["empty"][0], k=31))),
             ("group_large_k21", {}, lambda g: result(g.compute(big_input(False), k=21)))]
    free, _ = torch.cuda.mem_get_info(0)
    if free >= 120e9:
        cases.append(("group_large_overflow", {}, lambda g: result(g.compute(big_input(True), k=31))))
    else:
        cases.append(("group_large_overflow", None, None))
    return cases


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("out")
    ap.add_argument("--root", default=os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    args = ap.parse_args()
    sys.path.insert(0, os.path.abspath(args.root))
    global kb
    import kmercamel_b200 as kb
    import torch
    d = inputs()
    res = {}
    for name, (opts, fn) in single_cases(d, torch).items():
        c = kb.Context(0)
        for o, v in opts.items():
            c.set_option(o, v)
        res[name] = run_case(c, lambda: fn(c))
        c.close()
        print(name, res[name].get("code"), flush=True)
    for name, opts, fn in group_cases(d, torch):
        if fn is None:
            res[name] = "skipped: needs 120 GB of free device memory"
            continue
        g = kb.Group([0, 0])
        for o, v in opts.items():
            g.set_option(o, v)
        res[name] = run_case(g, lambda: fn(g))
        res[name + "_then_good"] = run_case(g, lambda: result(g.compute(d["genome"][0], k=31)))
        g.close()
        print(name, res[name].get("code"), res[name + "_then_good"].get("code"), flush=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1, sort_keys=True)


if __name__ == "__main__":
    main()
