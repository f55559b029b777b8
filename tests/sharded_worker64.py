"""Worker of tests/test_gpu_group_positions64.py::test_torchrun_processes_past_2_32 (launched through torch.distributed.run).

Every rank is a process with its own libkcgpu context and its own copy of the big input of test_gpu_positions64.py (generated on
its device from the same seed); the heaps are allocated for a cap above 2^32 and mapped into each other through CUDA IPC handles
(gathered over gloo, so that both ranks may share one GPU).  Rank 0 compares the concatenated slices with kc_compute_device on one
GPU over the small input and writes the verdict.  KC_TEST_POISON >= 0 sets option arena_poison on the group context."""
import json
import os
import sys

import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import kmercamel_b200 as kb  # noqa: E402
from kmercamel_b200 import sharded  # noqa: E402
from test_gpu_positions64 import inputs  # noqa: E402


def main():
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    dist.init_process_group("gloo", rank=rank, world_size=world)
    dev = int(os.environ.get("LOCAL_RANK", "0")) % torch.cuda.device_count()
    torch.cuda.set_device(dev)
    gen = inputs.__wrapped__()  # the fixture's generator: big, small
    big, small = next(gen)
    ctx = kb.Context(dev, torch.cuda.current_stream().cuda_stream)
    poison = int(os.environ.get("KC_TEST_POISON", "-1"))
    if poison >= 0:
        ctx.set_option("arena_poison", poison)
    sharded.attach(ctx, rank, world, k=31, n_bytes_cap=big.numel() + (1 << 20))
    r = sharded.sharded_compute(ctx, big.data_ptr(), big.numel(), k=31)
    part = torch.frombuffer(bytearray(ctx.copy_to_host(r.ms_ptr, r.slice_len)), dtype=torch.uint8)
    meta = torch.tensor([r.slice_begin, r.slice_len, r.length, r.n_kmers], dtype=torch.int64)
    metas = [torch.empty_like(meta) for _ in range(world)]
    dist.all_gather(metas, meta)
    buf = torch.zeros(int(r.length) + 64, dtype=torch.uint8)
    buf[r.slice_begin:r.slice_begin + r.slice_len] = part
    dist.all_reduce(buf, op=dist.ReduceOp.SUM)  # disjoint slices: SUM == concatenation
    ok = True
    verdict = {}
    if rank == 0:
        single = kb.Context(dev)
        want = single.compute_device(small.data_ptr(), small.numel(), k=31)
        want_ms = single.copy_to_host(want.ms_ptr, want.length)
        at = 0
        for m in metas:
            ok &= int(m[0]) == at and int(m[2]) == want.length and int(m[3]) == want.n_kmers
            at += int(m[1])
        ok &= at == want.length and buf[:want.length].numpy().tobytes() == want_ms
        verdict = {"world": world, "identical": bool(ok), "length": int(want.length), "n_kmers": int(want.n_kmers),
                   "sig_runs": ctx.stat("sig_runs"), "devices": torch.cuda.device_count(), "poison": poison}
        single.close()
    dist.barrier()
    ctx.group_close()
    if rank == 0:
        json.dump(verdict, open(sys.argv[1], "w"))
    dist.destroy_process_group()
    sys.exit(0 if ok else 1)


if __name__ == "__main__":
    main()
