"""Multi-GPU check of the NVLS all-reduce kernel (csrc/collective.cu) against NCCL, plus timing.

    torchrun --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 tools/nvls_check.py
"""
import os
import sys

import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from dmesh_renderer_b200.multiview import PackedSceneGrads  # noqa: E402

rank, local, ws = int(os.environ["RANK"]), int(os.environ["LOCAL_RANK"]), int(os.environ["WORLD_SIZE"])
torch.cuda.set_device(local)
dev = torch.device("cuda", local)
dist.init_process_group("nccl", device_id=dev)
# scene size: C2 by default, `nvls_check.py C4` for the 76 MB buffer of the multi-view configuration
P, F = (3_000_000, 1_000_000) if len(sys.argv) > 1 and sys.argv[1] == "C4" else (600_000, 200_000)
g = PackedSceneGrads(torch.zeros(P, 3, device=dev), torch.zeros(P, 3, device=dev), torch.zeros(F, device=dev))
if rank == 0:
    print("NVLS path:", g._nvls is not None, "| collective:", g.collective, "| floats", g.flat.numel(), "padded", g._full.numel(), flush=True)
gen = torch.Generator(device=dev).manual_seed(100 + rank)
for trial in range(3):
    x = torch.randn(g.flat.numel(), device=dev, generator=gen)
    ref = x.clone()
    dist.all_reduce(ref)
    g.flat.copy_(x)
    g.all_reduce()
    torch.cuda.synchronize()
    err = (g.flat - ref).abs().max().item()
    rel = ((g.flat - ref).norm() / ref.norm()).item()
    pad_ok = bool((g._full[g.flat.numel():] == 0).all().item())
    if rank == 0:
        print("trial %d: max abs diff vs NCCL %.3e, rel L2 %.3e, padding zero %s" % (trial, err, rel, pad_ok), flush=True)
    assert rel < 1e-6 and pad_ok
    if g._nvls is not None and rank == 0:
        print("trial %d bit-identical to NCCL: %s" % (trial, bool(torch.equal(g.flat, ref))), flush=True)


def timeit(fn, n=50):
    for _ in range(10):
        fn()
    torch.cuda.synchronize()
    dist.barrier()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(n):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / n * 1e3


t_fused = timeit(g.all_reduce)
t_nccl = timeit(lambda: dist.all_reduce(g.flat))
if rank == 0:
    print("all-reduce of %.1f MB on %d GPUs: NVLS kernel with in-kernel barriers %.1f us, NCCL %.1f us"
          % (g.flat.numel() * 4 / 1e6, ws, t_fused, t_nccl), flush=True)
dist.destroy_process_group()
