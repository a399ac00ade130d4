"""Views per second of one tet multi-view optimisation step (multiview.tet_multiview_step).

    python tools/tet_multiview_timing.py [--steps 5] [--rounds 5] [--warmup 2] [--seed 0] [--out FILE]     (1 GPU)
    torchrun --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 tools/tet_multiview_timing.py [...]  (N GPUs)

Scene: C3's geometry (the 64^3 Kuhn grid, P = 274,625, F = 3,170,304, 512^2) seen by 64 Fibonacci-sphere cameras
(scenes.tet_grid_scene(..., B=64)); every rank renders its shard_views() slice, `--views-per-call` views per call
(default 8), with the packed [dL_dvcolor | dL_dfopacity] buffer (3P + F floats) as the direct gradient sink and one
all-reduce per step.  Fixed seeded cotangents stand in for the loss.  A step is timed with CUDA events over --steps
steps, ending in a device synchronise; each of --rounds rounds gives one time per rank, and the step time of a round
is the slowest rank's.  On one GPU the same step is also timed with plain autograd accumulation (fresh gradient
tensors every call, added to .grad by autograd, .grad reset to None every step), alternating with the direct sink
round by round.  Rank 0 prints one JSON object with the card's name and power limit.
"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

from camera_grad_timing import card  # noqa: E402
from dmesh_renderer_b200 import TetRenderer, TetRenderSettings, scenes  # noqa: E402
from dmesh_renderer_b200.multiview import PackedSceneGrads, shard_views, tet_multiview_step  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--views", type=int, default=64)
    ap.add_argument("--views-per-call", type=int, default=8)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--seed", type=int, default=0, help="ray_random_seed")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("tet_multiview_timing.py needs a CUDA device")
    distributed = "RANK" in os.environ
    rank, local, ws = 0, 0, 1
    if distributed:
        rank, local, ws = int(os.environ["RANK"]), int(os.environ["LOCAL_RANK"]), int(os.environ["WORLD_SIZE"])
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if distributed:
        dist.init_process_group("nccl", device_id=dev)

    cpu = scenes.tet_grid_scene("C3x%d" % a.views, 2, 64, 512, 512, B=a.views)
    mine = shard_views(a.views, rank, ws)
    sl = slice(mine.start, mine.stop)
    put = lambda t: t.to(dev)
    verts, faces, tets, face_tets, tet_faces = map(put, (cpu.verts, cpu.faces, cpu.tets, cpu.face_tets, cpu.tet_faces))
    mv, pj, vd, fi = [put(t[sl].contiguous()) for t in (cpu.mv_mats, cpu.proj_mats, cpu.verts_depth, cpu.faces_intense)]
    P, F, Bl = verts.shape[0], faces.shape[0], len(mine)
    gen = torch.Generator(device=dev).manual_seed(1234 + rank)
    gc = torch.rand(Bl, 3, cpu.H, cpu.W, generator=gen, device=dev) * 2 - 1
    gd = torch.rand(Bl, 1, cpu.H, cpu.W, generator=gen, device=dev) * 2 - 1
    renderer = TetRenderer(TetRenderSettings(cpu.H, cpu.W, put(cpu.bg), a.seed))
    vpc = a.views_per_call

    g = PackedSceneGrads(None, put(cpu.verts_color), put(cpu.faces_opacity))
    calls = []

    def cotangents(c, d):
        first = sum(calls)
        calls.append(c.shape[0])
        return gc[first:first + c.shape[0]], gd[first:first + c.shape[0]]

    def direct_step():
        calls.clear()
        tet_multiview_step(renderer, g, verts, faces, tets, face_tets, tet_faces, mv, pj, vd, fi, cotangents,
                           views_per_call=vpc, first_view=mine.start)

    vc = put(cpu.verts_color).requires_grad_()
    fo = put(cpu.faces_opacity).requires_grad_()

    def autograd_step():
        vc.grad = fo.grad = None
        for s in range(0, Bl, vpc):
            e = min(Bl, s + vpc)
            c, d, _ = renderer(verts, faces, vc, fo, mv[s:e], pj[s:e], vd[s:e], fi[s:e], tets, face_tets, tet_faces,
                               first_view=mine.start + s)
            torch.autograd.backward([c, d], [gc[s:e], gd[s:e]])

    variants = {"direct": direct_step}
    if ws == 1:
        variants["autograd"] = autograd_step
    for fn in variants.values():
        for _ in range(a.warmup):
            fn()
    torch.cuda.synchronize()
    times = {k: [] for k in variants}
    for _ in range(a.rounds):
        for k, fn in variants.items():
            if distributed:
                dist.barrier()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(a.steps):
                fn()
            e1.record()
            torch.cuda.synchronize()
            ms = torch.tensor([e0.elapsed_time(e1) / a.steps], device=dev)
            if distributed:
                dist.all_reduce(ms, op=dist.ReduceOp.MAX)
            times[k].append(float(ms.item()))
    if rank == 0:
        name, power = card()
        res = {"gpu": name, "power_limit": power, "gpus": ws, "views": a.views, "views_per_call": vpc,
               "H": cpu.H, "W": cpu.W, "P": P, "F": F, "T": int(tets.shape[0]), "ray_random_seed": a.seed,
               "packed_floats": g.flat.numel(), "collective": g.collective, "steps_per_round": a.steps,
               "rounds": a.rounds}
        for k, t in times.items():
            t = sorted(t)
            med = t[len(t) // 2]
            res[k] = {"step_ms_median": med, "step_ms_min": t[0], "step_ms_max": t[-1], "views_per_s": a.views * 1e3 / med}
        line = json.dumps(res)
        print(line, flush=True)
        if a.out:
            with open(a.out, "a") as f:
                f.write(line + "\n")
    if distributed:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
