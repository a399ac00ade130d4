"""Multi-GPU end-to-end check of the tet renderer's camera-sharded step: tet_multiview_step (real TetRenderer kernels,
direct gradient sink, ONE all-reduce of the packed scene gradients -- NVLS kernel when the node has NVSwitch
multicast, else NCCL) against the same B views rendered in one call on one GPU.  Cases: ray_random_seed 0 and > 0
(the sharded calls pass first_view, so jittered rays must match too), vertex_grads off (3P + F buffer) and on
(6P + F buffer).

    torchrun --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 tools/tet_multiview_check.py [B=8]
"""
import os
import sys

import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from dmesh_renderer_b200 import TetRenderer, TetRenderSettings, scenes  # noqa: E402
from dmesh_renderer_b200.multiview import PackedSceneGrads, shard_views, tet_multiview_step  # noqa: E402

rank, local, ws = int(os.environ["RANK"]), int(os.environ["LOCAL_RANK"]), int(os.environ["WORLD_SIZE"])
torch.cuda.set_device(local)
dev = torch.device("cuda", local)
dist.init_process_group("nccl", device_id=dev)
B = int(sys.argv[1]) if len(sys.argv) > 1 else 8


def rel_l2(a, b):
    a, b = a.double(), b.double()
    return ((a - b).norm() / b.norm().clamp_min(1e-30)).item()


for label, cpu in (("small", scenes.tet_grid_scene("tmvc", 31, 12, 160, 192, B=B, opacity=(0.0, 0.3))),
                   ("C3-like", scenes.tet_grid_scene("tmvc3", 32, 32, 384, 384, B=B))):
    s = scenes.to_device(cpu, dev)
    gc, gd = [t.to(dev) for t in scenes.cotangents(cpu)]
    P, F = s.verts.shape[0], s.faces.shape[0]
    for seed in (0, 9):
        for vertex in (False, True):
            renderer = TetRenderer(TetRenderSettings(s.H, s.W, s.bg, seed), vertex_grads=vertex)

            # ---- reference: all B views in one call on this GPU, ordinary autograd accumulation
            ref = [s.verts.clone().requires_grad_(vertex), s.verts_color.clone().requires_grad_(),
                   s.faces_opacity.clone().requires_grad_()]
            c0, d0, a0 = renderer(ref[0], s.faces, ref[1], ref[2], s.mv_mats, s.proj_mats, s.verts_depth,
                                  s.faces_intense, s.tets, s.face_tets, s.tet_faces)
            torch.autograd.backward([c0, d0], [gc, gd])

            # ---- sharded: this rank's views, two calls per step, direct sink, one all-reduce
            mine = shard_views(B, rank, ws)
            sl = slice(mine.start, mine.stop)
            g = PackedSceneGrads(s.verts.clone() if vertex else None, s.verts_color.clone(), s.faces_opacity.clone())
            assert g.flat.numel() == (6 * P if vertex else 3 * P) + F
            calls = []

            def cotangents(c, d):
                first = mine.start + sum(calls)
                calls.append(c.shape[0])
                return gc[first:first + c.shape[0]], gd[first:first + c.shape[0]]

            outs = tet_multiview_step(renderer, g, g.leaves[0] if vertex else s.verts, s.faces, s.tets, s.face_tets,
                                      s.tet_faces, s.mv_mats[sl], s.proj_mats[sl], s.verts_depth[sl],
                                      s.faces_intense[sl], cotangents, views_per_call=max(1, len(mine) // 2),
                                      first_view=mine.start)
            torch.cuda.synchronize()
            fwd_same = all(torch.equal(torch.cat(got), want[sl]) for got, want in zip(zip(*outs), (c0, d0, a0)))
            names = (("verts",) if vertex else ()) + ("verts_color", "faces_opacity")
            errs = {n: rel_l2(leaf.grad, r.grad) for n, leaf, r in zip(names, g.leaves, ref[-len(names):])}
            # every rank must hold the same reduced gradients and the same forward images as the one-GPU call
            mx = g.flat.clone()
            dist.all_reduce(mx, op=dist.ReduceOp.MAX)
            same = bool(torch.equal(mx, g.flat))
            if rank == 0:
                print("%s seed=%d vertex_grads=%s: B=%d over %d ranks, buffer %d floats, collective=%s, rel L2 vs one "
                      "GPU: %s, identical on all ranks: %s, forward bit-identical: %s" %
                      (label, seed, vertex, B, ws, g.flat.numel(), g.collective,
                       {k: "%.2e" % v for k, v in errs.items()}, same, fwd_same), flush=True)
            ok = torch.tensor([1 if same and fwd_same and all(v <= 1e-4 for v in errs.values()) else 0], device=dev)
            dist.all_reduce(ok, op=dist.ReduceOp.MIN)
            assert int(ok.item()) == 1, (label, seed, vertex, errs, same, fwd_same)
            del g
if rank == 0:
    print("tet_multiview_check ok", flush=True)
dist.destroy_process_group()
