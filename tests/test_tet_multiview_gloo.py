"""CPU, world_size 2, gloo: the camera-sharded tet step (multiview.tet_multiview_step) must give every rank the same
view-summed scene gradients as one process rendering all views, through ONE all-reduce of the packed buffer without
positions, [dL_dvcolor | dL_dfopacity] = (3P + F) floats.  The renderer is a CPU stand-in on the oracle (seed 0)."""
import os
import sys

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle"))


class _OracleTet(torch.autograd.Function):
    @staticmethod
    def forward(ctx, verts, faces, verts_color, faces_opacity, mv, proj, verts_depth, faces_intense, tets, face_tets,
                tet_faces, H, W, bg):
        import oracle
        from dmesh_renderer_b200.scenes import Scene
        s = Scene("x", "tet", H, W, verts, faces, verts_color, faces_opacity, mv, proj, verts_depth, faces_intense, bg,
                  tets, face_tets, tet_faces)
        o = oracle.TetOracle(s)
        out = o.outputs()
        ctx.o = o
        active = torch.from_numpy(out["active"]) > 0.5
        ctx.mark_non_differentiable(active)
        return torch.from_numpy(out["color"]), torch.from_numpy(out["depth"]), active

    @staticmethod
    def backward(ctx, gc, gd, ga):
        g_vcol, g_fopa = ctx.o.backward(gc.contiguous(), gd.contiguous())
        f = lambda a: torch.from_numpy(np.asarray(a, np.float32))
        return (None, None, f(g_vcol), f(g_fopa)) + (None,) * 10


class OracleTetRenderer:
    """TetRenderer stand-in (ray_random_seed 0: first_view changes nothing) returning the verts_color /
    faces_opacity gradients of the CPU oracle."""

    def __init__(self, H, W, bg):
        self.H, self.W, self.bg = H, W, bg

    def __call__(self, verts, faces, verts_color, faces_opacity, mv_mats, proj_mats, verts_depth, faces_intense, tets,
                 face_tets, tet_faces, first_view=0):
        assert first_view >= 0
        return _OracleTet.apply(verts, faces, verts_color, faces_opacity, mv_mats, proj_mats, verts_depth,
                                faces_intense, tets, face_tets, tet_faces, self.H, self.W, self.bg)


def _scene():
    from dmesh_renderer_b200 import scenes
    return scenes.tet_grid_scene("tmv", 21, 4, 48, 64, B=4, opacity=(0.0, 0.5))


def _cot(color, depth):
    return color.detach() * 0.5 - 0.25, depth.detach() - 0.5


def _step(s, sl, first_view, views_per_call):
    from dmesh_renderer_b200.multiview import PackedSceneGrads, tet_multiview_step
    g = PackedSceneGrads(None, s.verts_color.clone(), s.faces_opacity.clone())
    tet_multiview_step(OracleTetRenderer(s.H, s.W, s.bg), g, s.verts, s.faces, s.tets, s.face_tets, s.tet_faces,
                       s.mv_mats[sl], s.proj_mats[sl], s.verts_depth[sl], s.faces_intense[sl], _cot,
                       views_per_call=views_per_call, first_view=first_view)
    return g


def _run_rank(rank, ws, port, out):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=ws)
    try:
        from dmesh_renderer_b200.multiview import shard_views
        s = _scene()
        mine = shard_views(s.mv_mats.shape[0], rank, ws)
        g = _step(s, slice(mine.start, mine.stop), mine.start, 1)
        torch.save(g.flat.clone(), os.path.join(out, "rank%d.pt" % rank))
    finally:
        dist.destroy_process_group()


@pytest.mark.timeout(300)
def test_two_ranks_match_single_process(tmp_path):
    import socket
    with socket.socket() as sk:
        sk.bind(("127.0.0.1", 0))
        port = sk.getsockname()[1]
    mp.spawn(_run_rank, args=(2, port, str(tmp_path)), nprocs=2, join=True)
    r0, r1 = torch.load(tmp_path / "rank0.pt"), torch.load(tmp_path / "rank1.pt")
    assert torch.equal(r0, r1)                       # all-reduce leaves identical buffers everywhere

    s = _scene()
    g = _step(s, slice(None), 0, None)
    rel = ((r0 - g.flat).norm() / g.flat.norm()).item()
    assert g.flat.abs().sum() > 0
    assert rel < 1e-5, rel
    P, F = s.verts.shape[0], s.faces.shape[0]
    assert g.flat.numel() == 3 * P + F               # the tet buffer without positions
