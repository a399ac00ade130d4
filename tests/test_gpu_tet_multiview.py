"""Tet renderer in the camera-sharded multi-view step: jitter keyed by the view's index in the job (first_view), the
direct gradient sink (PackedSceneGrads.direct()) in every backward mode, tet_multiview_step on one GPU, and (two or
more GPUs) tools/tet_multiview_check.py under torchrun."""
import pytest
import torch

from dmesh_renderer_b200 import TetRenderer, TetRenderSettings, _C, scenes
from dmesh_renderer_b200.multiview import PackedSceneGrads, tet_multiview_step
from test_gpu_nvls_allreduce import torchrun

pytestmark = pytest.mark.gpu

SINK_TOL = 1e-5


def rel_l2(a, b):
    a, b = a.double(), b.double()
    return ((a - b).norm() / b.norm().clamp_min(1e-30)).item()


_scenes = {}


def scene(B):
    if B not in _scenes:
        cpu = scenes.tet_grid_scene("tmv%d" % B, 22, 8, 96, 112, B=B, opacity=(0.0, 0.3))
        _scenes[B] = (scenes.to_device(cpu, "cuda"), [t.cuda() for t in scenes.cotangents(cpu)])
    return _scenes[B]


@torch.no_grad()
def test_jitter_depends_on_the_views_index_in_the_job():
    s, _ = scene(6)
    r = TetRenderer(TetRenderSettings(s.H, s.W, s.bg, 7))
    args = lambda a, b: (s.verts, s.faces, s.verts_color, s.faces_opacity, s.mv_mats[a:b], s.proj_mats[a:b],
                         s.verts_depth[a:b], s.faces_intense[a:b], s.tets, s.face_tets, s.tet_faces)
    full = r(*args(0, 6))
    assert torch.equal(r(*args(0, 6), first_view=0)[0], full[0])
    for a, b in ((2, 5), (5, 6), (1, 2), (0, 3)):
        part = r(*args(a, b), first_view=a)
        for x, y in zip(part, full):
            assert torch.equal(x, y[a:b]), (a, b)
        if a > 0:   # without first_view the call's views get the rays of views 0 .. b - a - 1
            assert not torch.equal(r(*args(a, b))[0], full[0][a:b]), (a, b)


# (vertex_grads, camera gradients, intensity_grads): every backward entry point and kernel combination
MODES = {"_".join(n for n, on in zip(("vertex", "camera", "intensity"), m) if on) or "plain": m
         for m in [(v, c, i) for v in (False, True) for c in (False, True) for i in (False, True)]}


@pytest.mark.parametrize("mode", list(MODES))
@pytest.mark.parametrize("deterministic", [False, True], ids=["default", "det"])
def test_direct_sink_equals_autograd_accumulation(mode, deterministic):
    """Two calls per step (views_per_call=2): the sink's kernels add into the packed buffer what autograd would have
    added to .grad.  Camera and intensity gradients still arrive through autograd; tensors other than the sink's
    leaves take the ordinary path.  Deterministic mode does the same fp32 adds of the same converted per-call sums
    on both paths, so it is bit-identical."""
    vertex, camera, intensity = MODES[mode]
    s, (gc, gd) = scene(4)
    renderer = TetRenderer(TetRenderSettings(s.H, s.W, s.bg, 3), deterministic=deterministic, vertex_grads=vertex,
                           intensity_grads=intensity)

    def per_view():
        return [s.mv_mats.clone().requires_grad_(camera), s.proj_mats.clone().requires_grad_(camera),
                s.faces_intense.clone().requires_grad_(intensity)]

    def run(v, vc, fo, pv):
        for a in (0, 2):
            c, d, _ = renderer(v, s.faces, vc, fo, pv[0][a:a + 2], pv[1][a:a + 2], s.verts_depth[a:a + 2],
                               pv[2][a:a + 2], s.tets, s.face_tets, s.tet_faces, first_view=a)
            torch.autograd.backward([c, d], [gc[a:a + 2], gd[a:a + 2]])

    ref = [s.verts.clone().requires_grad_(vertex), s.verts_color.clone().requires_grad_(),
           s.faces_opacity.clone().requires_grad_()]
    ref_pv = per_view()
    run(*ref, ref_pv)

    launches = []
    orig = _C.render_tets_backward

    def spy(*a, **k):
        launches.append(k.get("accumulate_into") is not None)
        return orig(*a, **k)
    _C.render_tets_backward = spy
    try:
        for positions in (False, True):
            launches.clear()
            g = PackedSceneGrads(s.verts.clone() if positions else None, s.verts_color.clone(),
                                 s.faces_opacity.clone())
            v = g.leaves[0] if positions else s.verts.clone().requires_grad_(vertex)
            pv = per_view()
            with g.direct():
                run(v, *g.leaves[-2:], pv)
            assert launches == [True, True]
            assert g.flat.numel() == (6 if positions else 3) * s.verts.shape[0] + s.faces.shape[0]
            got = [v.grad, g.leaves[-2].grad, g.leaves[-1].grad]
            for n, x, r in zip(("verts", "verts_color", "faces_opacity"), got, ref):
                if r.grad is None:                    # vertex_grads off: the verts slot stays zero
                    assert n == "verts" and (x is None or float(x.abs().max()) == 0.0), n
                    continue
                assert float(r.grad.abs().max()) > 0, n
                if deterministic:
                    assert torch.equal(x, r.grad), n
                else:
                    assert rel_l2(x, r.grad) <= SINK_TOL, (n, rel_l2(x, r.grad))
            for n, x, r in zip(("mv_mats", "proj_mats", "faces_intense"), pv, ref_pv):
                assert (x.grad is None) == (r.grad is None), n
                if r.grad is not None:
                    assert rel_l2(x.grad, r.grad) <= SINK_TOL, n
            # tensors that are not the sink's leaves: ordinary autograd path even while the sink is active
            other = [t.detach().clone().requires_grad_(t.requires_grad) for t in ref]
            with g.direct():
                run(*other, per_view())
            assert launches[-2:] == [False, False]
            for o, r in zip(other, ref):
                if r.grad is not None:
                    assert rel_l2(o.grad, r.grad) <= SINK_TOL
        assert not _C._grad_sinks
    finally:
        _C.render_tets_backward = orig


@pytest.mark.parametrize("positions", [False, True], ids=["3P+F", "6P+F"])
@pytest.mark.parametrize("seed", [0, 5])
@pytest.mark.parametrize("views_per_call", [1, 3, None])
def test_single_gpu_step_equals_one_call(views_per_call, seed, positions):
    B = 6
    s, (gc, gd) = scene(B)
    renderer = TetRenderer(TetRenderSettings(s.H, s.W, s.bg, seed), vertex_grads=positions)
    ref = [s.verts.clone().requires_grad_(positions), s.verts_color.clone().requires_grad_(),
           s.faces_opacity.clone().requires_grad_()]
    c0, d0, a0 = renderer(ref[0], s.faces, ref[1], ref[2], s.mv_mats, s.proj_mats, s.verts_depth, s.faces_intense,
                          s.tets, s.face_tets, s.tet_faces)
    torch.autograd.backward([c0, d0], [gc, gd])

    g = PackedSceneGrads(s.verts.clone() if positions else None, s.verts_color.clone(), s.faces_opacity.clone())
    v = g.leaves[0] if positions else s.verts
    done = []

    def cotangents(c, d):
        a = sum(done)
        done.append(c.shape[0])
        return gc[a:a + c.shape[0]], gd[a:a + c.shape[0]]

    outs = tet_multiview_step(renderer, g, v, s.faces, s.tets, s.face_tets, s.tet_faces, s.mv_mats, s.proj_mats,
                              s.verts_depth, s.faces_intense, cotangents, views_per_call=views_per_call)
    assert len(outs) == -(-B // (views_per_call or B))
    for got, want in zip(zip(*outs), (c0, d0, a0)):
        assert torch.equal(torch.cat(got), want)
    got = ([g.leaves[0].grad] if positions else []) + [g.leaves[-2].grad, g.leaves[-1].grad]
    want = ([ref[0].grad] if positions else []) + [ref[1].grad, ref[2].grad]
    for x, r in zip(got, want):
        assert rel_l2(x, r) <= SINK_TOL


@pytest.mark.timeout(600)
def test_tet_multiview_step_two_ranks_equals_one_gpu():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs at least 2 GPUs")
    r = torchrun("tet_multiview_check.py", 29575, timeout=500)
    out = r.stdout
    assert r.returncode == 0, out[-3000:] + r.stderr[-3000:]
    assert "tet_multiview_check ok" in out, out[-3000:]
    lines = [ln for ln in out.splitlines() if "over 2 ranks" in ln]
    assert len(lines) == 8, out[-3000:]
    for ln in lines:
        if "no multicast address" not in ln:
            assert "collective=nvls" in ln, ln       # the hand-written in-switch all-reduce really ran
        assert "identical on all ranks: True" in ln and "forward bit-identical: True" in ln, ln
