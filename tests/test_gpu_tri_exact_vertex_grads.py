"""Tri renderer: exact vertex-position gradients (exact_vertex_grads=True).

The yardstick is the fp64 reference of the camera-gradient tests (tests/test_gpu_tri_camera_grads.py): the forward
function as implemented, on the fragments the CPU oracle composites, differentiated by autograd.  Its dL/dverts is the
exact derivative; the renderer's default keeps the reference implementation's formula and is not compared with it.
"""
import numpy as np
import pytest
import torch

import tri_fragments  # noqa: F401  (built on first use by oracle_fragments)
from test_gpu_tri_camera_grads import (CAM_TOL, GRAD_TOL, IMG_TOL, SCENES, _stages, oracle_fragments, reference_grads,
                                       rel_l2)
from test_tri_exact_vertex_grads_reference import rigid_residual
import dmesh_renderer_b200 as dmr
from dmesh_renderer_b200 import TriRenderer, TriRenderSettings, _C, _lib, multiview, scenes

pytestmark = pytest.mark.gpu
f64 = torch.float64


def closed_mesh(name="torus", seed=31, n=24, m=12, H=96, W=112, B=3):
    """A seeded, jittered torus: connected and closed, every vertex shared by six faces."""
    g = torch.Generator().manual_seed(seed)
    i, j = torch.meshgrid(torch.arange(n), torch.arange(m), indexing="ij")
    a, b = i.reshape(-1) * (2 * np.pi / n), j.reshape(-1) * (2 * np.pi / m)
    R, r = 0.6, 0.25
    verts = torch.stack([(R + r * torch.cos(b)) * torch.cos(a), (R + r * torch.cos(b)) * torch.sin(a), r * torch.sin(b)], 1)
    verts = (verts + 0.01 * torch.randn(verts.shape, generator=g)).float().contiguous()
    vid = lambda ii, jj: (ii % n) * m + (jj % m)
    i, j = i.reshape(-1), j.reshape(-1)
    faces = torch.cat([torch.stack([vid(i, j), vid(i + 1, j), vid(i + 1, j + 1)], 1),
                       torch.stack([vid(i, j), vid(i + 1, j + 1), vid(i, j + 1)], 1)]).to(torch.int32).contiguous()
    P, F = verts.shape[0], faces.shape[0]
    verts_color = torch.rand(P, 3, generator=g)
    faces_opacity = torch.rand(F, generator=g) * 0.6 + 0.1
    faces_intense = torch.rand(B, F, generator=g) * 0.5 + 0.5
    mv, pj = scenes.cameras(scenes.fibonacci_dirs(B, g), 3.0, W, H, 0.5, 6.0)
    return scenes.Scene(name, "tri", H, W, verts, faces, verts_color, faces_opacity, mv, pj,
                        scenes.ndc_depth(verts, mv, pj), faces_intense, torch.ones(3))


ALL = dict(SCENES, torus=closed_mesh)
_refs = {}


def reference_for(name, fused):
    key = (name, fused)
    if key not in _refs:
        cpu = ALL[name]()
        gc, gd = scenes.cotangents(cpu)
        frags, _ = oracle_fragments(cpu)
        _refs[key] = (cpu, gc, gd, frags, reference_grads(cpu, frags, gc, gd, fused))
    return _refs[key]


def gpu_run(cpu, gc, gd, fused=False, deterministic=False, exact=True, camera=False, scale=1.0):
    s = scenes.to_device(cpu, "cuda")
    mv = s.mv_mats.detach().clone().requires_grad_(camera)
    pj = s.proj_mats.detach().clone().requires_grad_(camera)
    leaves = [t.clone().requires_grad_() for t in (s.verts, s.verts_color, s.faces_opacity, s.faces_intense)]
    vd = None if fused else s.verts_depth.clone().requires_grad_()
    color, depth = TriRenderer(TriRenderSettings(s.H, s.W, s.bg), deterministic=deterministic, exact_vertex_grads=exact)(
        leaves[0], s.faces, leaves[1], leaves[2], mv, pj, vd, leaves[3])
    torch.autograd.backward([color, depth], [gc.cuda() * scale, gd.cuda() * scale])
    g = dict(verts=leaves[0].grad, verts_color=leaves[1].grad, faces_opacity=leaves[2].grad,
             faces_intense=leaves[3].grad, mv_mats=mv.grad, proj_mats=pj.grad)
    if vd is not None:
        g["verts_depth"] = vd.grad
    return color.detach(), depth.detach(), g


def grazing_vertices(cpu, frags):
    """Vertices of faces that some pixel sees at a grazing angle (|rd.n| < 1e-2 |n|): there fp32 (u, v) carry a large
    relative error and dL/dverts grows like 1/D (see test_tri_exact_vertex_grads_reference)."""
    from test_tri_exact_vertex_grads_reference import reference_hits
    gc, gd = scenes.cotangents(cpu)
    _, hits = reference_hits(cpu, frags, gc, gd, False)
    n = torch.linalg.cross(hits["E2"], hits["E1"])
    cos = (hits["rd"] * n).sum(1).abs() / n.norm(dim=1)
    faces = torch.unique(hits["f"][cos < 1e-2])
    mask = np.zeros(cpu.verts.shape[0], bool)
    mask[cpu.faces.long()[faces].reshape(-1).numpy()] = True
    return mask, faces.numel()


_worst = {}


@pytest.mark.parametrize("deterministic", [False, True], ids=["default", "det"])
@pytest.mark.parametrize("fused", [False, True], ids=["explicit_depth", "fused_depth"])
@pytest.mark.parametrize("name", list(ALL))
def test_exact_vertex_grads_match_fp64_reference(name, fused, deterministic):
    cpu, gc, gd, frags, (rc, rd, rg) = reference_for(name, fused)
    color, depth, g = gpu_run(cpu, gc, gd, fused=fused, deterministic=deterministic)
    # self-checks of the reference
    assert (color.cpu().double() - rc).abs().max().item() <= IMG_TOL
    assert (depth.cpu().double() - rd).abs().max().item() <= IMG_TOL
    for k in ["verts_color", "faces_opacity", "faces_intense"] + ([] if fused else ["verts_depth"]):
        e = rel_l2(g[k].cpu().numpy(), rg[k].numpy())
        assert e <= GRAD_TOL, "%s rel L2 %.3e" % (k, e)
    got, ref = g["verts"].cpu().numpy(), rg["verts"].numpy()
    mask, nf = grazing_vertices(cpu, frags)
    e_all = rel_l2(got, ref)
    e = rel_l2(got[~mask], ref[~mask])
    print("\n[exact dL/dverts] %s %s %s: rel L2 %.2e (%d grazing faces left out; %.2e with them)" % (
        name, "fused" if fused else "explicit", "det" if deterministic else "default", e, nf, e_all))
    assert nf <= 0.01 * cpu.faces.shape[0]
    assert e <= CAM_TOL


@pytest.mark.parametrize("deterministic", [False, True], ids=["default", "det"])
@pytest.mark.parametrize("fused", [False, True], ids=["explicit_depth", "fused_depth"])
def test_other_gradients_as_in_reference_mode(fused, deterministic):
    cpu = SCENES["cam4"]()
    gc, gd = scenes.cotangents(cpu)
    _, _, ex = gpu_run(cpu, gc, gd, fused=fused, deterministic=deterministic, exact=True, camera=True)
    _, _, rf = gpu_run(cpu, gc, gd, fused=fused, deterministic=deterministic, exact=False, camera=True)
    same = []
    for k in ex:
        if k == "verts":
            continue
        assert rel_l2(ex[k].cpu().numpy(), rf[k].cpu().numpy()) <= 1e-6, k
        if torch.equal(ex[k], rf[k]):
            same.append(k)
    print("\n[exact vs reference mode] %s %s: bit-identical: %s" % (
        "fused" if fused else "explicit", "det" if deterministic else "default", ", ".join(same) or "none"))


@pytest.mark.parametrize("fused", [False, True], ids=["explicit_depth", "fused_depth"])
@pytest.mark.parametrize("name", ["small_tri", "cam4", "torus"])
def test_rigid_motion_identity(name, fused):
    cpu = ALL[name]()
    gc, gd = scenes.cotangents(cpu)
    res = {}
    for exact in (True, False):
        _, _, g = gpu_run(cpu, gc, gd, fused=fused, deterministic=True, exact=exact, camera=True)
        r, s = rigid_residual(cpu.verts, cpu.mv_mats, g["verts"].cpu(), g["mv_mats"].cpu())
        res[exact] = r / s
    print("\n[rigid motion] %s %s: exact %.2e, reference formula %.2e (residual / sum of |terms|)" % (
        name, "fused" if fused else "explicit", res[True], res[False]))
    assert res[True] <= 1e-3


@pytest.mark.parametrize("fused", [False, True], ids=["explicit_depth", "fused_depth"])
def test_deterministic_reproducible_linear_zero(fused):
    cpu = SCENES["cam4"]()
    gc, gd = scenes.cotangents(cpu)
    runs = [gpu_run(cpu, gc, gd, fused=fused, deterministic=True)[2] for _ in range(4)]
    for r in runs[1:]:
        for k in runs[0]:
            assert torch.equal(r[k], runs[0][k]) if r[k] is not None else runs[0][k] is None, k
    for sc in (0.125, 32.0):
        g = gpu_run(cpu, gc, gd, fused=fused, deterministic=True, scale=sc)[2]
        assert torch.equal(g["verts"], runs[0]["verts"] * sc), sc
    zero = gpu_run(cpu, gc * 0, gd * 0, fused=fused, deterministic=True)[2]
    for k, t in zero.items():
        if t is not None:
            assert torch.count_nonzero(t) == 0, k


@pytest.mark.parametrize("name", ["cam4", "torus"])
def test_packed_scene_grads_direct(name):
    """PackedSceneGrads.direct() / multiview_step with an exact-mode renderer equals plain autograd accumulation."""
    cpu = ALL[name]()
    s = scenes.to_device(cpu, "cuda")
    gct, gdt = [t.cuda() for t in scenes.cotangents(cpu)]
    renderer = TriRenderer(TriRenderSettings(s.H, s.W, s.bg), deterministic=True, exact_vertex_grads=True)
    cot = lambda color, depth: (gct, gdt)

    def step(sink):
        verts, vcol, fopa = (t.clone().requires_grad_() for t in (s.verts, s.verts_color, s.faces_opacity))
        if sink:
            sg = multiview.PackedSceneGrads(verts, vcol, fopa)
            multiview.multiview_step(renderer, sg, s.faces, s.mv_mats, s.proj_mats, s.verts_depth, s.faces_intense, cot)
            return sg.flat.clone()
        color, depth = renderer(verts, s.faces, vcol, fopa, s.mv_mats, s.proj_mats, s.verts_depth, s.faces_intense)
        torch.autograd.backward([color, depth], [gct, gdt])
        return torch.cat([verts.grad.reshape(-1), vcol.grad.reshape(-1), fopa.grad.reshape(-1)])

    direct, plain = step(True), step(False)
    assert torch.equal(direct, plain)
    # and it is the exact gradient, not the reference formula
    ref = TriRenderer(TriRenderSettings(s.H, s.W, s.bg), deterministic=True, exact_vertex_grads=False)
    verts = s.verts.clone().requires_grad_()
    color, depth = ref(verts, s.faces, s.verts_color, s.faces_opacity, s.mv_mats, s.proj_mats, s.verts_depth,
                       s.faces_intense)
    torch.autograd.backward([color, depth], [gct, gdt])
    assert not torch.equal(verts.grad.reshape(-1), plain[:verts.numel()])


def _backward_launches(renderer, s, gc, gd, fused, camera):
    lib = _lib.load()
    verts = s.verts.clone().requires_grad_()
    mv = s.mv_mats.clone().requires_grad_(camera)
    args = (verts, s.faces, s.verts_color, s.faces_opacity, mv, s.proj_mats, None if fused else s.verts_depth,
            s.faces_intense)
    renderer(*args)                              # warm-up: same shapes for the speculative binning buffer
    torch.cuda.synchronize()
    _lib.check(lib.dmr_profile_enable(1))
    try:
        _stages()
        color, depth = renderer(*args)
        torch.cuda.synchronize()
        _stages()
        n1 = lib.dmr_launch_count()
        torch.autograd.backward([color, depth], [gc, gd])
        n2 = lib.dmr_launch_count()
        torch.cuda.synchronize()
        return n2 - n1, _stages(), verts.grad
    finally:
        lib.dmr_profile_enable(0)


@pytest.mark.parametrize("camera", [False, True], ids=["plain", "camera"])
@pytest.mark.parametrize("deterministic", [False, True], ids=["default", "det"])
@pytest.mark.parametrize("fused", [False, True], ids=["explicit_depth", "fused_depth"])
def test_same_launches_and_stages(fused, deterministic, camera):
    cpu = SCENES["cam4"]()
    s = scenes.to_device(cpu, "cuda")
    gc, gd = [t.cuda() for t in scenes.cotangents(cpu)]
    st = TriRenderSettings(s.H, s.W, s.bg)
    off = _backward_launches(TriRenderer(st, deterministic, exact_vertex_grads=False), s, gc, gd, fused, camera)
    on = _backward_launches(TriRenderer(st, deterministic, exact_vertex_grads=True), s, gc, gd, fused, camera)
    assert off[0] == on[0] and off[1] == on[1], (off[:2], on[:2])
    assert ("tri_render_backward_camera" in on[1]) == camera and "tri_grad_finish" in on[1]
    assert not torch.equal(off[2], on[2])


def test_default_and_override():
    cpu = SCENES["cam4"]()
    s = scenes.to_device(cpu, "cuda")
    gc, gd = [t.cuda() for t in scenes.cotangents(cpu)]
    st = TriRenderSettings(s.H, s.W, s.bg)

    def verts_grad(renderer=None, **kw):
        verts = s.verts.clone().requires_grad_()
        args = (verts, s.faces, s.verts_color, s.faces_opacity, s.mv_mats, s.proj_mats, s.verts_depth, s.faces_intense)
        if renderer is not None:
            color, depth = renderer(*args)
        else:
            a = list(args)
            a[4], a[5] = s.mv_mats.transpose(1, 2), s.proj_mats.transpose(1, 2)
            color, depth = dmr.render_tri(*a, st, deterministic=True, **kw)
        torch.autograd.backward([color, depth], [gc, gd])
        return verts.grad

    exact = verts_grad(TriRenderer(st, True, exact_vertex_grads=True))
    reference = verts_grad(TriRenderer(st, True, exact_vertex_grads=False))
    assert not torch.equal(exact, reference)
    assert torch.equal(verts_grad(TriRenderer(st, True)), reference)          # the default is the reference formula
    assert torch.equal(verts_grad(exact_vertex_grads=True), exact)
    old = dmr.set_exact_vertex_grads(True)
    try:
        assert old is False
        assert torch.equal(verts_grad(TriRenderer(st, True)), exact)
        assert torch.equal(verts_grad(), exact)
        assert torch.equal(verts_grad(TriRenderer(st, True, exact_vertex_grads=False)), reference)
        assert torch.equal(verts_grad(exact_vertex_grads=False), reference)
    finally:
        assert dmr.set_exact_vertex_grads(old) is True
    assert torch.equal(verts_grad(TriRenderer(st, True)), reference)


def test_c_level_reference_call_unchanged():
    """The reference-shaped 18-argument _C.render_tris_backward is the reference formula; exact_vertex_grads=True
    changes dL/dverts only."""
    cpu = SCENES["cam4"]()
    s = scenes.to_device(cpu, "cuda")
    gc, gd = [t.cuda() for t in scenes.cotangents(cpu)]
    mv, pj = s.mv_mats.transpose(1, 2).contiguous(), s.proj_mats.transpose(1, 2).contiguous()
    imv, ipj = torch.inverse(mv), torch.inverse(pj)
    args = (s.bg, s.verts, s.faces, s.verts_color, s.faces_opacity, mv, pj, imv, ipj, s.verts_depth, s.faces_intense)
    out = _C.render_tris(*args, s.H, s.W)
    bargs = args + (gc, gd, out[0]) + tuple(out[3:])
    plain = _C.render_tris_backward(*bargs, deterministic=True)
    ref = _C.render_tris_backward(*bargs, deterministic=True, exact_vertex_grads=False)
    ex = _C.render_tris_backward(*bargs, deterministic=True, exact_vertex_grads=True)
    assert len(ex) == 5
    for a, b in zip(plain, ref):
        assert torch.equal(a, b)
    assert not torch.equal(ex[0], plain[0])
    for k in range(1, 5):
        assert rel_l2(ex[k].cpu().numpy(), plain[k].cpu().numpy()) <= 1e-6
