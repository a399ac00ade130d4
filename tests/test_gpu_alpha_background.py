"""Tri and tet renderers: the alpha image (return_alpha=True) and the gradient with respect to the background colour
(bg.requires_grad).

Yardsticks: the fp64 references of the camera-gradient tests (tests/test_gpu_tri_camera_grads.py,
tests/test_gpu_tet_camera_grads.py) extended by alpha = 1 - T_final (tests/test_alpha_background_reference.py), and,
with no oracle at all, a second render with white colours, unit intensities and a black background, whose colour
channel 0 IS alpha.
"""
import numpy as np
import pytest
import torch

import tri_fragments  # noqa: F401  (built on first use by oracle_fragments)
from test_alpha_background_reference import reference_alpha, transmittance
from test_gpu_tet_camera_grads import CASES, SCENES as TET_SCENES, trail_cap
from test_gpu_tet_camera_grads import reference_render as tet_reference_render
from test_gpu_tet_intensity_grads import kept_cotangents
from test_gpu_tri_camera_grads import SCENES as TRI_SCENES, fused_ndc_depth, oracle_fragments, rel_l2
from test_gpu_tri_camera_grads import reference_render as tri_reference_render
from test_gpu_vs_oracle_and_golden import edge_scene
from dmesh_renderer_b200 import TetRenderer, TetRenderSettings, TriRenderer, TriRenderSettings, multiview, scenes

pytestmark = pytest.mark.gpu
f64 = torch.float64
ALPHA_TOL, GRAD_TOL = 1e-5, 1e-4
TRI_ALL = dict(TRI_SCENES, edge=edge_scene)
TRI_MODES = {"plain": (False, False), "camera": (True, False), "exact": (False, True), "exact_camera": (True, True)}
TET_MODES = {"plain": (False, False, False), "camera": (True, False, False), "vertex": (False, True, False),
             "intensity": (False, False, True), "camera_vertex_intensity": (True, True, True)}


def random_bg(seed=9):
    return torch.rand(3, generator=torch.Generator().manual_seed(seed))


def alpha_cotangent(like, seed=77):
    g = torch.Generator().manual_seed(seed)
    B, _, H, W = like.shape
    return torch.rand(B, 1, H, W, generator=g) * 2 - 1


# ---------------------------------------------------------------------------------------------- tri
def tri_gpu(cpu, gc, gd, ga, det=False, fused=False, camera=False, exact=False, bg=None, return_alpha=True,
            renderer_kw=None):
    """One TriRenderer call with every input a leaf; returns (color, depth, alpha, {name: grad})."""
    s = scenes.to_device(cpu, "cuda")
    mv = s.mv_mats.detach().clone().requires_grad_(camera)
    pj = s.proj_mats.detach().clone().requires_grad_(camera)
    leaves = [t.clone().requires_grad_() for t in (s.verts, s.verts_color, s.faces_opacity, s.faces_intense)]
    vd = None if fused else s.verts_depth.clone().requires_grad_()
    bgl = (s.bg if bg is None else bg.cuda()).detach().clone().requires_grad_()
    out = TriRenderer(TriRenderSettings(s.H, s.W, bgl), deterministic=det, exact_vertex_grads=exact,
                      return_alpha=return_alpha, **(renderer_kw or {}))(leaves[0], s.faces, leaves[1], leaves[2], mv, pj,
                                                                         vd, leaves[3])
    cots = [gc.cuda(), gd.cuda()] + ([ga.cuda()] if return_alpha else [])
    torch.autograd.backward(list(out), cots)
    g = dict(verts=leaves[0].grad, verts_color=leaves[1].grad, faces_opacity=leaves[2].grad,
             faces_intense=leaves[3].grad, mv_mats=mv.grad, proj_mats=pj.grad, bg=bgl.grad)
    if vd is not None:
        g["verts_depth"] = vd.grad
    return out[0].detach(), out[1].detach(), out[2].detach() if return_alpha else None, g


def tri_reference(cpu, frags, gc, gd, ga, fused):
    """fp64 alpha, dL/dfaces_opacity and dL/dbg for the cotangents (gc, gd, ga)."""
    B, H, W = cpu.mv_mats.shape[0], cpu.H, cpu.W
    fopa = cpu.faces_opacity.to(f64).clone().requires_grad_()
    bg = cpu.bg.to(f64).clone().requires_grad_()
    verts, mv, pj = cpu.verts.to(f64), cpu.mv_mats.to(f64), cpu.proj_mats.to(f64)
    vdepth = fused_ndc_depth(verts, mv, pj) if fused else cpu.verts_depth.to(f64)
    color, depth = tri_reference_render(frags, cpu.faces, H, W, bg, verts, cpu.verts_color.to(f64), fopa, mv, pj,
                                        cpu.faces_intense.to(f64), vdepth)
    alpha = reference_alpha(frags, B, H, W, fopa)
    torch.autograd.backward([color, depth, alpha], [gc.to(f64), gd.to(f64), ga.to(f64)])
    return alpha.detach(), fopa.grad, bg.grad


_tri_refs = {}


def tri_case(name):
    if name not in _tri_refs:
        cpu = TRI_ALL[name]()
        cpu = cpu._replace(bg=random_bg())            # the stock scenes use ones
        gc, gd = scenes.cotangents(cpu)
        ga = alpha_cotangent(gd)
        frags, _ = oracle_fragments(cpu)
        _tri_refs[name] = (cpu, gc, gd, ga, frags, {})
    return _tri_refs[name]


def tri_ref(name, fused):
    cpu, gc, gd, ga, frags, cache = tri_case(name)
    if fused not in cache:
        cache[fused] = tri_reference(cpu, frags, gc, gd, ga, fused)
    return cpu, gc, gd, ga, cache[fused]


@pytest.mark.parametrize("mode", list(TRI_MODES))
@pytest.mark.parametrize("deterministic", [False, True], ids=["default", "det"])
@pytest.mark.parametrize("fused", [False, True], ids=["explicit_depth", "fused_depth"])
@pytest.mark.parametrize("name", list(TRI_ALL))
def test_tri_alpha_and_grads_match_fp64_reference(name, fused, deterministic, mode):
    cpu, gc, gd, ga, (ra, rfo, rbg) = tri_ref(name, fused)
    camera, exact = TRI_MODES[mode]
    _, _, alpha, g = tri_gpu(cpu, gc, gd, ga, det=deterministic, fused=fused, camera=camera, exact=exact)
    assert (alpha.cpu().double() - ra).abs().max().item() <= ALPHA_TOL
    e = rel_l2(g["faces_opacity"].cpu().numpy(), rfo.numpy())
    assert e <= GRAD_TOL, "faces_opacity rel L2 %.3e" % e
    e = rel_l2(g["bg"].cpu().numpy(), rbg.numpy())
    assert e <= 1e-5, "bg rel L2 %.3e" % e


def _white(cpu, bg=None):
    return cpu._replace(verts_color=torch.ones_like(cpu.verts_color), faces_intense=torch.ones_like(cpu.faces_intense),
                        bg=torch.zeros(3) if bg is None else bg)


@pytest.mark.parametrize("deterministic", [False, True], ids=["default", "det"])
@pytest.mark.parametrize("name", ["small_tri", "C1", "edge"])
def test_tri_alpha_equals_a_white_render(name, deterministic):
    cpu, gc, gd, ga, _, _ = tri_case(name)
    z3, z1 = torch.zeros_like(gc), torch.zeros_like(gd)
    # the alpha path alone: cotangent a on alpha
    _, _, alpha, g = tri_gpu(cpu, z3, z1, ga, det=deterministic)
    # the colour path of a white render with black background: cotangent (a, 0, 0) on the colour
    color, _, _, gw = tri_gpu(_white(cpu), torch.cat([ga, z1, z1], 1), z1, None, det=deterministic, return_alpha=False)
    assert (alpha - color[:, :1]).abs().max().item() <= ALPHA_TOL
    e = rel_l2(g["faces_opacity"].cpu().numpy(), gw["faces_opacity"].cpu().numpy())
    assert e <= GRAD_TOL, e


@pytest.mark.parametrize("mode", list(TRI_MODES))
@pytest.mark.parametrize("fused", [False, True], ids=["explicit_depth", "fused_depth"])
def test_tri_other_grads_unchanged_and_opacity_linear(fused, mode):
    cpu, gc, gd, ga, _, _ = tri_case("small_tri")
    camera, exact = TRI_MODES[mode]
    kw = dict(fused=fused, camera=camera, exact=exact)
    ga = ga * 0.9                                       # |dL_dalpha| <= max(|dL_dC|, |dL_dD|): the same fixed-point scale
    _, _, _, g0 = tri_gpu(cpu, gc, gd, None, det=True, return_alpha=False, **kw)
    _, _, _, g1 = tri_gpu(cpu, gc, gd, ga, det=True, **kw)
    for k, v in g0.items():
        if k in ("faces_opacity", "bg") or v is None:
            continue
        assert torch.equal(v, g1[k]), k
    for det in (False, True):
        _, _, _, a = tri_gpu(cpu, gc, gd, ga, det=det, **kw)
        _, _, _, b = tri_gpu(cpu, gc, gd, torch.zeros_like(ga), det=det, **kw)
        _, _, _, c = tri_gpu(cpu, torch.zeros_like(gc), torch.zeros_like(gd), ga, det=det, **kw)
        e = rel_l2(a["faces_opacity"].cpu().numpy(), (b["faces_opacity"] + c["faces_opacity"]).cpu().numpy())
        assert e <= 1e-5, (det, e)


@pytest.mark.parametrize("deterministic", [False, True], ids=["default", "det"])
def test_tri_background_grad(deterministic):
    cpu, gc, gd, ga, _, _ = tri_case("cam4")            # four views
    color, _, alpha, g = tri_gpu(cpu, gc, gd, ga, det=deterministic)
    want = ((1 - alpha.double()) * gc.cuda().double()).sum((0, 2, 3))
    assert torch.allclose(g["bg"].double(), want, rtol=1e-6, atol=1e-6 * want.abs().max().item())
    # reproducible bits, in both modes
    _, _, _, g2 = tri_gpu(cpu, gc, gd, ga, det=deterministic)
    assert torch.equal(g["bg"], g2["bg"])
    # central difference in bg (the colour is linear in bg)
    eps = 1e-2
    s = scenes.to_device(cpu, "cuda")
    for c in range(3):
        d = torch.zeros(3)
        d[c] = eps
        ls = []
        for sign in (1, -1):
            col, _ = TriRenderer(TriRenderSettings(s.H, s.W, (cpu.bg + sign * d).cuda()))(
                s.verts, s.faces, s.verts_color, s.faces_opacity, s.mv_mats, s.proj_mats, s.verts_depth, s.faces_intense)
            ls.append((col.double() * gc.cuda().double()).sum().item())
        cd = (ls[0] - ls[1]) / (2 * eps)
        assert abs(cd - g["bg"][c].item()) <= 1e-3 * max(1.0, abs(cd)), (c, cd, g["bg"][c].item())


def _far_away(cpu):
    return cpu._replace(verts=cpu.verts + torch.tensor([1000.0, 0.0, 0.0]))


@pytest.mark.parametrize("deterministic", [False, True], ids=["default", "det"])
def test_tri_nothing_on_screen_and_no_vertices(deterministic):
    cpu, gc, gd, ga, _, _ = tri_case("small_tri")
    # R == 0: every face off-screen; alpha 0, dL/dbg = sum dL_dC, no opacity gradient
    _, _, alpha, g = tri_gpu(_far_away(cpu), gc, gd, ga, det=deterministic)
    assert alpha.abs().max().item() == 0.0
    want = gc.double().sum((0, 2, 3))
    assert torch.allclose(g["bg"].cpu().double(), want, rtol=1e-6, atol=1e-6 * want.abs().max().item())
    assert g["faces_opacity"].abs().max().item() == 0.0
    # P == 0: zero images that do not depend on bg
    empty = cpu._replace(verts=torch.zeros(0, 3), faces=torch.zeros(0, 3, dtype=torch.int32),
                         verts_color=torch.zeros(0, 3), faces_opacity=torch.zeros(0),
                         verts_depth=torch.zeros(cpu.verts_depth.shape[0], 0),
                         faces_intense=torch.zeros(cpu.faces_intense.shape[0], 0))
    _, _, alpha, g = tri_gpu(empty, gc, gd, ga, det=deterministic)
    assert alpha.abs().max().item() == 0.0 and alpha.shape == gd.shape
    assert g["bg"].abs().max().item() == 0.0


def test_tri_float64_background_and_off_by_default():
    cpu, gc, gd, ga, _, _ = tri_case("small_tri")
    s = scenes.to_device(cpu, "cuda")
    args = (s.verts, s.faces, s.verts_color, s.faces_opacity, s.mv_mats, s.proj_mats, s.verts_depth, s.faces_intense)
    bg64 = cpu.bg.double().cuda().requires_grad_()
    color, depth = TriRenderer(TriRenderSettings(s.H, s.W, bg64))(*args)
    torch.autograd.backward([color, depth], [gc.cuda(), gd.cuda()])
    bg32 = cpu.bg.cuda().requires_grad_()
    color, depth = TriRenderer(TriRenderSettings(s.H, s.W, bg32))(*args)
    torch.autograd.backward([color, depth], [gc.cuda(), gd.cuda()])
    assert bg64.grad.dtype == torch.float64 and bg64.grad.shape == (3,)
    assert torch.equal(bg64.grad.float(), bg32.grad)
    bg = cpu.bg.cuda()
    fo = s.faces_opacity.clone().requires_grad_()
    color, depth = TriRenderer(TriRenderSettings(s.H, s.W, bg))(s.verts, s.faces, s.verts_color, fo, *args[4:])
    torch.autograd.backward([color, depth], [gc.cuda(), gd.cuda()])
    assert bg.grad is None


def test_tri_deterministic_range():
    """An alpha cotangent 2^20 above the colour / depth cotangents: the fixed-point scale follows it."""
    cpu, gc, gd, ga, frags, _ = tri_case("small_tri")
    big = ga * 2.0 ** 20
    _, rfo, _ = tri_reference(cpu, frags, gc, gd, big, False)
    _, _, _, g = tri_gpu(cpu, gc, gd, big, det=True)
    assert torch.isfinite(g["faces_opacity"]).all()
    e = rel_l2(g["faces_opacity"].cpu().numpy(), rfo.numpy())
    assert e <= GRAD_TOL, e


# ---------------------------------------------------------------------------------------------- tet
def tet_gpu(cpu, gc, gd, ga, seed=0, det=False, camera=False, vertex=False, intensity=False, bg=None,
            return_alpha=True):
    s = scenes.to_device(cpu, "cuda")
    v = s.verts.clone().requires_grad_(vertex)
    mv = s.mv_mats.detach().clone().requires_grad_(camera)
    pj = s.proj_mats.detach().clone().requires_grad_(camera)
    vc, fo = s.verts_color.clone().requires_grad_(), s.faces_opacity.clone().requires_grad_()
    fi = s.faces_intense.clone().requires_grad_(intensity)
    bgl = (s.bg if bg is None else bg.cuda()).detach().clone().requires_grad_()
    out = TetRenderer(TetRenderSettings(s.H, s.W, bgl, seed), deterministic=det, vertex_grads=vertex,
                      intensity_grads=intensity, return_alpha=return_alpha)(
        v, s.faces, vc, fo, mv, pj, s.verts_depth, fi, s.tets, s.face_tets, s.tet_faces)
    imgs = [out[0], out[1]] + ([out[3]] if return_alpha else [])
    torch.autograd.backward(imgs, [gc.cuda(), gd.cuda()] + ([ga.cuda()] if return_alpha else []))
    g = dict(verts=v.grad, verts_color=vc.grad, faces_opacity=fo.grad, faces_intense=fi.grad, mv_mats=mv.grad,
             proj_mats=pj.grad, bg=bgl.grad)
    return out[0].detach(), out[2], out[3].detach() if return_alpha else None, g


def tet_reference(cpu, frags, gc, gd, ga):
    """fp64 alpha (active pixels: 1 - T_final; inactive: 0), dL/dfaces_opacity (walked steps only) and dL/dbg."""
    B, H, W = cpu.mv_mats.shape[0], cpu.H, cpu.W
    fopa = cpu.faces_opacity.to(f64).clone().requires_grad_()
    color, depth = tet_reference_render(frags, cpu, cpu.verts_color.to(f64), fopa, cpu.mv_mats.to(f64),
                                        cpu.proj_mats.to(f64), cpu.faces_intense.to(f64))
    active = torch.from_numpy(frags["active"]).bool()
    cnt_all = torch.from_numpy(frags["counts"].astype(np.int64))
    keep = torch.repeat_interleave(active, cnt_all)
    cnt = cnt_all * active
    f = torch.from_numpy(frags["face"].astype(np.int64))[keep]
    r = torch.from_numpy(frags["reach"])[keep]
    Tf = transmittance(cnt, torch.where(r, fopa[f], fopa[f].detach()))
    alpha = torch.where(active, 1 - Tf, torch.zeros_like(Tf)).view(B, 1, H, W)
    torch.autograd.backward([color, depth, alpha], [gc.to(f64), gd.to(f64), ga.to(f64)])
    w = torch.where(active, Tf.detach(), torch.ones_like(Tf)).view(B, 1, H, W)
    return alpha.detach(), fopa.grad, (w * gc.to(f64)).sum((0, 2, 3))


_tet_refs = {}


def tet_case(case):
    if case not in _tet_refs:
        name, seed, _cap = CASES[case]
        cpu = TET_SCENES[name]()._replace(bg=random_bg())
        gc, gd, frags = kept_cotangents(cpu, seed)
        keep = (gd != 0).float()                        # pixels whose march parts from the oracle's get no cotangent
        ga = alpha_cotangent(gd) * keep
        _tet_refs[case] = (cpu, gc, gd, ga, frags, tet_reference(cpu, frags, gc, gd, ga))
    return _tet_refs[case]


@pytest.mark.parametrize("mode", list(TET_MODES))
@pytest.mark.parametrize("deterministic", [False, True], ids=["default", "det"])
@pytest.mark.parametrize("case", list(CASES))
def test_tet_alpha_and_grads_match_fp64_reference(case, deterministic, mode):
    name, seed, cap = CASES[case]
    cpu, gc, gd, ga, frags, (ra, rfo, rbg) = tet_case(case)
    camera, vertex, intensity = TET_MODES[mode]
    with trail_cap(cap):
        _, _, alpha, g = tet_gpu(cpu, gc, gd, ga, seed=seed, det=deterministic, camera=camera, vertex=vertex,
                                 intensity=intensity)
    keep = (gd != 0)
    assert ((alpha.cpu().double() - ra).abs() * keep).max().item() <= ALPHA_TOL
    e = rel_l2(g["faces_opacity"].cpu().numpy(), rfo.numpy())
    assert e <= GRAD_TOL, "faces_opacity rel L2 %.3e" % e
    # the GPU's own weights: dL/dbg = sum (1 - alpha) dL_dC (1 - alpha = 1 on inactive pixels)
    want = ((1 - alpha.double()) * gc.cuda().double()).sum((0, 2, 3))
    assert torch.allclose(g["bg"].double(), want, rtol=1e-6, atol=1e-6 * want.abs().max().item())
    e = rel_l2(g["bg"].cpu().numpy(), rbg.numpy())
    assert e <= 1e-5, "bg rel L2 %.3e" % e


def test_tet_delaunay_seen_from_inside():
    from test_gpu_tet_general_meshes import BUILD
    cpu = BUILD["inside"]()._replace(bg=random_bg())
    gc, gd, frags = kept_cotangents(cpu, 0)
    keep = (gd != 0).float()
    ga = alpha_cotangent(gd) * keep
    ra, rfo, rbg = tet_reference(cpu, frags, gc, gd, ga)
    for det in (False, True):
        _, _, alpha, g = tet_gpu(cpu, gc, gd, ga, det=det)
        assert ((alpha.cpu().double() - ra).abs() * keep).max().item() <= ALPHA_TOL
        assert rel_l2(g["faces_opacity"].cpu().numpy(), rfo.numpy()) <= GRAD_TOL
        assert rel_l2(g["bg"].cpu().numpy(), rbg.numpy()) <= 1e-5


@pytest.mark.parametrize("deterministic", [False, True], ids=["default", "det"])
@pytest.mark.parametrize("case", ["small_tet", "jitter", "irregular"])
def test_tet_alpha_equals_a_white_render(case, deterministic):
    name, seed, _ = CASES[case]
    cpu, gc, gd, ga, _, _ = tet_case(case)
    z3, z1 = torch.zeros_like(gc), torch.zeros_like(gd)
    _, active, alpha, g = tet_gpu(cpu, z3, z1, ga, seed=seed, det=deterministic)
    color, _, _, gw = tet_gpu(_white(cpu), torch.cat([ga, z1, z1], 1), z1, None, seed=seed, det=deterministic,
                              return_alpha=False)
    assert (alpha - color[:, :1]).abs().max().item() <= ALPHA_TOL
    assert (alpha[:, 0][~active] == 0).all()
    e = rel_l2(g["faces_opacity"].cpu().numpy(), gw["faces_opacity"].cpu().numpy())
    assert e <= GRAD_TOL, e


@pytest.mark.parametrize("mode", list(TET_MODES))
def test_tet_other_grads_unchanged_and_opacity_linear(mode):
    cpu, gc, gd, ga, _, _ = tet_case("small_tet")
    camera, vertex, intensity = TET_MODES[mode]
    kw = dict(camera=camera, vertex=vertex, intensity=intensity)
    ga = ga * 0.9
    _, _, _, g0 = tet_gpu(cpu, gc, gd, None, det=True, return_alpha=False, **kw)
    _, _, _, g1 = tet_gpu(cpu, gc, gd, ga, det=True, **kw)
    for k, v in g0.items():
        if k in ("faces_opacity", "bg") or v is None:
            continue
        assert torch.equal(v, g1[k]), k
    for det in (False, True):
        _, _, _, a = tet_gpu(cpu, gc, gd, ga, det=det, **kw)
        _, _, _, b = tet_gpu(cpu, gc, gd, torch.zeros_like(ga), det=det, **kw)
        _, _, _, c = tet_gpu(cpu, torch.zeros_like(gc), torch.zeros_like(gd), ga, det=det, **kw)
        e = rel_l2(a["faces_opacity"].cpu().numpy(), (b["faces_opacity"] + c["faces_opacity"]).cpu().numpy())
        assert e <= 1e-5, (det, e)


@pytest.mark.parametrize("deterministic", [False, True], ids=["default", "det"])
def test_tet_background_grad(deterministic):
    cpu, gc, gd, ga, _, _ = tet_case("grid4")           # four views
    _, _, alpha, g = tet_gpu(cpu, gc, gd, ga, det=deterministic)
    _, _, _, g2 = tet_gpu(cpu, gc, gd, ga, det=deterministic)
    assert torch.equal(g["bg"], g2["bg"])
    s = scenes.to_device(cpu, "cuda")
    eps = 1e-2
    for c in range(3):
        d = torch.zeros(3)
        d[c] = eps
        ls = []
        for sign in (1, -1):
            col, _, _ = TetRenderer(TetRenderSettings(s.H, s.W, (cpu.bg + sign * d).cuda(), 0))(
                s.verts, s.faces, s.verts_color, s.faces_opacity, s.mv_mats, s.proj_mats, s.verts_depth, s.faces_intense,
                s.tets, s.face_tets, s.tet_faces)
            ls.append((col.double() * gc.cuda().double()).sum().item())
        cd = (ls[0] - ls[1]) / (2 * eps)
        assert abs(cd - g["bg"][c].item()) <= 1e-3 * max(1.0, abs(cd)), (c, cd, g["bg"][c].item())
    # nothing on screen: every pixel inactive, alpha 0, dL/dbg = sum dL_dC
    _, active, alpha, g = tet_gpu(_far_away(cpu), gc, gd, ga, det=deterministic)
    assert not active.any() and alpha.abs().max().item() == 0.0
    want = gc.double().sum((0, 2, 3))
    assert torch.allclose(g["bg"].cpu().double(), want, rtol=1e-6, atol=1e-6 * want.abs().max().item())
    # float64 background
    _, _, _, g64 = tet_gpu(cpu, gc, gd, ga, det=deterministic, bg=cpu.bg.double())
    assert g64["bg"].dtype == torch.float64


def test_tet_deterministic_range():
    cpu, gc, gd, ga, frags, _ = tet_case("small_tet")
    big = ga * 2.0 ** 20
    _, rfo, _ = tet_reference(cpu, frags, gc, gd, big)
    _, _, _, g = tet_gpu(cpu, gc, gd, big, det=True)
    assert torch.isfinite(g["faces_opacity"]).all()
    assert rel_l2(g["faces_opacity"].cpu().numpy(), rfo.numpy()) <= GRAD_TOL


# ---------------------------------------------------------------------------------------------- multi-view steps
def _cot3(color, depth, alpha):
    return color.detach() * 0.5 - 0.25, depth.detach() - 0.5, alpha.detach() - 0.5


def test_multiview_steps_with_alpha_and_bg_slot():
    """Inside PackedSceneGrads.direct() with a bg slot, one GPU: the steps equal plain autograd accumulation."""
    # tri
    s = scenes.to_device(scenes.config("small_tri"), "cuda")
    bg0 = random_bg().cuda()

    def tri_leaves():
        return [t.clone() for t in (s.verts, s.verts_color, s.faces_opacity)] + [bg0.clone()]

    v, vc, fo, bg = tri_leaves()
    sg = multiview.PackedSceneGrads(v, vc, fo, bg=bg)
    r = TriRenderer(TriRenderSettings(s.H, s.W, bg), return_alpha=True)
    multiview.multiview_step(r, sg, s.faces, s.mv_mats, s.proj_mats, s.verts_depth, s.faces_intense, _cot3,
                             views_per_call=1)
    ref = [t.requires_grad_() for t in tri_leaves()]
    r2 = TriRenderer(TriRenderSettings(s.H, s.W, ref[3]), return_alpha=True)
    for b in range(s.mv_mats.shape[0]):
        out = r2(ref[0], s.faces, ref[1], ref[2], s.mv_mats[b:b + 1], s.proj_mats[b:b + 1], s.verts_depth[b:b + 1],
                 s.faces_intense[b:b + 1])
        torch.autograd.backward(list(out), list(_cot3(*out)))
    flat = torch.cat([t.grad.reshape(-1) for t in ref])
    assert rel_l2(sg.flat.cpu().numpy(), flat.cpu().numpy()) <= 1e-5
    assert torch.allclose(bg.grad, ref[3].grad, rtol=1e-5, atol=1e-5)
    # tet, packed buffer without positions
    s = scenes.to_device(scenes.config("small_tet"), "cuda")

    def tet_leaves():
        return [t.clone() for t in (s.verts_color, s.faces_opacity)] + [bg0.clone()]

    vc, fo, bg = tet_leaves()
    sg = multiview.PackedSceneGrads(None, vc, fo, bg=bg)
    r = TetRenderer(TetRenderSettings(s.H, s.W, bg, 0), return_alpha=True)
    outs = multiview.tet_multiview_step(r, sg, s.verts, s.faces, s.tets, s.face_tets, s.tet_faces, s.mv_mats,
                                        s.proj_mats, s.verts_depth, s.faces_intense, _cot3, views_per_call=1)
    assert len(outs[0]) == 4
    ref = [t.requires_grad_() for t in tet_leaves()]
    r2 = TetRenderer(TetRenderSettings(s.H, s.W, ref[2], 0), return_alpha=True)
    for b in range(s.mv_mats.shape[0]):
        out = r2(s.verts, s.faces, ref[0], ref[1], s.mv_mats[b:b + 1], s.proj_mats[b:b + 1], s.verts_depth[b:b + 1],
                 s.faces_intense[b:b + 1], s.tets, s.face_tets, s.tet_faces, first_view=b)
        imgs = [out[0], out[1], out[3]]
        torch.autograd.backward(imgs, list(_cot3(*imgs)))
    flat = torch.cat([t.grad.reshape(-1) for t in ref])
    assert rel_l2(sg.flat.cpu().numpy(), flat.cpu().numpy()) <= 1e-5
