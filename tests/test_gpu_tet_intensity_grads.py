"""Tet renderer: gradients with respect to the face intensities (intensity_grads=True).

The yardstick is the fp64 reference of tests/test_tet_vertex_grads_reference.py (its `faces_intense` leaf), evaluated
on the fragments of the CPU oracle's march, and Euler's identity (tests/test_tet_intensity_grads_reference.py).  The
scenes get random per-view intensities, some of them 0.  Pixels whose GPU march parts from the oracle's get a zero
cotangent on both sides, as in tests/test_gpu_tet_camera_grads.py.
"""
import numpy as np
import pytest
import torch

import dmesh_renderer_b200 as dmr
from dmesh_renderer_b200 import TetRenderer, TetRenderSettings, _lib, scenes
from test_gpu_tet_camera_grads import (CASES, MAX_PARTED, SCENES, _stages, gpu_forward, grid4_scene, oracle_fragments,
                                       rel_l2, trail_cap)
from test_tet_intensity_grads_reference import euler_terms, fully_walked, with_intensities
from test_tet_vertex_grads_reference import reference_grads_verts, reference_render_verts

pytestmark = pytest.mark.gpu

f64 = torch.float64
INT_TOL = 1e-4
INT_STAGES = {"tet_march_backward_intensity", "tet_march_backward_camera_intensity",
              "tet_march_backward_vertex_intensity", "tet_march_backward_camera_vertex_intensity", "tet_intensity_finish"}
COMBOS = {"plain": (False, False), "camera": (True, False), "vertex": (False, True), "camera_vertex": (True, True)}


def gpu_run(cpu, gc, gd, seed=0, deterministic=False, intensity_grads=True, fint_grad=True, camera=False, vertex=False,
            scale=1.0):
    s = scenes.to_device(cpu, "cuda")
    v = s.verts.clone().requires_grad_(vertex)
    mv = s.mv_mats.detach().clone().requires_grad_(camera)
    pj = s.proj_mats.detach().clone().requires_grad_(camera)
    vc, fo = s.verts_color.clone().requires_grad_(), s.faces_opacity.clone().requires_grad_()
    fi = s.faces_intense.clone().requires_grad_(fint_grad)
    color, depth, active = TetRenderer(TetRenderSettings(s.H, s.W, s.bg, seed), deterministic=deterministic,
                                       vertex_grads=vertex, intensity_grads=intensity_grads)(
        v, s.faces, vc, fo, mv, pj, s.verts_depth, fi, s.tets, s.face_tets, s.tet_faces)
    torch.autograd.backward([color, depth], [gc.cuda() * scale, gd.cuda() * scale])
    return dict(faces_intense=fi.grad, verts=v.grad, verts_color=vc.grad, faces_opacity=fo.grad, mv_mats=mv.grad,
                proj_mats=pj.grad, color=color.detach())


def kept_cotangents(cpu, seed):
    """The scene's cotangents, zero at pixels whose GPU march parts from the oracle's; and the oracle's fragments."""
    gc, gd = scenes.cotangents(cpu)
    fw = gpu_forward(cpu, seed)
    frags, out = oracle_fragments(cpu, fw["coords"])
    assert out["mismatch"] == 0
    B, H, W = gd.shape[0], cpu.H, cpu.W
    parted = (fw["first_face"] != out["first_face"]) | (fw["n_contrib"] != frags["counts"]) | \
        (np.abs(fw["color"] - out["color"]).max(1).reshape(-1) > 1e-5) | \
        (np.abs(fw["depth"] - out["depth"]).reshape(-1) > 1e-5)
    assert parted.sum() <= MAX_PARTED, parted.sum()
    keep = torch.from_numpy(~parted).view(B, 1, H, W).float()
    return gc * keep, gd * keep, frags


_refs = {}


def reference_for(case):
    if case not in _refs:
        name, seed, _cap = CASES[case]
        cpu = with_intensities(SCENES[name]())
        gc, gd, frags = kept_cotangents(cpu, seed)
        _refs[case] = (cpu, gc, gd, reference_grads_verts(cpu, frags, gc, gd))
    return _refs[case]


@pytest.mark.parametrize("combo", list(COMBOS))
@pytest.mark.parametrize("deterministic", [False, True], ids=["default", "det"])
@pytest.mark.parametrize("case", list(CASES))
def test_intensity_grads_match_fp64_reference(case, deterministic, combo):
    name, seed, cap = CASES[case]
    camera, vertex = COMBOS[combo]
    cpu, gc, gd, (_, _, rg, _) = reference_for(case)
    with trail_cap(cap):
        g = gpu_run(cpu, gc, gd, seed=seed, deterministic=deterministic, camera=camera, vertex=vertex)
        torch.cuda.synchronize()
    for k in ("verts_color", "faces_opacity"):
        assert rel_l2(g[k].cpu().numpy(), rg[k].numpy()) <= 1e-4, k
    gi, ri = g["faces_intense"].cpu().numpy(), rg["faces_intense"].numpy()
    errs = [rel_l2(gi[b], ri[b]) for b in range(gi.shape[0])]
    print("\n[tet intensity grads] %s %s %s: max rel L2 over views %.2e" % (
        case, "det" if deterministic else "default", combo, max(errs)))
    assert all(np.abs(ri[b]).max() > 0 for b in range(ri.shape[0]))
    assert max(errs) <= INT_TOL, errs
    assert (g["verts"] is not None) == vertex and (g["mv_mats"] is not None) == camera


@pytest.mark.parametrize("deterministic", [False, True], ids=["default", "det"])
@pytest.mark.parametrize("name", ["tiny_tet", "small_tet", "grid4"])
def test_eulers_identity_on_gpu_gradients(name, deterministic):
    cpu = with_intensities(SCENES[name](), black=True)
    gc, gd, frags = kept_cotangents(cpu, 0)
    gc = gc * fully_walked(cpu, frags).float()
    g = gpu_run(cpu, gc, gd * 0, deterministic=deterministic)
    gi = g["faces_intense"].cpu()
    lhs, rhs, s = euler_terms(cpu.faces_intense, gi, gc, g["color"].cpu())
    print("\n[tet intensity Euler, GPU] %s %s: relative residual %s" % (
        name, "det" if deterministic else "default", ((lhs - rhs).abs() / s).tolist()))
    assert (s > 0).all()
    assert ((lhs - rhs).abs() <= 1e-5 * s).all()
    assert ((cpu.faces_intense == 0) & (gi != 0)).any()     # faces of intensity 0 get their gradient too


@pytest.mark.parametrize("case", ["small_tet", "short_trail", "jitter", "irregular"])
def test_other_gradients_with_and_without_intensity_grads(case):
    name, seed, cap = CASES[case]
    cpu = with_intensities(SCENES[name]())
    gc, gd = scenes.cotangents(cpu)
    kw = dict(seed=seed, camera=True, vertex=True)
    with trail_cap(cap):
        on = gpu_run(cpu, gc, gd, deterministic=True, **kw)
        off = gpu_run(cpu, gc, gd, deterministic=True, intensity_grads=False, **kw)
        on_d = gpu_run(cpu, gc, gd, **kw)
        off_d = gpu_run(cpu, gc, gd, intensity_grads=False, **kw)
        torch.cuda.synchronize()
    assert off["faces_intense"] is None and on["faces_intense"] is not None
    assert torch.equal(on["verts_color"], off["verts_color"])
    for k in ("verts_color", "faces_opacity", "mv_mats", "proj_mats", "verts"):
        assert rel_l2(on_d[k].cpu().numpy(), off_d[k].cpu().numpy()) <= 1e-6, k
        assert rel_l2(on[k].cpu().numpy(), off[k].cpu().numpy()) <= 1e-6, k


@pytest.mark.parametrize("deterministic", [False, True], ids=["default", "det"])
def test_opt_in_launches_and_stages(deterministic):
    cpu = with_intensities(grid4_scene())
    gc, gd = [t.cuda() for t in scenes.cotangents(cpu)]
    s = scenes.to_device(cpu, "cuda")
    lib = _lib.load()
    vc = s.verts_color.clone().requires_grad_()

    def run(intensity_grads, fint_grad, camera=False, vertex=False):
        v = s.verts.clone().requires_grad_(vertex)
        fi = s.faces_intense.clone().requires_grad_(fint_grad)
        mv = s.mv_mats.clone().requires_grad_(camera)
        r = TetRenderer(TetRenderSettings(s.H, s.W, s.bg, 0), deterministic=deterministic, vertex_grads=vertex,
                        intensity_grads=intensity_grads)
        color, depth, _ = r(v, s.faces, vc, s.faces_opacity, mv, s.proj_mats, s.verts_depth, fi, s.tets, s.face_tets,
                            s.tet_faces)
        torch.cuda.synchronize()
        _stages()
        n1 = lib.dmr_launch_count()
        torch.autograd.backward([color, depth], [gc, gd])
        n2 = lib.dmr_launch_count()
        torch.cuda.synchronize()
        return n2 - n1, _stages(), fi.grad

    run(False, False)                                     # warm-up: record cache, speculative binning buffer
    _lib.check(lib.dmr_profile_enable(1))
    try:
        for camera, vertex in COMBOS.values():
            today = run(False, False, camera, vertex)
            assert today[2] is None and not (today[1] & INT_STAGES)
            for flags in ((False, True), (True, False)):  # flag off with requires_grad, flag on without
                n, st, grad = run(*flags, camera, vertex)
                assert grad is None and n == today[0] and st == today[1], (flags, camera, vertex)
            n, st, grad = run(True, True, camera, vertex)
            assert grad is not None and torch.count_nonzero(grad) > 0
            stage = "tet_march_backward" + ("_camera" if camera else "") + ("_vertex" if vertex else "") + "_intensity"
            assert st & INT_STAGES == ({stage, "tet_intensity_finish"} if deterministic else {stage}), st
            assert st - INT_STAGES == today[1] - {stage.replace("_intensity", "")}, st
            assert n == today[0] + (1 if deterministic else 0)   # the fixed-point conversion
    finally:
        lib.dmr_profile_enable(0)


@pytest.mark.parametrize("name", ["small_tet", "grid4", "C3"])
def test_deterministic_reproducible_linear_and_poisoned(name):
    cpu = with_intensities({"grid4": grid4_scene}.get(name, lambda: scenes.config(name))())
    gc, gd = scenes.cotangents(cpu)
    runs = [gpu_run(cpu, gc, gd, deterministic=True)["faces_intense"] for _ in range(3)]
    for r in runs[1:]:
        assert torch.equal(r, runs[0])
    assert torch.isfinite(runs[0]).all() and torch.count_nonzero(runs[0]) > 0
    for sc in (2.0 ** -20, 0.125, 32.0):
        assert torch.equal(gpu_run(cpu, gc, gd, deterministic=True, scale=sc)["faces_intense"], runs[0] * sc), sc
    assert torch.count_nonzero(gpu_run(cpu, gc * 0, gd * 0, deterministic=True)["faces_intense"]) == 0
    for bad in (float("inf"), float("-inf"), float("nan")):
        gcb = gc.clone()
        gcb.view(-1)[gcb.numel() // 2] = bad
        assert torch.isnan(gpu_run(cpu, gcb, gd, deterministic=True)["faces_intense"]).all(), bad


@pytest.mark.parametrize("deterministic", [False, True], ids=["default", "det"])
def test_views_are_independent(deterministic):
    """The rows of a 4-view call are the gradients of the four single-view calls."""
    cpu = with_intensities(grid4_scene())
    gc, gd = scenes.cotangents(cpu)
    g = gpu_run(cpu, gc, gd, deterministic=deterministic)["faces_intense"]
    for b in range(cpu.mv_mats.shape[0]):
        sub = cpu._replace(mv_mats=cpu.mv_mats[b:b + 1], proj_mats=cpu.proj_mats[b:b + 1],
                           verts_depth=cpu.verts_depth[b:b + 1], faces_intense=cpu.faces_intense[b:b + 1])
        g1 = gpu_run(sub, gc[b:b + 1], gd[b:b + 1], deterministic=deterministic)["faces_intense"]
        assert rel_l2(g[b].cpu().numpy(), g1[0].cpu().numpy()) <= 1e-6, b


# ---------------------------------------------------------------------------------------------- public API
def lambert(verts, faces, lights):
    """|n_f . l_b| per view and face: lights [B,3] -> [B,F]; lights [3] (one light for every view) -> [F]."""
    p = verts[faces.long()]
    n = torch.linalg.cross(p[:, 1] - p[:, 0], p[:, 2] - p[:, 0])
    n = n / n.norm(dim=1, keepdim=True)
    return (n @ lights.T).T.abs() if lights.dim() == 2 else (n @ lights).abs()


VARIANTS = ["float32", "float64", "expanded"]


@pytest.mark.parametrize("deterministic", [False, True], ids=["default", "det"])
@pytest.mark.parametrize("variant", VARIANTS)
def test_lambertian_intensity_through_the_public_api(variant, deterministic):
    base = grid4_scene()
    B = base.mv_mats.shape[0]
    g = torch.Generator().manual_seed(3)
    lights = torch.randn(3 if variant == "expanded" else (B, 3), generator=g, dtype=f64)
    lights = lights / lights.norm(dim=-1, keepdim=True)
    fint64 = lambert(base.verts.to(f64), base.faces, lights)
    cpu = base._replace(faces_intense=fint64.expand(B, -1).float().contiguous())
    gc, gd, frags = kept_cotangents(cpu, 0)
    # fp64 reference, chained through the same function
    v64 = cpu.verts.to(f64).requires_grad_()
    d = lambda t: t.to(f64)
    color, _, _ = reference_render_verts(frags, cpu, v64.detach(), d(cpu.verts_color), d(cpu.faces_opacity),
                                         d(cpu.mv_mats), d(cpu.proj_mats), lambert(v64, cpu.faces, lights).expand(B, -1))
    color.backward(gc.to(f64))                            # depth does not depend on the intensities
    ref = v64.grad

    s = scenes.to_device(cpu, "cuda")
    dt = f64 if variant == "float64" else torch.float32

    def run(intensity_grads):
        v = s.verts.to(dt).clone().requires_grad_()
        fi = lambert(v, s.faces, lights.to("cuda", dt)).expand(B, -1)
        assert fi.dtype == dt and (fi.stride(0) == 0) == (variant == "expanded")
        color, depth, _ = TetRenderer(TetRenderSettings(s.H, s.W, s.bg, 0), deterministic=deterministic,
                                      intensity_grads=intensity_grads)(
            v, s.faces, s.verts_color, s.faces_opacity, s.mv_mats, s.proj_mats, s.verts_depth, fi, s.tets,
            s.face_tets, s.tet_faces)
        torch.autograd.backward([color, depth], [gc.cuda(), gd.cuda()])
        return v.grad

    gv = run(True)
    assert gv.dtype == dt
    e = rel_l2(gv.cpu().numpy(), ref.numpy())
    print("\n[tet intensity grads, Lambertian] %s %s: verts rel L2 %.2e" % (
        variant, "det" if deterministic else "default", e))
    assert ref.abs().max() > 0 and e <= 1e-4
    assert run(False) is None
    old = dmr.set_tet_intensity_grads(True)
    try:
        assert torch.equal(run(None), gv) if deterministic else run(None) is not None
    finally:
        assert dmr.set_tet_intensity_grads(old) is True
