"""Tet renderer: gradients with respect to the vertex positions (vertex_grads=True).

The yardstick is the fp64 reference of tests/test_tet_vertex_grads_reference.py (the camera-gradient tests' reference
with a `verts` leaf), evaluated on the fragments of the CPU oracle's march.  Pixels whose GPU march parts from the
oracle's get a zero cotangent on both sides, as in tests/test_gpu_tet_camera_grads.py.
"""
import ctypes

import numpy as np
import pytest
import torch

import dmesh_renderer_b200 as dmr
from dmesh_renderer_b200 import TetRenderer, TetRenderSettings, _C, _lib, scenes
from test_gpu_tet_camera_grads import (CASES, MAX_PARTED, SCENES, _stages, gpu_forward, grid4_scene, oracle_fragments,
                                       rel_l2, trail_cap)
from test_tet_vertex_grads_reference import reference_grads_verts, rigid_residual

pytestmark = pytest.mark.gpu

VERT_TOL = 1e-3
VERT_STAGES = {"tet_march_backward_vertex", "tet_march_backward_camera_vertex", "tet_vertex_finish"}


def gpu_run(cpu, gc, gd, seed=0, deterministic=False, vertex_grads=True, verts_grad=True, camera=False, scale=1.0):
    s = scenes.to_device(cpu, "cuda")
    v = s.verts.clone().requires_grad_(verts_grad)
    mv = s.mv_mats.detach().clone().requires_grad_(camera)
    pj = s.proj_mats.detach().clone().requires_grad_(camera)
    vc, fo = s.verts_color.clone().requires_grad_(), s.faces_opacity.clone().requires_grad_()
    color, depth, active = TetRenderer(TetRenderSettings(s.H, s.W, s.bg, seed), deterministic=deterministic,
                                       vertex_grads=vertex_grads)(
        v, s.faces, vc, fo, mv, pj, s.verts_depth, s.faces_intense, s.tets, s.face_tets, s.tet_faces)
    torch.autograd.backward([color, depth], [gc.cuda() * scale, gd.cuda() * scale])
    return dict(verts=v.grad, verts_color=vc.grad, faces_opacity=fo.grad, mv_mats=mv.grad, proj_mats=pj.grad)


_refs = {}


def reference_for(case):
    if case not in _refs:
        name, seed, _cap = CASES[case]
        cpu = SCENES[name]()
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
        gc, gd = gc * keep, gd * keep
        _refs[case] = (cpu, gc, gd, reference_grads_verts(cpu, frags, gc, gd))
    return _refs[case]


@pytest.mark.parametrize("camera", [False, True], ids=["plain", "camera"])
@pytest.mark.parametrize("deterministic", [False, True], ids=["default", "det"])
@pytest.mark.parametrize("case", list(CASES))
def test_vertex_grads_match_fp64_reference(case, deterministic, camera):
    name, seed, cap = CASES[case]
    cpu, gc, gd, (_, _, rg, grazing) = reference_for(case)
    with trail_cap(cap):
        g = gpu_run(cpu, gc, gd, seed=seed, deterministic=deterministic, camera=camera)
        torch.cuda.synchronize()
    for k in ("verts_color", "faces_opacity"):
        assert rel_l2(g[k].cpu().numpy(), rg[k].numpy()) <= 1e-4, k
    gv, rv = g["verts"].cpu().numpy(), rg["verts"].numpy()
    # vertices of faces walked at a grazing angle (|rd.n| < 1e-2 |n|) are left out on both sides: there the fp32
    # (t, u, v) are ill-conditioned (the gradient grows like 1 / D), which the fp64 reference does not reproduce
    keep = np.ones(gv.shape[0], bool)
    keep[cpu.faces.long()[grazing].reshape(-1).numpy()] = False
    e, e_all = rel_l2(gv[keep], rv[keep]), rel_l2(gv, rv)
    print("\n[tet vertex grads] %s %s %s: rel L2 %.2e (%d grazing faces left out), %.2e with them" % (
        case, "det" if deterministic else "default", "camera" if camera else "plain", e, grazing.numel(), e_all))
    assert np.abs(rv).max() > 0 and keep.mean() > 0.9
    assert e <= VERT_TOL
    if camera:
        for k in ("mv_mats", "proj_mats"):
            for b in range(cpu.mv_mats.shape[0]):
                assert rel_l2(g[k][b].cpu().numpy(), rg[k][b].numpy()) <= 1e-3, (k, b)


@pytest.mark.parametrize("deterministic", [False, True], ids=["default", "det"])
@pytest.mark.parametrize("name", ["tiny_tet", "small_tet", "grid4"])
def test_rigid_motion_identity_on_gpu_gradients(name, deterministic):
    cpu = {"grid4": grid4_scene}.get(name, lambda: scenes.config(name))()
    gc, gd = scenes.cotangents(cpu)
    g = gpu_run(cpu, gc, gd, deterministic=deterministic, camera=True)
    gv, gm = g["verts"].cpu(), g["mv_mats"].cpu()
    r, s, sv = rigid_residual(cpu.verts, cpu.mv_mats, gv, gm)
    r0, s0, _ = rigid_residual(cpu.verts, cpu.mv_mats, torch.zeros_like(gv), gm)   # negative control
    print("\n[tet rigid motion, GPU] %s %s: residual %.2e of %.2e (without dL/dverts: %.2e)" % (
        name, "det" if deterministic else "default", r / s, s, r0 / s0))
    assert sv > 0.01 * s
    assert r <= 1e-5 * s
    assert r0 >= 1e-2 * s0


@pytest.mark.parametrize("case", ["small_tet", "short_trail", "jitter", "irregular"])
def test_other_gradients_with_and_without_vertex_grads(case):
    name, seed, cap = CASES[case]
    cpu = SCENES[name]()
    gc, gd = scenes.cotangents(cpu)
    with trail_cap(cap):
        on = gpu_run(cpu, gc, gd, seed=seed, deterministic=True, camera=True)
        off = gpu_run(cpu, gc, gd, seed=seed, deterministic=True, camera=True, vertex_grads=False)
        on_d = gpu_run(cpu, gc, gd, seed=seed, camera=True)
        off_d = gpu_run(cpu, gc, gd, seed=seed, camera=True, vertex_grads=False)
        torch.cuda.synchronize()
    assert off["verts"] is None and on["verts"] is not None
    assert torch.equal(on["verts_color"], off["verts_color"])
    for k in ("verts_color", "faces_opacity", "mv_mats", "proj_mats"):
        assert rel_l2(on_d[k].cpu().numpy(), off_d[k].cpu().numpy()) <= 1e-6, k
        assert rel_l2(on[k].cpu().numpy(), off[k].cpu().numpy()) <= 1e-6, k


@pytest.mark.parametrize("deterministic", [False, True], ids=["default", "det"])
def test_opt_in_launches_and_stages(deterministic):
    cpu = grid4_scene()
    gc, gd = [t.cuda() for t in scenes.cotangents(cpu)]
    s = scenes.to_device(cpu, "cuda")
    lib = _lib.load()
    vc = s.verts_color.clone().requires_grad_()

    def run(vertex_grads, verts_grad):
        v = s.verts.clone().requires_grad_(verts_grad)
        r = TetRenderer(TetRenderSettings(s.H, s.W, s.bg, 0), deterministic=deterministic, vertex_grads=vertex_grads)
        color, depth, _ = r(v, s.faces, vc, s.faces_opacity, s.mv_mats, s.proj_mats, s.verts_depth, s.faces_intense,
                            s.tets, s.face_tets, s.tet_faces)
        torch.cuda.synchronize()
        _stages()
        n1 = lib.dmr_launch_count()
        torch.autograd.backward([color, depth], [gc, gd])
        n2 = lib.dmr_launch_count()
        torch.cuda.synchronize()
        return n2 - n1, _stages(), v.grad

    run(False, False)                                     # warm-up: record cache, speculative binning buffer
    _lib.check(lib.dmr_profile_enable(1))
    try:
        today = run(False, False)
        assert today[2] is None and not (today[1] & VERT_STAGES) and "tet_march_backward" in today[1]
        for flags in ((False, True), (True, False)):      # flag off with requires_grad, flag on without
            n, st, grad = run(*flags)
            assert grad is None and n == today[0] and st == today[1], flags
        n, st, grad = run(True, True)
        assert grad is not None and torch.count_nonzero(grad) > 0
        assert {"tet_march_backward_vertex", "tet_vertex_finish"} <= st and "tet_march_backward" not in st
        assert n == today[0] + 1                          # the position fold
    finally:
        lib.dmr_profile_enable(0)


def test_process_wide_switch_and_float64_verts():
    cpu = scenes.config("tiny_tet")
    gc, gd = scenes.cotangents(cpu)
    ref = gpu_run(cpu, gc, gd, deterministic=True)["verts"]
    s = scenes.to_device(cpu, "cuda")
    old = dmr.set_tet_vertex_grads(True)
    try:
        v = s.verts.double().requires_grad_()
        color, depth, _ = TetRenderer(TetRenderSettings(s.H, s.W, s.bg, 0), deterministic=True)(
            v, s.faces, s.verts_color, s.faces_opacity, s.mv_mats, s.proj_mats, s.verts_depth, s.faces_intense, s.tets,
            s.face_tets, s.tet_faces)
        torch.autograd.backward([color, depth], [gc.cuda(), gd.cuda()])
    finally:
        assert dmr.set_tet_vertex_grads(old) is True
    assert v.grad.dtype == torch.float64 and torch.equal(v.grad.float(), ref)


@pytest.mark.parametrize("name", ["small_tet", "grid4", "C3"])
def test_deterministic_reproducible_linear_and_poisoned(name):
    cpu = {"grid4": grid4_scene}.get(name, lambda: scenes.config(name))()
    gc, gd = scenes.cotangents(cpu)
    runs = [gpu_run(cpu, gc, gd, deterministic=True)["verts"] for _ in range(4)]
    for r in runs[1:]:
        assert torch.equal(r, runs[0])
    assert torch.isfinite(runs[0]).all() and torch.count_nonzero(runs[0]) > 0
    for sc in (2.0 ** -20, 0.125, 32.0):
        assert torch.equal(gpu_run(cpu, gc, gd, deterministic=True, scale=sc)["verts"], runs[0] * sc), sc
    assert torch.count_nonzero(gpu_run(cpu, gc * 0, gd * 0, deterministic=True)["verts"]) == 0
    for bad in (float("inf"), float("-inf"), float("nan")):
        gcb = gc.clone()
        gcb.view(-1)[gcb.numel() // 2] = bad
        assert torch.isnan(gpu_run(cpu, gcb, gd, deterministic=True)["verts"]).all(), bad


@pytest.mark.parametrize("deterministic", [False, True], ids=["default", "det"])
def test_multiview_call_is_the_sum_of_single_views(deterministic):
    cpu = grid4_scene()
    gc, gd = scenes.cotangents(cpu)
    g = gpu_run(cpu, gc, gd, deterministic=deterministic)["verts"]
    total = torch.zeros_like(g)
    for b in range(cpu.mv_mats.shape[0]):
        sub = cpu._replace(mv_mats=cpu.mv_mats[b:b + 1], proj_mats=cpu.proj_mats[b:b + 1],
                           verts_depth=cpu.verts_depth[b:b + 1], faces_intense=cpu.faces_intense[b:b + 1])
        total += gpu_run(sub, gc[b:b + 1], gd[b:b + 1], deterministic=deterministic)["verts"]
    assert rel_l2(g.cpu().numpy(), total.cpu().numpy()) <= 1e-6


def test_workspace_one_byte_short_is_rejected():
    lib = _lib.load()
    cpu = scenes.config("tiny_tet")
    s = scenes.to_device(cpu, "cuda")
    mv, pj = s.mv_mats.transpose(1, 2).contiguous(), s.proj_mats.transpose(1, 2).contiguous()
    imv, ipj = torch.inverse(mv), torch.inverse(pj)
    out = _C.render_tets(s.bg, s.verts, s.faces, s.verts_color, s.faces_opacity, mv, pj, imv, ipj, s.verts_depth,
                         s.faces_intense, s.tets, s.face_tets, s.tet_faces, s.H, s.W, 0)
    gc, gd = [t.cuda() for t in scenes.cotangents(cpu)]
    B, P, F, T = mv.shape[0], s.verts.shape[0], s.faces.shape[0], s.tets.shape[0]
    p = lambda t: ctypes.c_void_p(t.data_ptr())
    null = ctypes.c_void_p(0)
    stream = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    for det in (0, 1):
        for cam in (0, 1):
            gv, go, gm = torch.zeros(P, 3, device="cuda"), torch.zeros(F, device="cuda"), torch.zeros(2, B, 16, device="cuda")
            dv = torch.zeros(P, 3, device="cuda")
            need = lib.dmr_tet_backward_vertex_bytes(B, P, F, s.W, s.H, det, cam)
            ws = torch.empty(need, dtype=torch.uint8, device="cuda")
            a = (B, P, F, T, s.W, s.H, 0, p(s.bg), p(mv), p(pj), p(imv), p(ipj), p(s.faces_intense), p(out[3]), p(out[4]),
                 p(out[4].tet_records), p(out[6]), p(gc), p(gd), p(gv), p(go), det)
            c = (p(gm[0]), p(gm[1])) if cam else (null, null)
            n0 = lib.dmr_launch_count()
            assert lib.dmr_tet_backward_vertex(*a, *c, p(dv), p(ws), need - 1, stream) == 1
            assert b"dmr_tet_backward_vertex_bytes" in lib.dmr_last_error()
            torch.cuda.synchronize()
            assert lib.dmr_launch_count() == n0
            assert torch.count_nonzero(gv) == 0 and torch.count_nonzero(dv) == 0 and torch.count_nonzero(gm) == 0
            assert lib.dmr_tet_backward_vertex(*a, *c, p(dv), p(ws), need, stream) == 0
            torch.cuda.synchronize()
            assert torch.count_nonzero(dv) > 0 and torch.count_nonzero(gv) > 0


def test_record_cache_follows_an_optimiser_step():
    """With vertex gradients the optimiser changes verts in place every step: the version counter moves, the cached
    adjacency records miss and are rebuilt, and the images equal those of a render with an empty cache."""
    cpu = scenes.config("small_tet")
    gc, gd = [t.cuda() for t in scenes.cotangents(cpu)]
    s = scenes.to_device(cpu, "cuda")
    v = s.verts.clone().requires_grad_()
    r = TetRenderer(TetRenderSettings(s.H, s.W, s.bg, 0), vertex_grads=True)
    render = lambda: r(v, s.faces, s.verts_color, s.faces_opacity, s.mv_mats, s.proj_mats, s.verts_depth,
                       s.faces_intense, s.tets, s.face_tets, s.tet_faces)
    opt = torch.optim.SGD([v], lr=1e-3)
    color, depth, _ = render()
    torch.autograd.backward([color, depth], [gc, gd])
    before = v._version
    opt.step()
    assert v._version > before
    c1, d1, a1 = render()
    _C._TetRecordCache.clear()
    c2, d2, a2 = render()
    torch.cuda.synchronize()
    assert torch.equal(c1, c2) and torch.equal(d1, d2) and torch.equal(a1, a2)
    assert not torch.equal(c1, color.detach())
