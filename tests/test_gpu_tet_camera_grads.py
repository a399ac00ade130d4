"""Tet renderer: gradients with respect to the camera matrices (mv_mats, proj_mats).

The yardstick is an fp64 re-implementation of the forward function as implemented, evaluated on exactly the
fragments the renderer composites (taken from the CPU oracle by tests/tet_fragments.cpp: per pixel, in compositing
order, the faces the march crosses, each flagged by whether the backward pass walks it) and differentiated by torch
autograd.  The discrete decisions -- the marched path, n_contrib, termination, the active mask and the clamp regions --
are held fixed, as in the renderer's own gradients; every input of a step the backward pass does not walk is
detached.  Before its camera gradients are trusted, the reference has to reproduce the GPU's images at active pixels
(IMG_TOL) and its gradients for colours and opacities (GRAD_TOL relative L2).
"""
import ctypes

import numpy as np
import pytest
import torch

import tet_fragments
from dmesh_renderer_b200 import TetRenderer, TetRenderSettings, _C, _lib, debug, scenes

pytestmark = pytest.mark.gpu

# IMG_TOL: the reference evaluates the fp32 renderer's steps in fp64
IMG_TOL, GRAD_TOL, CAM_TOL = 1e-4, 1e-4, 1e-3
f64 = torch.float64
CAM_KEYS = ("mv_mats", "proj_mats")


def rel_l2(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return float(np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-30))


def with_irregular_tets(s, nfaces=40, shift=2e-3, seed=5):
    """A copy of scene `s` (on the CPU) whose tables are INCONSISTENT for `nfaces` interior faces: the face's first
    vertex is replaced by a slightly shifted copy of it, so both tets next to the face have a side that is not made of
    their own four vertices (the march takes its out-of-line path there).  As in test_gpu_tet_vs_reference.py."""
    g = torch.Generator().manual_seed(seed)
    interior = ((s.face_tets[:, 0] >= 0) & (s.face_tets[:, 1] >= 0)).nonzero().flatten()
    pick = interior[torch.randperm(interior.numel(), generator=g)[:nfaces]]
    faces = s.faces.clone()
    old = faces[pick, 0].long()
    P = s.verts.shape[0]
    new_ids = torch.arange(P, P + pick.numel(), dtype=faces.dtype)
    faces[pick, 0] = new_ids
    verts = torch.cat([s.verts, s.verts[old] + shift * (torch.rand(pick.numel(), 3, generator=g) - 0.5)])
    verts_color = torch.cat([s.verts_color, torch.rand(pick.numel(), 3, generator=g)])
    verts_depth = torch.cat([s.verts_depth, s.verts_depth[:, old]], dim=1)
    return s._replace(verts=verts.contiguous(), faces=faces.contiguous(), verts_color=verts_color.contiguous(),
                      verts_depth=verts_depth.contiguous())


def grid4_scene():
    """Four views of a tet grid on a non-multiple-of-16 image."""
    return scenes.tet_grid_scene("grid4", 3, 8, 72, 88, B=4, opacity=(0.0, 0.3))


SCENES = {"tiny_tet": lambda: scenes.config("tiny_tet"), "small_tet": lambda: scenes.config("small_tet"),
          "grid4": grid4_scene, "irregular": lambda: with_irregular_tets(scenes.config("small_tet"))}
# case -> (scene, ray_random_seed, face-trail cap)
CASES = {"tiny_tet": ("tiny_tet", 0, 0), "small_tet": ("small_tet", 0, 0), "grid4": ("grid4", 0, 0),
         "jitter": ("small_tet", 7, 0), "short_trail": ("small_tet", 0, 3), "irregular": ("irregular", 0, 0)}


# ---------------------------------------------------------------------------------------------- fp64 reference
def oracle_fragments(cpu, coords=None, gradients=None):
    """Fragments of tet scene `cpu` (matrices as the renderer sees them: transposed, inverted with torch.inverse)."""
    mv, pj = cpu.mv_mats.transpose(1, 2).contiguous(), cpu.proj_mats.transpose(1, 2).contiguous()
    mats = [np.ascontiguousarray(m.numpy(), np.float32) for m in (mv, pj, torch.inverse(mv), torch.inverse(pj))]
    return tet_fragments.tet_fragments(cpu, mats, coords, gradients)


def _pix2ndc(v, S):
    # pix2ndc (common.cuh): evaluated in double, rounded to fp32
    return torch.from_numpy((((v.astype(np.float64) * 2.0 + 1.0) / S) - 1.0).astype(np.float32)).to(f64)


def _clamp_w(w):
    eps = 1e-4
    wd = w.detach()
    return torch.where((wd >= 0) & (wd < eps), torch.full_like(w, eps),
                       torch.where((wd < 0) & (wd > -eps), torch.full_like(w, -eps), w))


def reference_render(frags, cpu, vcol, fopa, mv, proj, fint):
    """fp64 colour [B,3,H,W] and depth [B,1,H,W] from the fragments; vcol [P,3], fopa [F], fint [B,F] and the matrices
    mv, proj ([B,4,4], maths convention) may require grad.  Inputs of steps the backward pass does not walk are
    detached."""
    B, H, W = cpu.mv_mats.shape[0], cpu.H, cpu.W
    HW, BI = H * W, B * H * W
    active = torch.from_numpy(frags["active"])
    cnt_all = torch.from_numpy(frags["counts"].astype(np.int64))
    keep = torch.repeat_interleave(active, cnt_all)                      # inactive pixels composite nothing
    cnt = cnt_all * active
    N = int(cnt.sum())
    pix = torch.repeat_interleave(torch.arange(BI), cnt)
    starts = torch.cumsum(cnt, 0) - cnt
    rank = torch.arange(N) - starts[pix]
    f = torch.from_numpy(frags["face"].astype(np.int64))[keep]
    r = torch.from_numpy(frags["reach"])[keep]
    b = pix // HW
    sel = lambda x: torch.where(r.view(-1, *([1] * (x.dim() - 1))), x, x.detach())
    # rays: pixel_ray<true> (common.cuh) through the exported pixel coordinates
    xy = frags["coords"][pix.numpy()]
    n = torch.stack([_pix2ndc(xy[:, 0], W), _pix2ndc(xy[:, 1], H), -torch.ones(N, dtype=f64), torch.ones(N, dtype=f64)], 1)
    # the values of the fp32 inverses the renderer uses, the derivative of the fp64 inverse
    inv_mv, inv_pj = [torch.linalg.inv(m) + (torch.inverse(m.detach().float()).double() - torch.linalg.inv(m.detach()))
                      for m in (mv, proj)]
    pv = torch.einsum("nij,nj->ni", inv_pj[b][:, :3, :], n)                 # pv.w is ignored
    d = torch.einsum("nij,nj->ni", inv_mv[b][:, :3, :3], pv)
    ro = sel(inv_mv[b][:, :3, 3])
    rd = sel(d / d.norm(dim=1, keepdim=True).clamp_min(1e-4))
    # (t, u, v): Moeller-Trumbore against the face's triangle in faces[] order
    fv = cpu.faces.long()[f]
    vv = cpu.verts.to(f64)
    p0, p1, p2 = vv[fv[:, 0]], vv[fv[:, 1]], vv[fv[:, 2]]
    T, E1, E2 = ro - p0, p1 - p0, p2 - p0
    Pv, Q = torch.linalg.cross(rd, E2), torch.linalg.cross(T, E1)
    D = (Pv * E1).sum(1)
    t, u, v = (Q * E2).sum(1) / D, (Pv * T).sum(1) / D, (Q * rd).sum(1) / D
    c = sel(vcol[fv])                                                        # [N,3,3]
    col = (c[:, 0] + (c[:, 1] - c[:, 0]) * u[:, None] + (c[:, 2] - c[:, 0]) * v[:, None]) * sel(fint[b, f])[:, None]
    # hit-point depth: xform43 with mv, then the z and w rows of proj, z / clamp_w(w)
    mvf, pjf = sel(mv[b]), sel(proj[b])
    pt = ro + t[:, None] * rd
    pm = torch.einsum("nij,nj->ni", mvf[:, :3, :3], pt) + mvf[:, :3, 3]
    z = (pjf[:, 2, :3] * pm).sum(1) + pjf[:, 2, 3]
    w = (pjf[:, 3, :3] * pm).sum(1) + pjf[:, 3, 3]
    pd = z / _clamp_w(w)
    alpha = sel(fopa[f])
    # front-to-back compositing per pixel on a dense [pixels with fragments, max fragments] layout
    live, slot = torch.unique(pix, return_inverse=True)
    K = int(cnt.max()) if N else 1
    dense = lambda vals: torch.zeros(live.numel(), K, *vals.shape[1:], dtype=f64).index_put((slot, rank), vals)
    a = dense(alpha)
    Tc = torch.cumprod(1 - a, 1)
    Tx = torch.cat([torch.ones(live.numel(), 1, dtype=f64), Tc[:, :-1]], 1)
    wgt = a * Tx
    C = (dense(col) * wgt[..., None]).sum(1)
    Dp = (dense(pd) * wgt).sum(1)
    Tf = Tc[:, -1]
    bg = cpu.bg.to(f64)
    color = bg[None, :].expand(BI, 3).index_put((live,), C + Tf[:, None] * bg[None, :])
    depth = torch.ones(BI, dtype=f64).index_put((live,), Dp + Tf)
    return color.view(B, H, W, 3).permute(0, 3, 1, 2), depth.view(B, 1, H, W)


def reference_grads(cpu, frags, gc, gd):
    """fp64 reference forward + backward.  Returns (color, depth, {name: grad})."""
    L = {k: getattr(cpu, k).to(f64).clone().requires_grad_() for k in
         ("verts_color", "faces_opacity", "mv_mats", "proj_mats", "faces_intense")}
    color, depth = reference_render(frags, cpu, L["verts_color"], L["faces_opacity"], L["mv_mats"], L["proj_mats"],
                                    L["faces_intense"])
    torch.autograd.backward([color, depth], [gc.to(f64), gd.to(f64)])
    grads = {k: (t.grad if t.grad is not None else torch.zeros_like(t)) for k, t in L.items()}
    return color.detach(), depth.detach(), grads


# ---------------------------------------------------------------------------------------------- GPU side
def gpu_run(cpu, gc, gd, seed=0, deterministic=False, mv_grad=True, pj_grad=True, scale=1.0):
    s = scenes.to_device(cpu, "cuda")
    mv = s.mv_mats.detach().clone().requires_grad_(mv_grad)
    pj = s.proj_mats.detach().clone().requires_grad_(pj_grad)
    vc, fo = s.verts_color.clone().requires_grad_(), s.faces_opacity.clone().requires_grad_()
    color, depth, active = TetRenderer(TetRenderSettings(s.H, s.W, s.bg, seed), deterministic=deterministic)(
        s.verts, s.faces, vc, fo, mv, pj, s.verts_depth, s.faces_intense, s.tets, s.face_tets, s.tet_faces)
    torch.autograd.backward([color, depth], [gc.cuda() * scale, gd.cuda() * scale])
    g = dict(verts_color=vc.grad, faces_opacity=fo.grad, mv_mats=mv.grad, proj_mats=pj.grad)
    return color.detach(), depth.detach(), active, g


class trail_cap:
    """dmr_debug_set_tet_trail_cap(cap) for the duration of a block (0 = automatic)."""

    def __init__(self, cap):
        self.cap = cap

    def __enter__(self):
        _lib.load().dmr_debug_set_tet_trail_cap(self.cap)

    def __exit__(self, *exc):
        _lib.load().dmr_debug_set_tet_trail_cap(0)
        return False


def gpu_forward(cpu, seed):
    """The GPU forward's images, first_face, n_contrib and (seed > 0) jittered pixel coordinates [B*H*W, 2]."""
    s = scenes.to_device(cpu, "cuda")
    mv, pj = s.mv_mats.transpose(1, 2), s.proj_mats.transpose(1, 2)
    out = _C.render_tets(s.bg, s.verts, s.faces, s.verts_color, s.faces_opacity, mv, pj, torch.inverse(mv),
                         torch.inverse(pj), s.verts_depth, s.faces_intense, s.tets, s.face_tets, s.tet_faces, s.H, s.W,
                         seed)
    d = dict(B=s.mv_mats.shape[0], P=s.verts.shape[0], F=s.faces.shape[0], W=s.W, H=s.H, T=s.tets.shape[0])
    return dict(color=out[0].cpu().numpy(), depth=out[1].cpu().numpy(),
                first_face=debug.view("tet", "first_face", out[6], **d),
                n_contrib=debug.view("tet", "n_contrib", out[6], **d),
                coords=debug.view("tet", "tet_jitter", out[6], **d).copy() if seed > 0 else None)


# Pixels whose GPU march parts from the oracle's (a different first face or step count, or images beyond the forward
# parity tolerance of test_gpu_tet_vs_reference.py: fp-level ties in a hit or normal-sign test of a grazing ray) are
# compared on different fragments; they get a zero cotangent on both sides, and there may be at most this many.
MAX_PARTED = 4

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
        _refs[case] = (cpu, gc, gd, frags, torch.from_numpy(~parted).view(B, H, W),
                       reference_grads(cpu, frags, gc, gd))
        print("\n[tet camera grads] %s: %d pixel(s) parted from the oracle's march" % (case, int(parted.sum())))
    return _refs[case]


@pytest.mark.parametrize("deterministic", [False, True], ids=["default", "det"])
@pytest.mark.parametrize("case", list(CASES))
def test_camera_grads_match_fp64_reference(case, deterministic):
    name, seed, cap = CASES[case]
    cpu, gc, gd, frags, same, (rc, rdp, rg) = reference_for(case)
    with trail_cap(cap):
        color, depth, active, g = gpu_run(cpu, gc, gd, seed=seed, deterministic=deterministic)
        torch.cuda.synchronize()
    act = torch.from_numpy(frags["active"]).view(active.shape)
    assert torch.equal(active.cpu()[same], act[same])
    assert act.float().mean().item() > 0.3
    # self-checks of the reference
    m = (act & same)[:, None]
    assert (color.cpu().double() - rc).abs().masked_select(m).max().item() <= IMG_TOL
    assert (depth.cpu().double() - rdp).abs().masked_select(m).max().item() <= IMG_TOL
    for k in ("verts_color", "faces_opacity"):
        e = rel_l2(g[k].cpu().numpy(), rg[k].numpy())
        assert e <= GRAD_TOL, "%s rel L2 %.3e" % (k, e)
    # camera gradients, per view
    errs = {}
    for k in CAM_KEYS:
        errs[k] = []
        for b in range(cpu.mv_mats.shape[0]):
            e = rel_l2(g[k][b].cpu().numpy(), rg[k][b].numpy())
            errs[k].append(e)
            assert e <= CAM_TOL, "%s view %d rel L2 %.3e" % (k, b, e)
    print("\n[tet camera grads] %s %s: max rel L2 mv %.2e proj %.2e (%d walked of %d fragments)" % (
        case, "det" if deterministic else "default", max(errs["mv_mats"]), max(errs["proj_mats"]),
        int(frags["reach"].sum()), len(frags["reach"])))


# ---------------------------------------------------------------------------------------------- properties
PROPERTY_SCENES = {"small_tet": lambda: scenes.config("small_tet"), "grid4": grid4_scene, "C3": lambda: scenes.config("C3")}


@pytest.mark.parametrize("deterministic", [False, True], ids=["default", "det"])
@pytest.mark.parametrize("name", list(PROPERTY_SCENES))
def test_reproducible_and_linear(name, deterministic):
    cpu = PROPERTY_SCENES[name]()
    gc, gd = scenes.cotangents(cpu)
    runs = [gpu_run(cpu, gc, gd, deterministic=deterministic)[3] for _ in range(4)]
    for r in runs[1:]:
        for k in CAM_KEYS:
            assert torch.equal(r[k], runs[0][k]), k
    for k in CAM_KEYS:
        assert torch.isfinite(runs[0][k]).all() and torch.count_nonzero(runs[0][k]) > 0
    # power-of-two cotangent scales: no float atomics and only linear operations on the camera path
    for sc in (2.0 ** -20, 0.125, 32.0):
        g = gpu_run(cpu, gc, gd, deterministic=deterministic, scale=sc)[3]
        for k in CAM_KEYS:
            assert torch.equal(g[k], runs[0][k] * sc), (k, sc)
    zero = gpu_run(cpu, gc * 0, gd * 0, deterministic=deterministic)[3]
    for k in CAM_KEYS:
        assert torch.count_nonzero(zero[k]) == 0


@pytest.mark.parametrize("deterministic", [False, True], ids=["default", "det"])
def test_views_are_independent(deterministic):
    """A 4-view call gives each view exactly the camera gradients of its single-view call."""
    cpu = grid4_scene()
    gc, gd = scenes.cotangents(cpu)
    g = gpu_run(cpu, gc, gd, deterministic=deterministic)[3]
    for b in range(cpu.mv_mats.shape[0]):
        sub = cpu._replace(mv_mats=cpu.mv_mats[b:b + 1], proj_mats=cpu.proj_mats[b:b + 1],
                           verts_depth=cpu.verts_depth[b:b + 1], faces_intense=cpu.faces_intense[b:b + 1])
        g1 = gpu_run(sub, gc[b:b + 1], gd[b:b + 1], deterministic=deterministic)[3]
        for k in CAM_KEYS:
            assert torch.equal(g[k][b], g1[k][0]), (k, b)


@pytest.mark.parametrize("deterministic", [False, True], ids=["default", "det"])
def test_only_one_matrix_requires_grad(deterministic):
    cpu = scenes.config("small_tet")
    gc, gd = scenes.cotangents(cpu)
    both = gpu_run(cpu, gc, gd, deterministic=deterministic)[3]
    mv_only = gpu_run(cpu, gc, gd, deterministic=deterministic, pj_grad=False)[3]
    pj_only = gpu_run(cpu, gc, gd, deterministic=deterministic, mv_grad=False)[3]
    assert mv_only["proj_mats"] is None and pj_only["mv_mats"] is None
    assert torch.equal(mv_only["mv_mats"], both["mv_mats"])
    assert torch.equal(pj_only["proj_mats"], both["proj_mats"])


def test_float64_matrices_get_float64_gradients():
    """TetRenderer casts the matrices to fp32 and transposes them; autograd carries the gradients back to the caller's
    float64 tensors."""
    cpu = scenes.config("tiny_tet")
    gc, gd = scenes.cotangents(cpu)
    ref = gpu_run(cpu, gc, gd, deterministic=True)[3]
    s = scenes.to_device(cpu, "cuda")
    mv = s.mv_mats.double().requires_grad_()
    pj = s.proj_mats.double().requires_grad_()
    color, depth, _ = TetRenderer(TetRenderSettings(s.H, s.W, s.bg, 0), deterministic=True)(
        s.verts, s.faces, s.verts_color, s.faces_opacity, mv, pj, s.verts_depth, s.faces_intense, s.tets, s.face_tets,
        s.tet_faces)
    torch.autograd.backward([color, depth], [gc.cuda(), gd.cuda()])
    assert mv.grad.dtype == torch.float64 and pj.grad.dtype == torch.float64
    assert torch.equal(mv.grad.float(), ref["mv_mats"]) and torch.equal(pj.grad.float(), ref["proj_mats"])


@pytest.mark.parametrize("case", ["small_tet", "short_trail", "jitter", "irregular"])
def test_other_gradients_with_and_without_camera(case):
    """Colour and opacity gradients with camera gradients on and off.  The camera instantiation of the backward kernel
    is compiled separately, and the compiler may round the per-step arithmetic it shares with the camera terms
    differently there (measured: faces_opacity differs in the last bits in deterministic mode, ~8e-8 relative L2), so
    colours are held bit-identical in deterministic mode and everything else to 1e-6 relative L2."""
    name, seed, cap = CASES[case]
    cpu = SCENES[name]()
    gc, gd = scenes.cotangents(cpu)
    with trail_cap(cap):
        on = gpu_run(cpu, gc, gd, seed=seed, deterministic=True)[3]
        off = gpu_run(cpu, gc, gd, seed=seed, deterministic=True, mv_grad=False, pj_grad=False)[3]
        on_d = gpu_run(cpu, gc, gd, seed=seed)[3]
        off_d = gpu_run(cpu, gc, gd, seed=seed, mv_grad=False, pj_grad=False)[3]
        torch.cuda.synchronize()
    assert off["mv_mats"] is None and off["proj_mats"] is None
    assert torch.equal(on["verts_color"], off["verts_color"])
    for k in ("verts_color", "faces_opacity"):
        assert rel_l2(on[k].cpu().numpy(), off[k].cpu().numpy()) <= 1e-6, k
        assert rel_l2(on_d[k].cpu().numpy(), off_d[k].cpu().numpy()) <= 1e-6, k


def _stages():
    lib = _lib.load()
    n = lib.dmr_profile_stage_count()
    ms = (ctypes.c_float * n)()
    _lib.check(lib.dmr_profile_read(ms))
    return {lib.dmr_profile_stage_name(i).decode() for i in range(n) if ms[i] >= 0}


CAMERA_STAGES = {"tet_march_backward_camera", "tet_camera_finish"}


@pytest.mark.parametrize("deterministic", [False, True], ids=["default", "det"])
def test_opt_in_no_camera_work_without_requires_grad(deterministic):
    cpu = grid4_scene()
    gc, gd = [t.cuda() for t in scenes.cotangents(cpu)]
    s = scenes.to_device(cpu, "cuda")
    lib = _lib.load()
    renderer = TetRenderer(TetRenderSettings(s.H, s.W, s.bg, 0), deterministic=deterministic)
    vc = s.verts_color.clone().requires_grad_()
    args = lambda mv, pj: (s.verts, s.faces, vc, s.faces_opacity, mv, pj, s.verts_depth, s.faces_intense, s.tets,
                           s.face_tets, s.tet_faces)
    renderer(*args(s.mv_mats, s.proj_mats))          # warm-up: record cache, speculative binning buffer
    torch.cuda.synchronize()
    _lib.check(lib.dmr_profile_enable(1))
    try:
        _stages()
        color, depth, _ = renderer(*args(s.mv_mats, s.proj_mats))
        n1 = lib.dmr_launch_count()
        torch.autograd.backward([color, depth], [gc, gd])
        n2 = lib.dmr_launch_count()
        torch.cuda.synchronize()
        st = _stages()
        assert not (st & CAMERA_STAGES) and "tet_march_backward" in st
        # the same backward through the _C shim, without camera_grads
        mv, pj = s.mv_mats.transpose(1, 2).contiguous(), s.proj_mats.transpose(1, 2).contiguous()
        imv, ipj = torch.inverse(mv), torch.inverse(pj)
        out = _C.render_tets(s.bg, s.verts, s.faces, s.verts_color, s.faces_opacity, mv, pj, imv, ipj, s.verts_depth,
                             s.faces_intense, s.tets, s.face_tets, s.tet_faces, s.H, s.W, 0)
        m0 = lib.dmr_launch_count()
        _C.render_tets_backward(s.bg, s.verts, s.faces, s.verts_color, s.faces_opacity, mv, pj, imv, ipj, s.verts_depth,
                                s.faces_intense, s.tets, s.face_tets, s.tet_faces, gc, gd, *out[3:], 0,
                                deterministic=deterministic)
        m1 = lib.dmr_launch_count()
        assert n2 - n1 == m1 - m0
        # with camera gradients the camera stages run, and the default march does not
        torch.cuda.synchronize()
        _stages()
        color, depth, _ = renderer(*args(s.mv_mats, s.proj_mats.clone().requires_grad_()))
        torch.autograd.backward([color, depth], [gc, gd])
        torch.cuda.synchronize()
        st = _stages()
        assert CAMERA_STAGES <= st and "tet_march_backward" not in st
    finally:
        lib.dmr_profile_enable(0)


def test_workspace_and_argument_checks():
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
    gv, go, gm = torch.zeros(P, 3, device="cuda"), torch.zeros(F, device="cuda"), torch.zeros(2, B, 16, device="cuda")
    tet_rec = out[4].tet_records
    need = lib.dmr_tet_backward_camera_bytes(B, P, F, s.W, s.H, 0)
    ws = torch.empty(need, dtype=torch.uint8, device="cuda")
    a = (B, P, F, T, s.W, s.H, 0, p(s.bg), p(mv), p(pj), p(imv), p(ipj), p(s.faces_intense), p(out[3]), p(out[4]),
         p(tet_rec), p(out[6]), p(gc), p(gd), p(gv), p(go), 0)
    stream = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    assert lib.dmr_tet_backward_camera(*a, p(gm[0]), None, p(ws), need, stream) == 1
    assert b"null" in lib.dmr_last_error()
    assert lib.dmr_tet_backward_camera(*a, p(gm[0]), p(gm[1]), p(ws), need - 1, stream) == 1
    assert b"dmr_tet_backward_camera_bytes" in lib.dmr_last_error()
    torch.cuda.synchronize()
    assert torch.count_nonzero(gv) == 0 and torch.count_nonzero(gm) == 0   # nothing was launched
    assert lib.dmr_tet_backward_camera(*a, p(gm[0]), p(gm[1]), p(ws), need, stream) == 0
    torch.cuda.synchronize()
    assert torch.count_nonzero(gm) > 0
