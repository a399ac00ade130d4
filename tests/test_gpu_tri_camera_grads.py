"""Tri renderer: gradients with respect to the camera matrices (mv_mats, proj_mats).

The yardstick is an fp64 re-implementation of the forward function as implemented, evaluated on exactly the
fragments the renderer composites (taken from the CPU oracle by tests/tri_fragments.cpp: per pixel, in compositing
order, the faces that pass in_tri and shade, up to n_contrib, with their clamp_bary region codes) and differentiated
by torch autograd.  The
discrete decisions -- coverage, depth order, n_contrib, the clamp region -- are held fixed, as in the renderer's own
gradients.  Before its camera gradients are trusted, the reference has to reproduce the GPU's images (IMG_TOL)
and its gradients for colours, opacities, intensities and vertex depths (1e-4 relative L2).  Vertex positions are not
compared: the renderer keeps the reference implementation's vertex-position formula (it differentiates t instead of
v for the second barycentric), the reference here uses the exact derivative.
"""
import numpy as np
import pytest
import torch

import tri_fragments
from dmesh_renderer_b200 import TriRenderer, TriRenderSettings, _C, _lib, multiview, scenes

# IMG_TOL: the reference evaluates the fp32 renderer's hits in fp64; near-degenerate (sliver) hits make the two differ
# by a few 1e-5 in colour on the small scenes here
IMG_TOL, GRAD_TOL, CAM_TOL = 1e-4, 1e-4, 1e-3
f64 = torch.float64


def rel_l2(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return float(np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-30))


def camera_scene():
    """Small scene with four views (non-multiple-of-16 image)."""
    return scenes.random_tri_scene("cam4", 21, 1500, 0.08, 72, 88, B=4)


SCENES = {"tiny_tri": lambda: scenes.config("tiny_tri"), "small_tri": lambda: scenes.config("small_tri"),
          "C1": lambda: scenes.config("C1"), "cam4": camera_scene}


# ---------------------------------------------------------------------------------------------- fp64 reference
def oracle_fragments(cpu):
    """Fragments of scene `cpu` (matrices as the renderer sees them: transposed, inverted with torch.inverse)."""
    mv, pj = cpu.mv_mats.transpose(1, 2).contiguous(), cpu.proj_mats.transpose(1, 2).contiguous()
    mats = [np.ascontiguousarray(m.numpy(), np.float32) for m in (mv, pj, torch.inverse(mv), torch.inverse(pj))]
    counts, face, code, ref = tri_fragments.tri_fragments(cpu, mats)
    return (counts, face, code), ref


def fused_ndc_depth(verts, mv, proj):
    """verts_depth=None: the vertex's NDC z as the renderer forms it (pv = MV[:3] (p, 1), clip = Proj (pv, 1),
    z / clamp_w(w), no derivative through a clamped w).  mv, proj: [B,4,4] maths convention."""
    pv = torch.einsum("bij,pj->bpi", mv[:, :3, :3], verts) + mv[:, None, :3, 3]
    z = torch.einsum("bj,bpj->bp", proj[:, 2, :3], pv) + proj[:, 2:3, 3]
    w = torch.einsum("bj,bpj->bp", proj[:, 3, :3], pv) + proj[:, 3:4, 3]
    eps = 1e-4
    wd = w.detach()
    wc = torch.where((wd >= 0) & (wd < eps), torch.full_like(w, eps), torch.where((wd < 0) & (wd > -eps),
                                                                                   torch.full_like(w, -eps), w))
    return z / wc


def reference_render(frags, faces, H, W, bg, verts, vcol, fopa, mv, proj, fint, vdepth):
    """fp64 colour [B,3,H,W] and depth [B,1,H,W] from the fragments; every float input may require grad.
    mv, proj: [B,4,4] maths convention; vdepth: [B,P]."""
    counts, face, code = frags
    B = counts.shape[0]
    cnt = torch.from_numpy(counts.reshape(-1).astype(np.int64))
    N = int(cnt.sum())
    pix = torch.repeat_interleave(torch.arange(B * H * W), cnt)
    starts = torch.cumsum(cnt, 0) - cnt
    rank = torch.arange(N) - starts[pix]
    b, y, x = pix // (H * W), (pix // W) % H, pix % W
    f = torch.from_numpy(face.astype(np.int64))
    code = torch.from_numpy(code.astype(np.int64))
    fv = faces.long()[f]                                                     # [N,3]
    # rays: pixel_ray<false> (common.cuh) -- NDC of the pixel centre rounded to fp32 like pix2ndc
    nx = torch.from_numpy(((((x.numpy() + 0.5) * 2.0 + 1.0) / W) - 1.0).astype(np.float32)).to(f64)
    ny = torch.from_numpy(((((y.numpy() + 0.5) * 2.0 + 1.0) / H) - 1.0).astype(np.float32)).to(f64)
    n = torch.stack([nx, ny, -torch.ones_like(nx), torch.ones_like(nx)], 1)
    # the values of the fp32 inverses the renderer uses, the derivative of the fp64 inverse
    inv_mv, inv_pj = [torch.linalg.inv(m) + (torch.inverse(m.detach().float()).double() - torch.linalg.inv(m.detach()))
                      for m in (mv, proj)]
    pv = torch.einsum("nij,nj->ni", inv_pj[b][:, :3, :], n)                 # pv.w is ignored
    d = torch.einsum("nij,nj->ni", inv_mv[b][:, :3, :3], pv)
    ro = inv_mv[b][:, :3, 3]
    rd = d / (d.norm(dim=1, keepdim=True) + 1e-7)
    p0, p1, p2 = verts[fv[:, 0]], verts[fv[:, 1]], verts[fv[:, 2]]
    T, E1, E2 = ro - p0, p1 - p0, p2 - p0
    Pv, Q = torch.linalg.cross(rd, E2), torch.linalg.cross(T, E1)
    D = (Pv * E1).sum(1)
    u, v = (Pv * T).sum(1) / D, (Q * rd).sum(1) / D
    # clamp_bary: the linear map of the exported region
    zero, one = torch.zeros_like(u), torch.ones_like(u)
    uc = torch.stack([u, zero, one, zero, zero, u, (1 + u - v) * 0.5], 1).gather(1, code[:, None])[:, 0]
    vc = torch.stack([v, zero, zero, one, v, zero, (1 - u + v) * 0.5], 1).gather(1, code[:, None])[:, 0]
    w = torch.stack([1 - uc - vc, uc, vc], 1)                                # [N,3]
    col = torch.einsum("nk,nkc->nc", w, vcol[fv]) * fint[b, f][:, None]
    dep = (w * vdepth[b[:, None], fv]).sum(1)
    alpha = fopa[f]
    # front-to-back compositing per pixel on a dense [pixels with fragments, max fragments] layout
    live, slot = torch.unique(pix, return_inverse=True)
    K = int(cnt.max()) if N else 1
    dense = lambda vals: torch.zeros(live.numel(), K, *vals.shape[1:], dtype=f64).index_put((slot, rank), vals)
    a = dense(alpha)
    Tc = torch.cumprod(1 - a, 1)
    Tx = torch.cat([torch.ones(live.numel(), 1, dtype=f64), Tc[:, :-1]], 1)
    wgt = a * Tx
    C = (dense(col) * wgt[..., None]).sum(1)                                 # [L,3]
    Dp = (dense(dep) * wgt).sum(1)
    Tf = Tc[:, -1]
    color = bg.to(f64)[None, :].expand(B * H * W, 3).index_put((live,), C + Tf[:, None] * bg.to(f64)[None, :])
    depth = torch.ones(B * H * W, dtype=f64).index_put((live,), Dp + Tf)
    return color.view(B, H, W, 3).permute(0, 3, 1, 2), depth.view(B, 1, H, W)


def reference_grads(cpu, frags, gc, gd, fused):
    """fp64 reference forward + backward.  Returns (color, depth, {name: grad})."""
    leaves = {k: getattr(cpu, k).to(f64).clone().requires_grad_() for k in
              ("verts", "verts_color", "faces_opacity", "mv_mats", "proj_mats", "faces_intense", "verts_depth")}
    L = leaves
    vdepth = fused_ndc_depth(L["verts"], L["mv_mats"], L["proj_mats"]) if fused else L["verts_depth"]
    color, depth = reference_render(frags, cpu.faces, cpu.H, cpu.W, cpu.bg, L["verts"], L["verts_color"],
                                    L["faces_opacity"], L["mv_mats"], L["proj_mats"], L["faces_intense"], vdepth)
    torch.autograd.backward([color, depth], [gc.to(f64), gd.to(f64)])
    grads = {k: (t.grad if t.grad is not None else torch.zeros_like(t)) for k, t in leaves.items()}
    return color.detach(), depth.detach(), grads


# ---------------------------------------------------------------------------------------------- GPU side
def gpu_run(cpu, gc, gd, fused=False, deterministic=False, camera=True, scale=1.0, verts_depth=None, mats=None):
    s = scenes.to_device(cpu, "cuda")
    mv = (mats[0] if mats is not None else s.mv_mats).detach().clone().requires_grad_(camera)
    pj = (mats[1] if mats is not None else s.proj_mats).detach().clone().requires_grad_(camera)
    leaves = [t.clone().requires_grad_() for t in (s.verts, s.verts_color, s.faces_opacity, s.faces_intense)]
    vd = None if fused else (verts_depth if verts_depth is not None else s.verts_depth.clone().requires_grad_())
    color, depth = TriRenderer(TriRenderSettings(s.H, s.W, s.bg), deterministic=deterministic)(
        leaves[0], s.faces, leaves[1], leaves[2], mv, pj, vd, leaves[3])
    torch.autograd.backward([color, depth], [gc.cuda() * scale, gd.cuda() * scale])
    g = dict(verts=leaves[0].grad, verts_color=leaves[1].grad, faces_opacity=leaves[2].grad,
             faces_intense=leaves[3].grad, mv_mats=mv.grad, proj_mats=pj.grad)
    if vd is not None and vd.is_leaf:
        g["verts_depth"] = vd.grad
    return color.detach(), depth.detach(), g


_refs = {}


def reference_for(name, fused):
    key = (name, fused)
    if key not in _refs:
        cpu = SCENES[name]()
        gc, gd = scenes.cotangents(cpu)
        frags, _ = oracle_fragments(cpu)
        _refs[key] = (cpu, gc, gd, reference_grads(cpu, frags, gc, gd, fused))
    return _refs[key]


@pytest.mark.gpu
@pytest.mark.parametrize("deterministic", [False, True], ids=["default", "det"])
@pytest.mark.parametrize("fused", [False, True], ids=["explicit_depth", "fused_depth"])
@pytest.mark.parametrize("name", list(SCENES))
def test_camera_grads_match_fp64_reference(name, fused, deterministic):
    cpu, gc, gd, (rc, rd, rg) = reference_for(name, fused)
    color, depth, g = gpu_run(cpu, gc, gd, fused=fused, deterministic=deterministic)
    # self-checks of the reference
    assert (color.cpu().double() - rc).abs().max().item() <= IMG_TOL
    assert (depth.cpu().double() - rd).abs().max().item() <= IMG_TOL
    checked = ["verts_color", "faces_opacity", "faces_intense"] + ([] if fused else ["verts_depth"])
    for k in checked:
        e = rel_l2(g[k].cpu().numpy(), rg[k].numpy())
        assert e <= GRAD_TOL, "%s rel L2 %.3e" % (k, e)
    # camera gradients, per view
    errs = []
    for k in ("mv_mats", "proj_mats"):
        for b in range(cpu.mv_mats.shape[0]):
            e = rel_l2(g[k][b].cpu().numpy(), rg[k][b].numpy())
            errs.append(e)
            assert e <= CAM_TOL, "%s view %d rel L2 %.3e" % (k, b, e)
    print("\n[camera grads] %s %s %s: max rel L2 mv %.2e proj %.2e" % (
        name, "fused" if fused else "explicit", "det" if deterministic else "default",
        max(errs[:len(errs) // 2]), max(errs[len(errs) // 2:])))


@pytest.mark.gpu
def test_dmesh_pattern_verts_depth_from_grad_matrices():
    """verts_depth built in torch from a grad-requiring mv (DMesh's own pattern): the summed autograd gradient of the
    matrices (through the rays and through verts_depth) equals the reference's."""
    cpu = SCENES["small_tri"]()
    gc, gd = scenes.cotangents(cpu)
    frags, _ = oracle_fragments(cpu)
    # reference: verts_depth = ndc_depth in fp64 from the same leaves
    L = {k: getattr(cpu, k).to(f64).clone().requires_grad_() for k in ("verts", "verts_color", "faces_opacity",
                                                                         "mv_mats", "proj_mats", "faces_intense")}
    vdepth = scenes.ndc_depth(L["verts"], L["mv_mats"], L["proj_mats"])
    color, depth = reference_render(frags, cpu.faces, cpu.H, cpu.W, cpu.bg, L["verts"], L["verts_color"],
                                    L["faces_opacity"], L["mv_mats"], L["proj_mats"], L["faces_intense"], vdepth)
    torch.autograd.backward([color, depth], [gc.to(f64), gd.to(f64)])
    # GPU: the same construction in fp32 on the CPU, the renderer on the GPU
    mv, pj = cpu.mv_mats.clone().requires_grad_(), cpu.proj_mats.clone().requires_grad_()
    vd = scenes.ndc_depth(cpu.verts, mv, pj).cuda()
    s = scenes.to_device(cpu, "cuda")
    c2, d2 = TriRenderer(TriRenderSettings(s.H, s.W, s.bg))(s.verts, s.faces, s.verts_color, s.faces_opacity,
                                                            mv.cuda(), pj.cuda(), vd, s.faces_intense)
    torch.autograd.backward([c2, d2], [gc.cuda(), gd.cuda()])
    for got, ref in ((mv.grad, L["mv_mats"].grad), (pj.grad, L["proj_mats"].grad)):
        for b in range(cpu.mv_mats.shape[0]):
            assert rel_l2(got[b].numpy(), ref[b].numpy()) <= CAM_TOL


def _split_views_equal(cpu, deterministic, fused=False):
    """Camera gradients of one B-view call against B single-view calls."""
    gc, gd = scenes.cotangents(cpu)
    _, _, g = gpu_run(cpu, gc, gd, fused=fused, deterministic=deterministic)
    B = cpu.mv_mats.shape[0]
    for b in range(B):
        sub = cpu._replace(mv_mats=cpu.mv_mats[b:b + 1], proj_mats=cpu.proj_mats[b:b + 1],
                           verts_depth=cpu.verts_depth[b:b + 1], faces_intense=cpu.faces_intense[b:b + 1])
        _, _, g1 = gpu_run(sub, gc[b:b + 1], gd[b:b + 1], fused=fused, deterministic=deterministic)
        for k in ("mv_mats", "proj_mats"):
            assert torch.isfinite(g[k][b]).all()
            if deterministic:
                assert torch.equal(g[k][b], g1[k][0]), (k, b)
            else:
                scale = max(g1[k][0].abs().max().item(), 1e-30)
                assert (g[k][b] - g1[k][0]).abs().max().item() <= 1e-5 * scale, (k, b)


@pytest.mark.gpu
@pytest.mark.parametrize("deterministic", [False, True], ids=["default", "det"])
def test_views_are_independent_small(deterministic):
    _split_views_equal(camera_scene(), deterministic)


@pytest.mark.gpu
@pytest.mark.parametrize("deterministic", [False, True], ids=["default", "det"])
def test_views_are_independent_c4_rank_share(deterministic):
    # one rank's share of C4 on 8 GPUs: 8 of its 64 views
    _split_views_equal(scenes.config("C4", views=64, view_slice=slice(0, 8)), deterministic)


@pytest.mark.gpu
@pytest.mark.parametrize("fused", [False, True], ids=["explicit_depth", "fused_depth"])
@pytest.mark.parametrize("deterministic", [False, True], ids=["default", "det"])
def test_reproducible_and_linear(deterministic, fused):
    cpu = camera_scene()
    gc, gd = scenes.cotangents(cpu)
    runs = [gpu_run(cpu, gc, gd, fused=fused, deterministic=deterministic)[2] for _ in range(4)]
    for r in runs[1:]:
        for k in ("mv_mats", "proj_mats"):
            if fused and not deterministic:
                # the fused depth's part is a function of dL_dvdepth, which the default backward accumulates with
                # float atomics (order-dependent low bits); the ray part has no atomics
                assert rel_l2(r[k].cpu().numpy(), runs[0][k].cpu().numpy()) <= 1e-6
            else:
                assert torch.equal(r[k], runs[0][k])
    zero = gpu_run(cpu, gc * 0, gd * 0, fused=fused, deterministic=deterministic)[2]
    for k in ("mv_mats", "proj_mats"):
        assert torch.count_nonzero(zero[k]) == 0
    if deterministic:
        for sc in (0.125, 32.0):
            g = gpu_run(cpu, gc, gd, fused=fused, deterministic=True, scale=sc)[2]
            for k in ("mv_mats", "proj_mats"):
                assert torch.equal(g[k], runs[0][k] * sc), (k, sc)


def _stages():
    lib = _lib.load()
    n = lib.dmr_profile_stage_count()
    import ctypes
    ms = (ctypes.c_float * n)()
    _lib.check(lib.dmr_profile_read(ms))
    return {lib.dmr_profile_stage_name(i).decode() for i in range(n) if ms[i] >= 0}


CAMERA_STAGES = {"tri_render_backward_camera", "tri_camera_finish", "depth_chain_camera", "depth_chain_camera_finish"}


@pytest.mark.gpu
@pytest.mark.parametrize("fused", [False, True], ids=["explicit_depth", "fused_depth"])
def test_opt_in_no_camera_work_without_requires_grad(fused):
    cpu = camera_scene()
    gc, gd = [t.cuda() for t in scenes.cotangents(cpu)]
    s = scenes.to_device(cpu, "cuda")
    lib = _lib.load()
    renderer = TriRenderer(TriRenderSettings(s.H, s.W, s.bg))
    verts = s.verts.clone().requires_grad_()
    vd = None if fused else s.verts_depth
    args = lambda mv, pj: (verts, s.faces, s.verts_color, s.faces_opacity, mv, pj, vd, s.faces_intense)
    renderer(*args(s.mv_mats, s.proj_mats))          # warm-up: same shapes for the speculative binning buffer
    torch.cuda.synchronize()
    _lib.check(lib.dmr_profile_enable(1))
    try:
        _stages()
        color, depth = renderer(*args(s.mv_mats, s.proj_mats))
        n1 = lib.dmr_launch_count()
        torch.autograd.backward([color, depth], [gc, gd])
        n2 = lib.dmr_launch_count()
        torch.cuda.synchronize()
        assert not (_stages() & CAMERA_STAGES)
        # the same backward through the _C shim, without camera_grads
        mv, pj = s.mv_mats.transpose(1, 2).contiguous(), s.proj_mats.transpose(1, 2).contiguous()
        imv, ipj = torch.inverse(mv), torch.inverse(pj)
        out = _C.render_tris(s.bg, s.verts, s.faces, s.verts_color, s.faces_opacity, mv, pj, imv, ipj, s.verts_depth,
                             s.faces_intense, s.H, s.W)
        m0 = lib.dmr_launch_count()
        g = _C.render_tris_backward(s.bg, s.verts, s.faces, s.verts_color, s.faces_opacity, mv, pj, imv, ipj,
                                    s.verts_depth, s.faces_intense, gc, gd, *out[:1], *out[3:])
        if fused:
            _C.tri_depth_chain(s.verts, mv, pj, g[3], g[0])
        m1 = lib.dmr_launch_count()
        assert n2 - n1 == m1 - m0
        # with camera gradients the camera stages do run
        torch.cuda.synchronize()
        _stages()
        color, depth = renderer(*args(s.mv_mats.clone().requires_grad_(), s.proj_mats))
        torch.autograd.backward([color, depth], [gc, gd])
        torch.cuda.synchronize()
        st = _stages()
        assert {"tri_render_backward_camera", "tri_camera_finish"} <= st
        assert ({"depth_chain_camera", "depth_chain_camera_finish"} <= st) == fused
    finally:
        lib.dmr_profile_enable(0)


@pytest.mark.gpu
@pytest.mark.parametrize("fused", [False, True], ids=["explicit_depth", "fused_depth"])
def test_other_gradients_unchanged_deterministic(fused):
    cpu = camera_scene()
    gc, gd = scenes.cotangents(cpu)
    _, _, on = gpu_run(cpu, gc, gd, fused=fused, deterministic=True, camera=True)
    _, _, off = gpu_run(cpu, gc, gd, fused=fused, deterministic=True, camera=False)
    assert off["mv_mats"] is None and off["proj_mats"] is None
    # Vertex positions and colours are bit-identical.  The camera instantiation of the backward kernel is compiled
    # separately, and the compiler may round the shared per-hit arithmetic of the other statistics differently there
    # (measured: faces_opacity differs in the last bits), so those are held to 1e-6 relative L2.
    for k in ("verts", "verts_color"):
        assert torch.equal(on[k], off[k]), k
    for k in off:
        if off[k] is not None:
            assert rel_l2(on[k].cpu().numpy(), off[k].cpu().numpy()) <= 1e-6, k


@pytest.mark.gpu
def test_packed_scene_grads_direct():
    """Under PackedSceneGrads.direct() (multiview_step) camera gradients go through autograd, equal those computed
    without the sink, and leave the packed buffer as it is without camera gradients."""
    cpu = camera_scene()
    s = scenes.to_device(cpu, "cuda")
    gct, gdt = [t.cuda() for t in scenes.cotangents(cpu)]
    renderer = TriRenderer(TriRenderSettings(s.H, s.W, s.bg), deterministic=True)
    cot = lambda color, depth: (gct, gdt)

    def step(camera, sink):
        verts, vcol, fopa = (t.clone().requires_grad_() for t in (s.verts, s.verts_color, s.faces_opacity))
        mv, pj = s.mv_mats.clone().requires_grad_(camera), s.proj_mats.clone().requires_grad_(camera)
        if sink:
            sg = multiview.PackedSceneGrads(verts, vcol, fopa)
            multiview.multiview_step(renderer, sg, s.faces, mv, pj, s.verts_depth, s.faces_intense, cot)
            flat = sg.flat.clone()
        else:
            color, depth = renderer(verts, s.faces, vcol, fopa, mv, pj, s.verts_depth, s.faces_intense)
            torch.autograd.backward([color, depth], [gct, gdt])
            flat = torch.cat([verts.grad.reshape(-1), vcol.grad.reshape(-1), fopa.grad.reshape(-1)])
        return flat, mv.grad, pj.grad

    f_cam, mv_cam, pj_cam = step(True, True)
    f_nocam, mv_none, _ = step(False, True)
    f_plain, mv_plain, pj_plain = step(True, False)
    assert mv_none is None
    assert mv_cam is not None and torch.equal(mv_cam, mv_plain) and torch.equal(pj_cam, pj_plain)
    assert torch.equal(f_cam, f_plain)
    # with and without camera gradients: see test_other_gradients_unchanged_deterministic
    assert rel_l2(f_cam.cpu().numpy(), f_nocam.cpu().numpy()) <= 1e-6


@pytest.mark.gpu
@pytest.mark.parametrize("fused", [False, True], ids=["explicit_depth", "fused_depth"])
def test_edge_scene(fused):
    from test_gpu_vs_oracle_and_golden import edge_scene
    _split_views_equal(edge_scene(), True, fused=fused)
    _split_views_equal(edge_scene(), False, fused=fused)
