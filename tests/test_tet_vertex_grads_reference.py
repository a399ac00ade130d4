"""CPU: the tet renderer's vertex-position gradients (vertex_grads=True), checked without a GPU.

Per walked step, with T = ro - p0, E1 = p1 - p0, E2 = p2 - p0, N = E2 x E1, D = rd.N and the step's dL/du, dL/dv, dL/dt
(k_u = dL/du / D, k_v, k_t likewise, k_n = k_u u + k_v v + k_t t):
    g_T  = k_u (rd x E2) + k_v (E1 x rd) - k_t N
    g_E1 = k_v (rd x T)  + k_t (E2 x T)  - k_n (rd x E2)
    g_E2 = k_u (T x rd)  + k_t (T x E1)  - k_n (E1 x rd)
    dL/dp0 = -g_T - g_E1 - g_E2,   dL/dp1 = g_E1,   dL/dp2 = g_E2
(tet_vert_step, csrc/tet_kernels.cu).  The closed form is checked against fp64 autograd of Moeller-Trumbore; the fp64
reference of the camera-gradient tests is extended with a `verts` leaf (every input of a step the backward pass does
not walk detached, the triangle included) and checked against the oracle and the rigid-motion identity.
"""
import ctypes

import numpy as np
import pytest
import torch

from dmesh_renderer_b200 import scenes
from test_gpu_tet_camera_grads import GRAD_TOL, IMG_TOL, SCENES, _clamp_w, _pix2ndc, oracle_fragments, rel_l2

f64 = torch.float64
cr = torch.linalg.cross


def closed_form(ro, rd, p0, p1, p2, gu, gv, gt):
    """dL/d(p0, p1, p2) and dL/dro of one step per row, from the step's dL/du, dL/dv, dL/dt."""
    T, E1, E2 = ro - p0, p1 - p0, p2 - p0
    N = cr(E2, E1)
    D = (rd * N).sum(-1, keepdim=True)
    Q = cr(T, E1)
    t, u, v = (Q * E2).sum(-1, keepdim=True) / D, (cr(rd, E2) * T).sum(-1, keepdim=True) / D, (Q * rd).sum(-1, keepdim=True) / D
    ku, kv, kt = gu / D, gv / D, gt / D
    kn = ku * u + kv * v + kt * t
    gT = ku * cr(rd, E2) + kv * cr(E1, rd) - kt * N
    gE1 = kv * cr(rd, T) + kt * cr(E2, T) - kn * cr(rd, E2)
    gE2 = ku * cr(T, rd) + kt * cr(T, E1) - kn * cr(E1, rd)
    return -gT - gE1 - gE2, gE1, gE2, gT


def test_closed_form_matches_autograd_of_moeller_trumbore():
    g = torch.Generator().manual_seed(3)
    n = 4000
    rn = lambda *s: torch.randn(*s, generator=g, dtype=f64)
    p0, p1, p2 = rn(n, 3), rn(n, 3), rn(n, 3)
    N = cr(p2 - p0, p1 - p0)
    # ray directions from nearly perpendicular to the normal (|rd.n| = 1e-3 |n| for the last quarter) to along it
    d = rn(n, 3)
    d = d / d.norm(dim=1, keepdim=True)
    nh = N / N.norm(dim=1, keepdim=True)
    tang = d - (d * nh).sum(1, keepdim=True) * nh
    tang = tang / tang.norm(dim=1, keepdim=True)
    c = torch.rand(n, 1, generator=g, dtype=f64)
    c[3 * n // 4:] = 1e-3
    rd = c * nh + (1 - c * c).sqrt() * tang
    ro = (p0 + p1 + p2) / 3 + 0.3 * rn(n, 3) - 2.0 * rd
    leaves = [x.clone().requires_grad_() for x in (ro, rd, p0, p1, p2)]
    r, dd, q0, q1, q2 = leaves
    T, E1, E2 = r - q0, q1 - q0, q2 - q0
    P, Q = cr(dd, E2), cr(T, E1)
    D = (P * E1).sum(1)
    t, u, v = (Q * E2).sum(1) / D, (P * T).sum(1) / D, (Q * dd).sum(1) / D
    gu, gv, gt = rn(n), rn(n), rn(n)
    (gu * u + gv * v + gt * t).sum().backward()
    cos = (rd * N).sum(1).abs() / N.norm(dim=1)
    assert float(cos.min()) <= 1.01e-3
    out = closed_form(ro, rd, p0, p1, p2, gu[:, None], gv[:, None], gt[:, None])
    for got, leaf in zip(out, (leaves[2], leaves[3], leaves[4], leaves[0])):
        e = (got - leaf.grad).norm(dim=1) / leaf.grad.norm(dim=1).clamp_min(1e-300)
        assert float(e.max()) <= 1e-10, float(e.max())


# ---------------------------------------------------------------------------------------------- fp64 reference
def reference_render_verts(frags, cpu, verts, vcol, fopa, mv, proj, fint, fp64_inverse=False):
    """reference_render of tests/test_gpu_tet_camera_grads.py with the vertex positions `verts` [P,3] as an input (it
    may require grad).  Every input of a step the backward pass does not walk is detached, the triangle included.
    `fp64_inverse`: take the values of the camera inverses from the fp64 inverse (by default they are those of the
    fp32 torch.inverse the renderer uses, with the derivative of the fp64 one), so that values and derivative belong to
    the same function -- the rigid-motion identity holds to rounding only then."""
    B, H, W = cpu.mv_mats.shape[0], cpu.H, cpu.W
    HW, BI = H * W, B * H * W
    active = torch.from_numpy(frags["active"])
    cnt_all = torch.from_numpy(frags["counts"].astype(np.int64))
    keep = torch.repeat_interleave(active, cnt_all)
    cnt = cnt_all * active
    N = int(cnt.sum())
    pix = torch.repeat_interleave(torch.arange(BI), cnt)
    starts = torch.cumsum(cnt, 0) - cnt
    rank = torch.arange(N) - starts[pix]
    f = torch.from_numpy(frags["face"].astype(np.int64))[keep]
    r = torch.from_numpy(frags["reach"])[keep]
    b = pix // HW
    sel = lambda x: torch.where(r.view(-1, *([1] * (x.dim() - 1))), x, x.detach())
    xy = frags["coords"][pix.numpy()]
    n = torch.stack([_pix2ndc(xy[:, 0], W), _pix2ndc(xy[:, 1], H), -torch.ones(N, dtype=f64), torch.ones(N, dtype=f64)], 1)
    if fp64_inverse:
        inv_mv, inv_pj = torch.linalg.inv(mv), torch.linalg.inv(proj)
    else:
        inv_mv, inv_pj = [torch.linalg.inv(m) + (torch.inverse(m.detach().float()).double() - torch.linalg.inv(m.detach()))
                          for m in (mv, proj)]
    pv = torch.einsum("nij,nj->ni", inv_pj[b][:, :3, :], n)
    d = torch.einsum("nij,nj->ni", inv_mv[b][:, :3, :3], pv)
    ro = sel(inv_mv[b][:, :3, 3])
    rd = sel(d / d.norm(dim=1, keepdim=True).clamp_min(1e-4))
    fv = cpu.faces.long()[f]
    p0, p1, p2 = sel(verts[fv[:, 0]]), sel(verts[fv[:, 1]]), sel(verts[fv[:, 2]])
    T, E1, E2 = ro - p0, p1 - p0, p2 - p0
    Pv, Q = cr(rd, E2), cr(T, E1)
    D = (Pv * E1).sum(1)
    t, u, v = (Q * E2).sum(1) / D, (Pv * T).sum(1) / D, (Q * rd).sum(1) / D
    c = sel(vcol[fv])
    col = (c[:, 0] + (c[:, 1] - c[:, 0]) * u[:, None] + (c[:, 2] - c[:, 0]) * v[:, None]) * sel(fint[b, f])[:, None]
    mvf, pjf = sel(mv[b]), sel(proj[b])
    pt = ro + t[:, None] * rd
    pm = torch.einsum("nij,nj->ni", mvf[:, :3, :3], pt) + mvf[:, :3, 3]
    z = (pjf[:, 2, :3] * pm).sum(1) + pjf[:, 2, 3]
    w = (pjf[:, 3, :3] * pm).sum(1) + pjf[:, 3, 3]
    pd = z / _clamp_w(w)
    alpha = sel(fopa[f])
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
    # grazing faces (|rd.n| < 1e-2 |n| at some walked step): fp32 (t, u, v) are ill-conditioned there
    cos = (rd.detach() * cr(E2, E1).detach()).sum(1).abs() / cr(E2, E1).detach().norm(dim=1)
    grazing = torch.unique(f[r & (cos < 1e-2)])
    return color.view(B, H, W, 3).permute(0, 3, 1, 2), depth.view(B, 1, H, W), grazing


def reference_grads_verts(cpu, frags, gc, gd, fp64_inverse=False):
    """fp64 reference forward + backward with a verts leaf.  Returns (color, depth, {name: grad}, grazing face ids)."""
    L = {k: getattr(cpu, k).to(f64).clone().requires_grad_() for k in
         ("verts", "verts_color", "faces_opacity", "mv_mats", "proj_mats", "faces_intense")}
    color, depth, grazing = reference_render_verts(frags, cpu, L["verts"], L["verts_color"], L["faces_opacity"],
                                                   L["mv_mats"], L["proj_mats"], L["faces_intense"], fp64_inverse)
    torch.autograd.backward([color, depth], [gc.to(f64), gd.to(f64)])
    grads = {k: (t.grad if t.grad is not None else torch.zeros_like(t)) for k, t in L.items()}
    return color.detach(), depth.detach(), grads, grazing


def rigid_residual(verts, mv, g_verts, g_mv, seed=5):
    """Directional derivative of the loss along a rigid motion of scene and camera together: the vertices move by
    w x p + tau and mv (maths convention, world -> camera) by -mv G, G = [[w]x, tau; 0, 0].  Returns
    (|sum of terms|, sum of |terms|, sum of |vertex terms|)."""
    g = torch.Generator().manual_seed(seed)
    w = (torch.rand(3, generator=g, dtype=f64) - 0.5) * 0.2
    tau = (torch.rand(3, generator=g, dtype=f64) - 0.5) * 0.2
    G = torch.zeros(4, 4, dtype=f64)
    G[:3, :3] = torch.tensor([[0, -w[2], w[1]], [w[2], 0, -w[0]], [-w[1], w[0], 0]], dtype=f64)
    G[:3, 3] = tau
    verts, mv = verts.to(f64), mv.to(f64)
    dp = cr(w.expand_as(verts), verts) + tau
    tv = (g_verts.to(f64) * dp).reshape(-1)
    terms = torch.cat([tv, (g_mv.to(f64) * (-mv @ G)).reshape(-1)])
    return float(terms.sum().abs()), float(terms.abs().sum()), float(tv.abs().sum())


NAMES = ["tiny_tet", "small_tet", "irregular"]


@pytest.mark.parametrize("name", NAMES)
def test_reference_reproduces_oracle_and_the_rigid_motion_identity(name):
    cpu = SCENES[name]()
    gc, gd = scenes.cotangents(cpu)
    frags, out = oracle_fragments(cpu, gradients=(gc, gd))
    color, depth, g, _ = reference_grads_verts(cpu, frags, gc, gd)
    act = torch.from_numpy(out["oracle_active"] > 0.5)[:, None]
    assert (color - torch.from_numpy(out["oracle_color"]).double()).abs().masked_select(act).max().item() <= IMG_TOL
    assert (depth - torch.from_numpy(out["oracle_depth"]).double()).abs().masked_select(act).max().item() <= IMG_TOL
    ovc, ofo = out["oracle_grads"]
    assert rel_l2(g["verts_color"].numpy(), ovc) <= GRAD_TOL
    assert rel_l2(g["faces_opacity"].numpy(), ofo) <= GRAD_TOL
    assert torch.isfinite(g["verts"]).all() and g["verts"].abs().max() > 0
    # vertex + camera gradients of the same function: a rigid motion of scene and camera together changes nothing
    _, _, g64, _ = reference_grads_verts(cpu, frags, gc, gd, fp64_inverse=True)
    r, s, sv = rigid_residual(cpu.verts, cpu.mv_mats, g64["verts"], g64["mv_mats"])
    print("\n[tet rigid motion, fp64] %s: residual %.2e of %.2e" % (name, r, s))
    assert sv > 0.01 * s and r <= 1e-10 * s


def test_backward_vertex_rejects_bad_arguments():
    """dmr_tet_backward_vertex validates its arguments before any CUDA call (no GPU needed)."""
    from dmesh_renderer_b200 import _lib
    lib = _lib.load()
    fake = ctypes.c_void_p(256)             # never dereferenced: every case fails before a kernel is enqueued
    null = ctypes.c_void_p(0)
    B, P, F, T, W, H = 2, 30, 40, 10, 32, 32

    def call(ptrs=None, det=0, mv=fake, pj=fake, dv=fake, ws=fake, nbytes=1 << 30):
        p = [fake] * 14 if ptrs is None else ptrs
        return lib.dmr_tet_backward_vertex(B, P, F, T, W, H, 0, *p, det, mv, pj, dv, ws, nbytes, null)

    assert call(mv=fake, pj=null) == 1 and b"dL_dmv" in lib.dmr_last_error()
    assert call(mv=null, pj=fake) == 1
    assert call(dv=null) == 1 and b"dL_dverts" in lib.dmr_last_error()
    for i in (0, 1, 2, 3, 4, 5, 7, 8, 9, 10, 11, 12, 13):   # every pointer the backward reads or writes
        ptrs = [fake] * 14
        ptrs[i] = null
        assert call(ptrs) == 1 and b"null" in lib.dmr_last_error(), i
    for det in (0, 1):
        for cam in (0, 1):
            mv = fake if cam else null
            need = lib.dmr_tet_backward_vertex_bytes(B, P, F, W, H, det, cam)
            base = (lib.dmr_tet_backward_camera_bytes(B, P, F, W, H, det) if cam else
                    lib.dmr_tet_backward_deterministic_bytes(P, F) if det else lib.dmr_tet_backward_workspace_bytes(P))
            assert need >= base + (8 if det else 4) * 4 * P, (det, cam)   # one more per-vertex accumulator
            assert call(det=det, mv=mv, pj=mv, nbytes=need - 1) == 1, (det, cam)
            assert b"dmr_tet_backward_vertex_bytes" in lib.dmr_last_error()
            assert call(det=det, mv=mv, pj=mv, ws=null, nbytes=need) == 1, (det, cam)
    assert lib.dmr_tet_backward_vertex_bytes(-1, P, F, W, H, 0, 0) == 0
    # sizes are checked first, and an empty call is a no-op
    assert lib.dmr_tet_backward_vertex(-1, P, F, T, W, H, 0, *([fake] * 14), 0, null, null, fake, fake, 0, null) != 0
    assert lib.dmr_tet_backward_vertex(0, P, F, T, W, H, 0, *([null] * 14), 0, null, null, null, null, 0, null) == 0
