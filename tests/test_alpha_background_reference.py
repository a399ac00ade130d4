"""CPU: the alpha image and the background gradient (return_alpha=True, bg.requires_grad) before any GPU run.

* The fp64 reference (the forward function as implemented, on the fragments the CPU oracle composites, as in
  tests/test_gpu_tri_camera_grads.py) extended by alpha = 1 - prod(1 - opacity) over a pixel's composited faces: its
  autograd derivatives with respect to the opacities and the background agree with central differences, and the
  opacity derivative of alpha is the background term the backward kernels use, T_final / (1 - opacity), i.e. the
  colour's background derivative with bg . dL_dC + dL_dD replaced by -dL_dalpha.
* The new C entry points validate their arguments before any CUDA call.
* PackedSceneGrads(..., bg=...) puts bg's gradient in the packed buffer, so the one all-reduce sums it over ranks.
"""
import ctypes
import os
import socket
import sys

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
f64 = torch.float64


def transmittance(cnt, opacity):
    """prod over each pixel's fragments of (1 - opacity): cnt [pixels] fragment counts, opacity [N] in pixel order.
    A dense product, so that an opacity of exactly 1 gets the derivative -prod(others), as in the renderers."""
    n = cnt.numel()
    N = int(cnt.sum())
    pix = torch.repeat_interleave(torch.arange(n), cnt)
    rank = torch.arange(N) - (torch.cumsum(cnt, 0) - cnt)[pix]
    K = max(int(cnt.max()) if N else 1, 1)
    return torch.ones(n, K, dtype=f64).index_put((pix, rank), 1 - opacity).prod(1)


def reference_alpha(frags, B, H, W, fopa):
    """fp64 alpha [B,1,H,W] = 1 - prod over the pixel's fragments of (1 - opacity); fopa [F] may require grad."""
    counts, face = frags[0], frags[1]
    cnt = torch.from_numpy(counts.reshape(-1).astype(np.int64))
    f = torch.from_numpy(face.astype(np.int64))
    return (1 - transmittance(cnt, fopa[f])).view(B, 1, H, W)


def tri_reference(name="tiny_tri", bg=None):
    from test_gpu_tri_camera_grads import SCENES, oracle_fragments
    cpu = SCENES[name]()
    if bg is not None:
        cpu = cpu._replace(bg=bg)
    frags, _ = oracle_fragments(cpu)
    return cpu, frags


def render64(cpu, frags, fopa, bg):
    from test_gpu_tri_camera_grads import reference_render
    B, H, W = cpu.mv_mats.shape[0], cpu.H, cpu.W
    color, depth = reference_render(frags, cpu.faces, H, W, bg, cpu.verts.to(f64), cpu.verts_color.to(f64), fopa,
                                    cpu.mv_mats.to(f64), cpu.proj_mats.to(f64), cpu.faces_intense.to(f64),
                                    cpu.verts_depth.to(f64))
    return color, depth, reference_alpha(frags, B, H, W, fopa)


def test_tri_reference_alpha_and_background_grads_match_central_differences():
    g = torch.Generator().manual_seed(3)
    bg0 = torch.rand(3, generator=g, dtype=f64)
    cpu, frags = tri_reference("tiny_tri", bg0.float())
    B, H, W = cpu.mv_mats.shape[0], cpu.H, cpu.W
    ga = torch.rand(B, 1, H, W, generator=g, dtype=f64) * 2 - 1
    gc = torch.rand(B, 3, H, W, generator=g, dtype=f64) * 2 - 1
    fopa = cpu.faces_opacity.to(f64).clone().requires_grad_()
    bg = bg0.clone().requires_grad_()
    color, depth, alpha = render64(cpu, frags, fopa, bg)
    loss = lambda c, a: (c * gc).sum() + (a * ga).sum()
    torch.autograd.backward([color, alpha], [gc, ga])
    # the background gradient is the plain reduction sum (1 - alpha) dL_dC
    want_bg = ((1 - alpha.detach()) * gc).sum((0, 2, 3))
    assert torch.allclose(bg.grad, want_bg, rtol=1e-12, atol=1e-12)
    # central differences: bg (linear: exact up to rounding) and a sample of opacities
    eps = 1e-6
    for c in range(3):
        d = torch.zeros(3, dtype=f64)
        d[c] = eps
        lp = loss(*render64(cpu, frags, fopa.detach(), bg0 + d)[0::2])
        lm = loss(*render64(cpu, frags, fopa.detach(), bg0 - d)[0::2])
        assert abs(float((lp - lm) / (2 * eps)) - float(bg.grad[c])) <= 1e-6 * max(1.0, abs(float(bg.grad[c])))
    hit = np.unique(frags[1])
    pick = hit[np.linspace(0, hit.size - 1, 12).astype(int)]
    for fi in pick:
        d = torch.zeros_like(fopa)
        d[fi] = eps
        lp = loss(*render64(cpu, frags, fopa.detach() + d, bg0)[0::2])
        lm = loss(*render64(cpu, frags, fopa.detach() - d, bg0)[0::2])
        cd = float((lp - lm) / (2 * eps))
        assert abs(cd - float(fopa.grad[fi])) <= 1e-6 * max(1.0, abs(cd)), fi


def test_alpha_opacity_derivative_is_the_background_term():
    """d alpha / d opacity_k = T_final / (1 - opacity_k) per composited face: the kernels' background term with the
    pixel constant bg . dL_dC + dL_dD replaced by -dL_dalpha."""
    cpu, frags = tri_reference("small_tri")
    B, H, W = cpu.mv_mats.shape[0], cpu.H, cpu.W
    counts, face = frags[0], frags[1]
    g = torch.Generator().manual_seed(4)
    ga = torch.rand(B, 1, H, W, generator=g, dtype=f64) * 2 - 1
    fopa = cpu.faces_opacity.to(f64).clone().requires_grad_()
    alpha = reference_alpha(frags, B, H, W, fopa)
    alpha.backward(ga)
    Tf = (1 - alpha.detach()).reshape(-1)
    cnt = torch.from_numpy(counts.reshape(-1).astype(np.int64))
    pix = torch.repeat_interleave(torch.arange(B * H * W), cnt)
    f = torch.from_numpy(face.astype(np.int64))
    op = cpu.faces_opacity.to(f64)[f]
    ok = op < 1
    term = -Tf[pix] / (1 - op) * (-ga.reshape(-1)[pix])
    want = torch.zeros_like(fopa).index_add(0, f[ok], term[ok])
    assert torch.allclose(fopa.grad, want, rtol=1e-10, atol=1e-12)


# ---------------------------------------------------------------------------------------------- argument checks
def test_new_entry_points_reject_bad_arguments():
    from dmesh_renderer_b200 import _lib
    lib = _lib.load()
    fake = ctypes.c_void_p(256)             # never dereferenced: every case fails before a kernel is enqueued
    null = ctypes.c_void_p(0)
    B, P, F, T, W, H, R = 2, 30, 10, 5, 32, 32, 100
    # alpha images: null buffers, bad sizes; an empty batch is a no-op
    for fn in (lib.dmr_tri_alpha, lib.dmr_tet_alpha):
        assert fn(B, W, H, null, fake, null) == 1 and b"null" in lib.dmr_last_error()
        assert fn(B, W, H, fake, null, null) == 1
        assert fn(-1, W, H, fake, fake, null) != 0 and b"size" in lib.dmr_last_error()
        assert fn(B, 0, H, fake, fake, null) != 0
        assert fn(0, W, H, null, null, null) == 0
    # background gradients: workspace query, null pointers, short workspace
    for nb, fn in ((lib.dmr_tri_background_grad_bytes, lib.dmr_tri_background_grad),
                   (lib.dmr_tet_background_grad_bytes, lib.dmr_tet_background_grad)):
        need = nb(B)
        assert need >= 3 * 4 * B and nb(-1) == 0
        assert fn(B, W, H, fake, fake, null, fake, need, null) == 1 and b"dL_dbg" in lib.dmr_last_error()
        assert fn(B, W, H, null, fake, fake, fake, need, null) == 1 and b"null" in lib.dmr_last_error()
        assert fn(B, W, H, fake, null, fake, fake, need, null) == 1
        assert fn(B, W, H, fake, fake, fake, fake, need - 1, null) == 1 and b"workspace" in lib.dmr_last_error()
        assert fn(B, W, H, fake, fake, fake, null, need, null) == 1
        assert fn(-1, W, H, fake, fake, fake, fake, need, null) != 0
    # tri backward with an alpha cotangent
    def tri(ptrs=None, det=0, exact=0, mv=fake, pj=fake, alpha=fake, ws=fake, nbytes=1 << 30, b=B, r=R):
        p = [fake] * 14 if ptrs is None else ptrs
        return lib.dmr_tri_backward_alpha(b, P, F, W, H, r, *p, det, exact, mv, pj, alpha, ws, nbytes, null)
    assert tri(mv=fake, pj=null) == 1 and b"dL_dmv" in lib.dmr_last_error()
    assert tri(alpha=null) == 1 and b"dL_dalpha" in lib.dmr_last_error()
    for i in (0, 1, 2, 4, 5, 6, 7, 8, 9, 10, 11, 12, 13):
        ptrs = [fake] * 14
        ptrs[i] = null
        assert tri(ptrs) == 1 and b"null" in lib.dmr_last_error(), i
    for det in (0, 1):
        for exact in (0, 1):
            for cam in (False, True):
                mv = fake if cam else null
                need = (lib.dmr_tri_backward_camera_bytes(B, P, F, W, H, det) if cam else
                        lib.dmr_tri_backward_deterministic_bytes(B, P, F) if det else
                        lib.dmr_tri_backward_workspace_bytes(B, P, F))
                assert tri(det=det, exact=exact, mv=mv, pj=mv, nbytes=need - 1) == 1, (det, exact, cam)
                assert b"workspace" in lib.dmr_last_error()
    assert tri(b=-1) != 0
    assert tri(ptrs=[null] * 14, r=0, mv=null, pj=null, ws=null, nbytes=0) == 0     # nothing composited: a no-op
    # tet backward with an alpha cotangent
    def tet(ptrs=None, det=0, mv=fake, pj=fake, dv=null, fi=null, alpha=fake, ws=fake, nbytes=1 << 30, b=B, t=T):
        p = [fake] * 14 if ptrs is None else ptrs
        return lib.dmr_tet_backward_alpha(b, P, F, t, W, H, 0, *p, det, mv, pj, dv, fi, alpha, ws, nbytes, null)
    assert tet(mv=null, pj=fake) == 1 and b"dL_dmv" in lib.dmr_last_error()
    assert tet(alpha=null) == 1 and b"dL_dalpha" in lib.dmr_last_error()
    for i in (0, 1, 2, 3, 4, 5, 7, 8, 9, 10, 11, 12, 13):
        ptrs = [fake] * 14
        ptrs[i] = null
        assert tet(ptrs) == 1 and b"null" in lib.dmr_last_error(), i
    for det in (0, 1):
        for cam in (0, 1):
            for vert in (0, 1):
                for fint in (0, 1):
                    mv = fake if cam else null
                    need = (lib.dmr_tet_backward_intensity_bytes(B, P, F, W, H, det, cam, vert) if fint else
                            lib.dmr_tet_backward_vertex_bytes(B, P, F, W, H, det, cam) if vert else
                            lib.dmr_tet_backward_camera_bytes(B, P, F, W, H, det) if cam else
                            lib.dmr_tet_backward_deterministic_bytes(P, F) if det else
                            lib.dmr_tet_backward_workspace_bytes(P) - 256)
                    rc = tet(det=det, mv=mv, pj=mv, dv=fake if vert else null, fi=fake if fint else null, nbytes=need - 1)
                    assert rc == 1 and b"workspace" in lib.dmr_last_error(), (det, cam, vert, fint)
    assert tet(b=-1) != 0
    assert tet(ptrs=[null] * 14, t=0, mv=null, pj=null, ws=null, nbytes=0) == 0      # no tets: a no-op


# ---------------------------------------------------------------------------------------------- gloo: the bg slot
B_ALL, H, W, P, F = 4, 6, 5, 7, 9


def _inputs():
    g = torch.Generator().manual_seed(11)
    return dict(verts=torch.rand(P, 3, generator=g), vcol=torch.rand(P, 3, generator=g), fopa=torch.rand(F, generator=g),
                bg=torch.rand(3, generator=g), mv=torch.rand(B_ALL, 4, 4, generator=g),
                w=torch.rand(B_ALL, 1, H, W, generator=g))


class _StandIn:
    """A TriRenderer-shaped CPU stand-in with an alpha image: alpha = sigmoid(w_b) * mean(opacity),
    colour = mean(colour) * alpha + (1 - alpha) * bg (bg read from the settings, as the renderers do)."""

    def __init__(self, bg, w_all):
        self.bg, self.w_all = bg, w_all

    def __call__(self, verts, faces, verts_color, faces_opacity, mv, proj, verts_depth, faces_intense):
        idx = mv[:, 0, 0].long()                        # the view index rides in the matrix
        alpha = torch.sigmoid(self.w_all[idx]) * faces_opacity.mean()
        color = verts_color.mean(0)[None, :, None, None] * alpha + (1 - alpha) * self.bg[None, :, None, None]
        depth = alpha * verts.sum()
        return color, depth, alpha


def _cot(color, depth, alpha):
    return color.detach() - 0.5, torch.ones_like(depth), alpha.detach() * 2 - 0.3


def _step(sl):
    from dmesh_renderer_b200.multiview import PackedSceneGrads, multiview_step
    d = _inputs()
    verts, vcol, fopa, bg = (d[k].clone() for k in ("verts", "vcol", "fopa", "bg"))
    g = PackedSceneGrads(verts, vcol, fopa, bg=bg)
    mv = torch.zeros(B_ALL, 4, 4)
    mv[:, 0, 0] = torch.arange(B_ALL).float()
    n = B_ALL
    multiview_step(_StandIn(bg, d["w"]), g, torch.zeros(F, 3, dtype=torch.int32), mv[sl], mv[sl], torch.zeros(n, P)[sl],
                   torch.zeros(n, F)[sl], _cot, views_per_call=1)
    return g, bg


def _run_rank(rank, ws, port, out):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=ws)
    try:
        from dmesh_renderer_b200.multiview import shard_views
        mine = shard_views(B_ALL, rank, ws)
        g, bg = _step(slice(mine.start, mine.stop))
        assert bg.grad.data_ptr() == g.flat[-3:].data_ptr()
        torch.save(g.flat.clone(), os.path.join(out, "rank%d.pt" % rank))
    finally:
        dist.destroy_process_group()


def test_packed_scene_grads_bg_slot_layout():
    from dmesh_renderer_b200.multiview import PackedSceneGrads
    d = _inputs()
    with pytest.raises(ValueError, match="bg"):
        PackedSceneGrads(d["verts"].clone(), d["vcol"].clone(), d["fopa"].clone(), bg=d["bg"].double())
    g, bg = _step(slice(0, B_ALL))
    assert g.flat.numel() == 6 * P + F + 3 and len(g.leaves) == 3
    assert bg.grad.data_ptr() == g.flat[6 * P + F:].data_ptr()
    # autograd accumulated straight into the slot: the value is the stand-in's own derivative
    dd = _inputs()
    bg2 = dd["bg"].clone().requires_grad_()
    r = _StandIn(bg2, dd["w"])
    mv = torch.zeros(B_ALL, 4, 4)
    mv[:, 0, 0] = torch.arange(B_ALL).float()
    out = r(dd["verts"], None, dd["vcol"], dd["fopa"], mv, mv, None, None)
    torch.autograd.backward([out[0]], [_cot(*out)[0]])          # only the colour depends on bg
    assert torch.allclose(bg.grad, bg2.grad, rtol=1e-6, atol=1e-7)
    g.zero_()
    assert bg.grad.abs().sum() == 0 and bg.grad.data_ptr() == g.flat[6 * P + F:].data_ptr()
    bg.grad = None                                   # zero_grad(set_to_none=True) is repaired by bind()
    assert g.bind() == 1 and bg.grad.data_ptr() == g.flat[6 * P + F:].data_ptr()


@pytest.mark.timeout(300)
def test_bg_slot_is_all_reduced(tmp_path):
    with socket.socket() as sk:
        sk.bind(("127.0.0.1", 0))
        port = sk.getsockname()[1]
    mp.spawn(_run_rank, args=(2, port, str(tmp_path)), nprocs=2, join=True)
    r0, r1 = torch.load(tmp_path / "rank0.pt"), torch.load(tmp_path / "rank1.pt")
    assert torch.equal(r0, r1)
    g, _ = _step(slice(0, B_ALL))
    assert torch.allclose(r0, g.flat, rtol=1e-5, atol=1e-6)
    assert r0[-3:].abs().sum() > 0
