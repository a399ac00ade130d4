"""CPU: the algebra of the tri renderer's exact vertex-position gradients (exact_vertex_grads=True), checked on the
fp64 reference of the camera-gradient tests (tests/test_gpu_tri_camera_grads.py) before any GPU run.

Per covered hit, with T = ro - p0, E1 = p1 - p0, E2 = p2 - p0, D = rd.(E2 x E1), u = rd.(E2 x T) / D,
v = rd.(T x E1) / D, t = (T x E1).E2 / D and k_u = dL_du / D, k_v = dL_dv / D, the gradient of one (view, face) needs
three vector sums over its hits:
    S1 = sum k_u rd,   S24 = sum (k_u u + k_v v) rd,   S3v = sum k_v rd
    g_E1 = S3v x T - S24 x E2,   g_E2 = T x S1 - E1 x S24,   g_T = S1 x E2 + E1 x S3v
    dL/dp0 = -g_E1 - g_E2 - g_T,   dL/dp1 = g_E1,   dL/dp2 = g_E2
The reference implementation's formula (the renderer's default) uses k_v t in S24 and the scalar S3 = sum k_v.

The per-hit values (rays, edges, u, v and dL/du, dL/dv after the clamp chain) are taken from the fp64 reference itself
while it runs: a TorchFunctionMode records the operands of its two cross products (rd x E2, T x E1) and the unclamped
u and v it stacks for the clamp.
"""
import ctypes
import os
import sys

import numpy as np
import pytest
import torch
from torch.overrides import TorchFunctionMode

from test_gpu_tri_camera_grads import SCENES, oracle_fragments, reference_grads

f64 = torch.float64
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def rel_l2(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return float(np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-30))


class _HitCapture(TorchFunctionMode):
    """Records the per-hit tensors of reference_render: the operands of torch.linalg.cross (first call rd, E2; second
    T, E1) and the unclamped u, v (element 0 of the two seven-way torch.stack calls of the clamp), with retain_grad.
    `fp64_inverse`: the reference takes the VALUES of the camera inverses from the fp32 torch.inverse the renderer uses
    (and the derivative from the fp64 inverse); with this flag that fp32 inverse is computed in fp64, so that values and
    derivative belong to the same function (the rigid-motion identity holds to rounding only then: the fp32 values put
    the rays ~1e-7 off, which leaves a residual of ~3e-6 of the terms)."""

    def __init__(self, fp64_inverse=False):
        super().__init__()
        self.cross, self.bary = [], []
        self.fp64_inverse = fp64_inverse

    def __torch_function__(self, func, types, args=(), kwargs=None):
        kwargs = kwargs or {}
        if func is torch.inverse and self.fp64_inverse:
            return torch.linalg.inv(args[0].double())
        if func is torch.linalg.cross:
            self.cross.append(tuple(a.detach() for a in args[:2]))
        elif func is torch.stack and isinstance(args[0], (list, tuple)) and len(args[0]) == 7 and args[0][0].requires_grad:
            args[0][0].retain_grad()
            self.bary.append(args[0][0])
        return func(*args, **kwargs)


def reference_hits(cpu, frags, gc, gd, fused, fp64_inverse=False):
    """fp64 reference forward + backward with its per-hit values.  Returns (grads, hits): grads as reference_grads,
    hits = dict(b, f [N] view and face of each hit, rd, T, E1, E2 [N,3], u, v, gu, gv [N])."""
    cap = _HitCapture(fp64_inverse)
    with cap:
        _, _, grads = reference_grads(cpu, frags, gc, gd, fused)
    assert len(cap.cross) == 2 and len(cap.bary) == 2, (len(cap.cross), len(cap.bary))
    (rd, E2), (T, E1) = cap.cross
    u, v = cap.bary
    counts, face, _ = frags
    B, H, W = counts.shape
    pix = torch.repeat_interleave(torch.arange(B * H * W), torch.from_numpy(counts.reshape(-1).astype(np.int64)))
    hits = dict(b=pix // (H * W), f=torch.from_numpy(face.astype(np.int64)), rd=rd, T=T, E1=E1, E2=E2,
                u=u.detach(), v=v.detach(), gu=u.grad, gv=v.grad)
    return grads, hits


def closed_form_vertex_grads(hits, faces, P, exact):
    """dL/dverts [P,3] from the per-(view, face) statistics (module docstring); exact=False: the reference's formula."""
    rd, T, E1, E2 = hits["rd"], hits["T"], hits["E1"], hits["E2"]
    D = (rd * torch.linalg.cross(E2, E1)).sum(1)
    ku, kv = hits["gu"] / D, hits["gv"] / D
    second = hits["v"] if exact else (torch.linalg.cross(T, E1) * E2).sum(1) / D     # v, or the reference's t
    F = faces.shape[0]
    key = hits["b"] * F + hits["f"]
    uniq, inv = torch.unique(key, return_inverse=True)
    n = uniq.numel()
    S1 = torch.zeros(n, 3, dtype=f64).index_add_(0, inv, ku[:, None] * rd)
    S24 = torch.zeros(n, 3, dtype=f64).index_add_(0, inv, (ku * hits["u"] + kv * second)[:, None] * rd)
    # T, E1, E2 are constant within a (view, face): take them from any of its hits
    first = torch.zeros(n, dtype=torch.long).index_put_((inv,), torch.arange(inv.numel()))
    Tk, E1k, E2k = T[first], E1[first], E2[first]
    cr = torch.linalg.cross
    if exact:
        S3v = torch.zeros(n, 3, dtype=f64).index_add_(0, inv, kv[:, None] * rd)
        gE1 = cr(S3v, Tk) - cr(S24, E2k)
        gE2 = cr(Tk, S1) - cr(E1k, S24)
        gT = cr(S1, E2k) + cr(E1k, S3v)
    else:
        S3 = torch.zeros(n, dtype=f64).index_add_(0, inv, kv)[:, None]
        gE1 = S3 * cr(E2k, Tk) - cr(S24, E2k)
        gE2 = cr(Tk, S1) - cr(E1k, S24) + S3 * cr(Tk, E1k)
        gT = cr(S1, E2k) + S3 * cr(E1k, E2k)
    fv = faces.long()[uniq % F]
    out = torch.zeros(P, 3, dtype=f64)
    for k, g in enumerate((-gE1 - gE2 - gT, gE1, gE2)):
        out.index_add_(0, fv[:, k], g)
    return out


def rigid_motion(seed=5):
    """A small rotation w and translation tau, and G = [[w]x, tau; 0, 0] (the motion x -> x + w x x + tau)."""
    g = torch.Generator().manual_seed(seed)
    w = (torch.rand(3, generator=g, dtype=f64) - 0.5) * 0.2
    tau = (torch.rand(3, generator=g, dtype=f64) - 0.5) * 0.2
    G = torch.zeros(4, 4, dtype=f64)
    G[:3, :3] = torch.tensor([[0, -w[2], w[1]], [w[2], 0, -w[0]], [-w[1], w[0], 0]], dtype=f64)
    G[:3, 3] = tau
    return w, tau, G


def rigid_residual(verts, mv, g_verts, g_mv, seed=5):
    """Directional derivative of the loss along a rigid motion of scene and camera together: the vertices move by
    w x p + tau and mv (maths convention, world -> camera) by -mv G (mv M^-1 to first order).  Returns
    (|sum of terms|, sum of |terms|); the first is zero for consistent gradients."""
    w, tau, G = rigid_motion(seed)
    verts, mv = verts.to(f64), mv.to(f64)
    dp = torch.linalg.cross(w.expand_as(verts), verts) + tau
    dmv = -mv @ G
    terms = torch.cat([(g_verts.to(f64) * dp).reshape(-1), (g_mv.to(f64) * dmv).reshape(-1)])
    return float(terms.sum().abs()), float(terms.abs().sum())


_cache = {}


def hits_for(name, fused=False, fp64_inverse=False):
    key = (name, fused, fp64_inverse)
    if key not in _cache:
        cpu = SCENES[name]()
        from dmesh_renderer_b200 import scenes
        gc, gd = scenes.cotangents(cpu)
        frags, _ = oracle_fragments(cpu)
        grads, hits = reference_hits(cpu, frags, gc, gd, fused, fp64_inverse)
        _cache[key] = (cpu, gc, gd, grads, hits)
    return _cache[key]


@pytest.mark.parametrize("name", ["tiny_tri", "small_tri"])
def test_closed_form_matches_autograd_and_oracle(name):
    cpu, gc, gd, grads, hits = hits_for(name)
    P = cpu.verts.shape[0]
    assert hits["u"].numel() > 0
    exact = closed_form_vertex_grads(hits, cpu.faces, P, exact=True)
    e = rel_l2(exact.numpy(), grads["verts"].numpy())
    print("\n[exact closed form] %s: rel L2 vs autograd %.2e" % (name, e))
    assert e <= 1e-9
    # the reference's t-statistics reproduce the CPU oracle's (i.e. the reference extension's) dL/dverts
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import oracle
    o = oracle.TriOracle(cpu)
    try:
        g_oracle = o.backward(gc, gd)[0]
    finally:
        o.close()
    ref = closed_form_vertex_grads(hits, cpu.faces, P, exact=False).numpy()
    # Faces hit at a grazing angle (|rd.n| < 1e-2: D tiny against |E2 x E1|) are left out on both sides: there the
    # oracle's fp32 (u, v) and t carry a large relative error (dL/dverts grows like 1/D), which fp64 does not reproduce
    # -- one such face of small_tri alone makes 1.3e-3 relative L2.
    n = torch.linalg.cross(hits["E2"], hits["E1"])
    cos = (hits["rd"] * n).sum(1).abs() / n.norm(dim=1)
    grazing = torch.unique(hits["f"][cos < 1e-2])
    keep = np.ones(P, bool)
    keep[cpu.faces.long()[grazing].reshape(-1).numpy()] = False
    e_ref = rel_l2(ref[keep], g_oracle[keep])
    print("[reference closed form] %s: rel L2 vs oracle %.2e (%d grazing faces left out; %.2e with them); reference "
          "vs exact %.2e" % (name, e_ref, grazing.numel(), rel_l2(ref, g_oracle), rel_l2(ref, exact.numpy())))
    assert grazing.numel() <= 0.01 * cpu.faces.shape[0]
    assert e_ref <= 1e-4


@pytest.mark.parametrize("fused", [False, True], ids=["explicit_depth", "fused_depth"])
@pytest.mark.parametrize("name", ["tiny_tri", "cam4"])
def test_rigid_motion_identity_fp64_reference(name, fused):
    cpu, gc, gd, grads, hits = hits_for(name, fused, fp64_inverse=True)
    r, s = rigid_residual(cpu.verts, cpu.mv_mats, grads["verts"], grads["mv_mats"])
    print("\n[rigid motion, fp64 autograd] %s %s: residual %.2e of %.2e" % (name, fused, r, s))
    assert s > 0 and r <= 1e-9 * s
    # the closed form in place of autograd's vertex gradient (the depth chain of the fused depth is autograd's part
    # beyond the geometry, so it is compared with explicit depth only); the reference formula is printed only
    if not fused:
        P = cpu.verts.shape[0]
        r, s = rigid_residual(cpu.verts, cpu.mv_mats, closed_form_vertex_grads(hits, cpu.faces, P, True), grads["mv_mats"])
        assert r <= 1e-9 * s
        r0, s0 = rigid_residual(cpu.verts, cpu.mv_mats, closed_form_vertex_grads(hits, cpu.faces, P, False),
                                grads["mv_mats"])
        print("[rigid motion] closed form exact %.2e, reference formula %.2e (relative)" % (r / s, r0 / s0))


def test_backward_exact_rejects_bad_arguments():
    """dmr_tri_backward_exact validates its arguments before any CUDA call (no GPU needed)."""
    from dmesh_renderer_b200 import _lib
    lib = _lib.load()
    fake = ctypes.c_void_p(256)             # never dereferenced: every case fails before a kernel is enqueued
    null = ctypes.c_void_p(0)
    B, P, F, W, H, R = 2, 30, 10, 32, 32, 100

    def call(ptrs=None, det=0, mv=fake, pj=fake, ws=fake, nbytes=1 << 30):
        p = [fake] * 14 if ptrs is None else ptrs
        return lib.dmr_tri_backward_exact(B, P, F, W, H, R, *p, det, mv, pj, ws, nbytes, null)

    assert call(mv=fake, pj=null) == 1 and b"dL_dmv" in lib.dmr_last_error()
    assert call(mv=null, pj=fake) == 1
    for i in (0, 1, 2, 4, 5, 6, 7, 8, 9, 10, 11, 12, 13):   # every pointer the backward reads or writes
        ptrs = [fake] * 14
        ptrs[i] = null
        assert call(ptrs) == 1 and b"null" in lib.dmr_last_error(), i
    for det in (0, 1):
        for cam in (False, True):
            mv = fake if cam else null
            need = (lib.dmr_tri_backward_camera_bytes(B, P, F, W, H, det) if cam else
                    lib.dmr_tri_backward_deterministic_bytes(B, P, F) if det else lib.dmr_tri_backward_workspace_bytes(B, P, F))
            assert call(det=det, mv=mv, pj=mv, nbytes=need - 1) == 1, (det, cam)
            assert b"workspace" in lib.dmr_last_error()
            assert call(det=det, mv=mv, pj=mv, ws=null, nbytes=need) == 1, (det, cam)
    # sizes are checked first, and an empty call is a no-op
    assert lib.dmr_tri_backward_exact(-1, P, F, W, H, R, *([fake] * 14), 0, null, null, fake, 0, null) != 0
    assert lib.dmr_tri_backward_exact(B, P, F, W, H, 0, *([null] * 14), 0, null, null, null, 0, null) == 0
