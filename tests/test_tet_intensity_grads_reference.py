"""CPU: the tet renderer's face-intensity gradients (intensity_grads=True), checked without a GPU.

The step's colour is intense * interp (interp = the interpolated vertex colour), so per walked step
    dL/dfaces_intense[b, face] += sum_ch dL/dcol[ch] T alpha interp[ch]
(tet_int_step, csrc/tet_kernels.cu).  The yardstick of the GPU tests is the fp64 reference of
tests/test_tet_vertex_grads_reference.py, whose `faces_intense` leaf carries this gradient; here it is checked against
central differences of the same fp64 forward, and against Euler's identity: with a black background the colour image
is homogeneous of degree 1 in the intensities, so sum_f I[b,f] dL/dI[b,f] = <dL/dcolor[b], color[b]> over the pixels
whose every fragment the backward pass walks.
"""
import ctypes

import numpy as np
import torch

from dmesh_renderer_b200 import scenes
from test_gpu_tet_camera_grads import oracle_fragments
from test_tet_vertex_grads_reference import reference_grads_verts, reference_render_verts

f64 = torch.float64


def with_intensities(cpu, seed=11, zero_frac=0.1, black=False):
    """A copy of scene `cpu` with random per-view face intensities in [0.2, 1], a fraction `zero_frac` of them 0, and
    (black=True) a black background."""
    g = torch.Generator().manual_seed(seed)
    fint = torch.rand(cpu.faces_intense.shape, generator=g) * 0.8 + 0.2
    fint[torch.rand(fint.shape, generator=g) < zero_frac] = 0.0
    s = cpu._replace(faces_intense=fint.contiguous())
    return s._replace(bg=torch.zeros(3)) if black else s


def fully_walked(cpu, frags):
    """[B,1,H,W] float mask of the pixels all of whose fragments are walked by the backward pass (inactive pixels
    included: they composite nothing)."""
    B, H, W = cpu.mv_mats.shape[0], cpu.H, cpu.W
    cnt = torch.from_numpy(frags["counts"].astype(np.int64))
    pix = torch.repeat_interleave(torch.arange(B * H * W), cnt)
    unreached = torch.zeros(B * H * W, dtype=torch.bool)
    unreached[pix[~torch.from_numpy(frags["reach"])]] = True
    return (~unreached).view(B, 1, H, W).to(f64)


def euler_terms(fint, g_fint, gc, color):
    """Per view: (sum_f I dL/dI, <dL/dcolor, color>, sum of |terms| on the left)."""
    t = fint.to(f64) * g_fint.to(f64)
    return t.sum(1), (gc.to(f64) * color.to(f64)).flatten(1).sum(1), t.abs().sum(1)


def test_reference_matches_central_differences():
    cpu = with_intensities(scenes.config("tiny_tet"))
    gc, gd = scenes.cotangents(cpu)
    frags, _ = oracle_fragments(cpu, gradients=(gc, gd))
    _, _, g, _ = reference_grads_verts(cpu, frags, gc, gd)
    gi = g["faces_intense"]
    d = lambda t: t.to(f64)

    def loss(fint):
        color, depth, _ = reference_render_verts(frags, cpu, d(cpu.verts), d(cpu.verts_color), d(cpu.faces_opacity),
                                                 d(cpu.mv_mats), d(cpu.proj_mats), fint)
        return float((color * gc.to(f64)).sum() + (depth * gd.to(f64)).sum())

    # entries with the largest gradients, faces of intensity 0 among them, and a few that get none
    zero = (cpu.faces_intense == 0) & (gi != 0)
    big = gi.abs().flatten().argsort(descending=True)[:12]
    idx = torch.cat([big, zero.flatten().nonzero().flatten()[:8], (gi == 0).flatten().nonzero().flatten()[:4]])
    assert zero.any() and (gi == 0).any()
    h = 1e-3
    base = cpu.faces_intense.to(f64)
    for i in idx.tolist():
        fp, fm = base.clone(), base.clone()
        fp.view(-1)[i] += h
        fm.view(-1)[i] -= h
        fd = (loss(fp) - loss(fm)) / (2 * h)
        assert abs(fd - float(gi.view(-1)[i])) <= 1e-8 * max(1.0, abs(fd)), (i, fd, float(gi.view(-1)[i]))


def test_reference_satisfies_eulers_identity():
    cpu = with_intensities(scenes.config("tiny_tet"), black=True)
    gc, gd = scenes.cotangents(cpu)
    frags, _ = oracle_fragments(cpu, gradients=(gc, gd))
    m = fully_walked(cpu, frags)
    gc = gc.to(f64) * m
    color, _, g, _ = reference_grads_verts(cpu, frags, gc, gd * 0)
    lhs, rhs, s = euler_terms(cpu.faces_intense, g["faces_intense"], gc, color)
    print("\n[tet intensity Euler, fp64] residual %s of %s" % ((lhs - rhs).abs().tolist(), s.tolist()))
    assert (s > 0).all()
    assert ((lhs - rhs).abs() <= 1e-10 * s).all()
    # faces of intensity 0 contribute nothing to the left side but do get a gradient
    assert ((cpu.faces_intense == 0) & (g["faces_intense"] != 0)).any()


def test_backward_intensity_rejects_bad_arguments():
    """dmr_tet_backward_intensity validates its arguments before any CUDA call (no GPU needed)."""
    from dmesh_renderer_b200 import _lib
    lib = _lib.load()
    fake = ctypes.c_void_p(256)             # never dereferenced: every case fails before a kernel is enqueued
    null = ctypes.c_void_p(0)
    B, P, F, T, W, H = 2, 30, 40, 10, 32, 32

    def call(ptrs=None, det=0, mv=fake, pj=fake, dv=fake, di=fake, ws=fake, nbytes=1 << 30):
        p = [fake] * 14 if ptrs is None else ptrs
        return lib.dmr_tet_backward_intensity(B, P, F, T, W, H, 0, *p, det, mv, pj, dv, di, ws, nbytes, null)

    assert call(mv=fake, pj=null) == 1 and b"dL_dmv" in lib.dmr_last_error()
    assert call(mv=null, pj=fake) == 1 and b"dL_dmv" in lib.dmr_last_error()
    assert call(di=null) == 1 and b"dL_dfaces_intense" in lib.dmr_last_error()
    for i in (0, 1, 2, 3, 4, 5, 7, 8, 9, 10, 11, 12, 13):   # every pointer the backward reads or writes
        ptrs = [fake] * 14
        ptrs[i] = null
        assert call(ptrs) == 1 and b"null" in lib.dmr_last_error(), i
    for det in (0, 1):
        for cam in (0, 1):
            for vert in (0, 1):
                mv = fake if cam else null
                dv = fake if vert else null
                need = lib.dmr_tet_backward_intensity_bytes(B, P, F, W, H, det, cam, vert)
                base = (lib.dmr_tet_backward_vertex_bytes(B, P, F, W, H, det, cam) if vert else
                        lib.dmr_tet_backward_camera_bytes(B, P, F, W, H, det) if cam else
                        lib.dmr_tet_backward_deterministic_bytes(P, F) if det else lib.dmr_tet_backward_workspace_bytes(P))
                # deterministic mode: one two-word fixed-point accumulator per (view, face); default mode: nothing more
                assert need >= base + (16 * B * F if det else 0), (det, cam, vert)
                if not det:
                    assert need == base, (cam, vert)
                key = (det, cam, vert)
                assert call(det=det, mv=mv, pj=mv, dv=dv, nbytes=need - 1) == 1, key
                assert b"dmr_tet_backward_intensity_bytes" in lib.dmr_last_error(), key
                assert call(det=det, mv=mv, pj=mv, dv=dv, ws=null, nbytes=need) == 1, key
                assert b"dmr_tet_backward_intensity_bytes" in lib.dmr_last_error(), key
    for bad in ((-1, P, F, W, H), (B, -1, F, W, H), (B, P, -1, W, H), (B, P, F, -1, H), (B, P, F, W, -1)):
        assert lib.dmr_tet_backward_intensity_bytes(*bad, 0, 0, 0) == 0, bad
    # sizes are checked first, and an empty call is a no-op
    for bad in ((-1, P, F, T, W, H), (B, -1, F, T, W, H), (B, P, -1, T, W, H), (B, P, F, -1, W, H), (B, P, F, T, 0, H)):
        assert lib.dmr_tet_backward_intensity(*bad, 0, *([fake] * 14), 0, null, null, null, fake, fake, 1 << 30,
                                              null) != 0, bad
    assert lib.dmr_tet_backward_intensity(0, P, F, T, W, H, 0, *([null] * 14), 0, null, null, null, null, null, 0,
                                          null) == 0
