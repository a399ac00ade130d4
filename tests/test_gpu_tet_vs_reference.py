"""GPU parity: CUDA tet path against the reference renderer: the UNMODIFIED reference extension (oracle/_ref) when
it is built; otherwise the CPU oracle (its port), itself checked against the recorded reference outputs of every scene
(tests/golden/parity_record.npz), and for jittered rays (ray_random_seed > 0) that record directly -- tests/ref_harness.py.

  * binning integers (tiles_touched, offsets, sorted keys/values, ranges),
    first_face / first_tet, n_contrib, active mask: bit-exact
  * images: <= 1e-5 max-abs; gradients: <= 1e-4 relative L2
"""
import numpy as np
import pytest
import torch

import binning_checks
import ref_harness
from dmesh_renderer_b200 import TetRenderer, TetRenderSettings, _C, debug, scenes
from test_gpu_tri_vs_reference import exactly_scaled

pytestmark = pytest.mark.gpu

IMG_TOL = 1e-5
GRAD_TOL = 1e-4


def rel_l2(a, b):
    a, b = a.double(), b.double()
    return ((a - b).norm() / b.norm().clamp_min(1e-30)).item()


def ours_forward(s, seed=0):
    mv, pj = s.mv_mats.transpose(1, 2), s.proj_mats.transpose(1, 2)
    imv, ipj = torch.inverse(mv), torch.inverse(pj)
    return _C.render_tets(s.bg, s.verts, s.faces, s.verts_color, s.faces_opacity, mv, pj, imv, ipj, s.verts_depth,
                          s.faces_intense, s.tets, s.face_tets, s.tet_faces, s.H, s.W, seed)


@pytest.mark.parametrize("name,seed", [("tiny_tet", 0), ("small_tet", 0), ("C3", 0), ("small_tet", 7)])
def test_tet_forward(name, seed):
    s = scenes.to_device(scenes.config(name), "cuda")
    if not ref_harness.tet_seed_supported(seed):      # jittered rays, no extension: the recorded reference output
        out = ours_forward(s, seed)
        R, ints = ref_harness.cuda_tet_ints(s, out)
        ref_harness.check_forward(ref_harness.scene_key(s, seed), R, ints, out[0], out[1])
        assert (out[2] > 0.5).float().mean().item() > 0.3
        return
    B, P, F, T = s.mv_mats.shape[0], s.verts.shape[0], s.faces.shape[0], s.tets.shape[0]
    ref = ref_harness.ref_tet_forward(s, seed)
    ri = ref_harness.ref_tet_intermediates(s, ref)
    color, depth, active, pb, fb, bb, ib = ours_forward(s, seed)
    R = ri["R"]
    dims = dict(B=B, P=P, F=F, W=s.W, H=s.H, R=R, T=T)
    tt = debug.view("tet", "tiles_touched", fb, **dims)
    np.testing.assert_array_equal(tt, ri["tiles_touched"])
    live = tt > 0
    dk = debug.view("tet", "depth_keys", fb, **dims)
    np.testing.assert_array_equal(dk[live], ri["min_depths"].view(np.uint32)[live])
    binning_checks.check_face_order_and_offsets(debug.view("tet", "face_order", fb, **dims), dk, tt,
                                                debug.view("tet", "offsets", fb, **dims), ri["offsets"])
    np.testing.assert_array_equal(debug.view("tet", "keys_sorted", bb, face_buffer=fb, **dims), ri["keys_sorted"])
    np.testing.assert_array_equal(debug.view("tet", "values_sorted", bb, **dims), ri["values_sorted"])
    np.testing.assert_array_equal(debug.view("tet", "ranges", ib, **dims), ri["ranges"])
    np.testing.assert_array_equal(debug.view("tet", "first_face", ib, **dims), ri["first_face"])
    np.testing.assert_array_equal(debug.view("tet", "first_tet", ib, **dims), ri["first_tet"])
    np.testing.assert_array_equal(debug.view("tet", "n_contrib", ib, **dims), ri["n_contrib"])
    assert torch.equal(active > 0.5, ref["active"] > 0.5)
    assert (color - ref["color"]).abs().max().item() <= IMG_TOL
    assert (depth - ref["depth"]).abs().max().item() <= IMG_TOL
    # the scene must actually exercise the march
    assert (active > 0.5).float().mean().item() > 0.3


@pytest.mark.parametrize("name,seed", [("tiny_tet", 0), ("small_tet", 0), ("C3", 0), ("small_tet", 7)])
def test_tet_gradients(name, seed):
    s = scenes.to_device(scenes.config(name), "cuda")
    gc, gd = [t.cuda() for t in scenes.cotangents(s)]
    rg = None                                         # jittered rays, no extension: the recorded reference gradients
    if ref_harness.tet_seed_supported(seed):
        ref = ref_harness.ref_tet_forward(s, seed)
        rg = ref_harness.ref_tet_backward(s, ref, gc, gd)

    vc = s.verts_color.clone().requires_grad_()
    fo = s.faces_opacity.clone().requires_grad_()
    renderer = TetRenderer(TetRenderSettings(s.H, s.W, s.bg, seed))
    color, depth, active = renderer(s.verts, s.faces, vc, fo, s.mv_mats, s.proj_mats, s.verts_depth, s.faces_intense,
                                    s.tets, s.face_tets, s.tet_faces)
    assert active.dtype == torch.bool
    torch.autograd.backward([color, depth], [gc, gd])
    if rg is None:
        ref_harness.check_grads(ref_harness.scene_key(s, seed), [vc.grad, fo.grad])
        return
    for n, g, r in (("verts_color", vc.grad, rg[0]), ("faces_opacity", fo.grad, rg[1])):
        e = rel_l2(g, r)
        assert e <= GRAD_TOL, "%s: rel L2 %.3e" % (n, e)


@pytest.mark.parametrize("cap", [1, 7])
@pytest.mark.parametrize("name", ["small_tet", "C3"])
def test_tet_gradients_short_trail(name, cap):
    """Rays that composite more faces than the face trail holds re-march the part beyond the cap
    through the adjacency records (as the reference does for the whole ray): same gradients."""
    from dmesh_renderer_b200 import _lib
    lib = _lib.load()
    s = scenes.to_device(scenes.config(name), "cuda")
    gc, gd = [t.cuda() for t in scenes.cotangents(s)]
    ref = ref_harness.ref_tet_forward(s, 0)
    rg = ref_harness.ref_tet_backward(s, ref, gc, gd)
    lib.dmr_debug_set_tet_trail_cap(cap)
    try:
        vc = s.verts_color.clone().requires_grad_()
        fo = s.faces_opacity.clone().requires_grad_()
        renderer = TetRenderer(TetRenderSettings(s.H, s.W, s.bg, 0))
        color, depth, active = renderer(s.verts, s.faces, vc, fo, s.mv_mats, s.proj_mats, s.verts_depth,
                                        s.faces_intense, s.tets, s.face_tets, s.tet_faces)
        torch.autograd.backward([color, depth], [gc, gd])
        torch.cuda.synchronize()
    finally:
        lib.dmr_debug_set_tet_trail_cap(0)
    assert (color - ref["color"]).abs().max().item() <= IMG_TOL
    for n, g, r in (("verts_color", vc.grad, rg[0]), ("faces_opacity", fo.grad, rg[1])):
        e = rel_l2(g, r)
        assert e <= GRAD_TOL, "%s: rel L2 %.3e" % (n, e)


@pytest.mark.parametrize("split", [1, 2, 3])
def test_tet_first_intersection_does_not_depend_on_the_tile_split(split):
    from dmesh_renderer_b200 import _lib
    lib = _lib.load()
    s = scenes.to_device(scenes.config("small_tet"), "cuda")
    B, P, F, T = s.mv_mats.shape[0], s.verts.shape[0], s.faces.shape[0], s.tets.shape[0]
    ref = ref_harness.ref_tet_forward(s, 0)
    ri = ref_harness.ref_tet_intermediates(s, ref)
    lib.dmr_debug_set_tet_first_split(split)
    try:
        color, depth, active, pb, fb, bb, ib = ours_forward(s, 0)
        torch.cuda.synchronize()
    finally:
        lib.dmr_debug_set_tet_first_split(0)
    dims = dict(B=B, P=P, F=F, W=s.W, H=s.H, R=ri["R"], T=T)
    np.testing.assert_array_equal(debug.view("tet", "first_face", ib, **dims), ri["first_face"])
    np.testing.assert_array_equal(debug.view("tet", "first_tet", ib, **dims), ri["first_tet"])
    np.testing.assert_array_equal(debug.view("tet", "n_contrib", ib, **dims), ri["n_contrib"])


def test_tet_validation_errors():
    s = scenes.to_device(scenes.config("tiny_tet"), "cuda")
    mv, pj = s.mv_mats.transpose(1, 2), s.proj_mats.transpose(1, 2)
    imv, ipj = torch.inverse(mv), torch.inverse(pj)
    with pytest.raises(RuntimeError, match="tet_faces must have dimensions"):
        _C.render_tets(s.bg, s.verts, s.faces, s.verts_color, s.faces_opacity, mv, pj, imv, ipj, s.verts_depth,
                       s.faces_intense, s.tets, s.face_tets, s.tet_faces[:5], s.H, s.W, 0)
    with pytest.raises(RuntimeError, match="face_tets must have dimensions"):
        _C.render_tets(s.bg, s.verts, s.faces, s.verts_color, s.faces_opacity, mv, pj, imv, ipj, s.verts_depth,
                       s.faces_intense, s.tets, s.face_tets[:, :1], s.tet_faces, s.H, s.W, 0)


@pytest.mark.parametrize("name,seed,cap", [("small_tet", 0, 0), ("C3", 0, 0), ("small_tet", 7, 3)])
def test_tet_deterministic_backward_is_reproducible_and_matches(name, seed, cap):
    """TetRenderer(..., deterministic=True): bit-identical gradients on every run (64-bit fixed-point accumulation
    instead of fp32 atomics), within the gradient tolerance of the reference extension, exactly linear under
    power-of-two scales of the cotangents; also with a short face trail (re-march path) and jittered rays (compared
    with the recorded reference gradients when the extension is not built)."""
    from dmesh_renderer_b200 import _lib
    lib = _lib.load()
    s = scenes.to_device(scenes.config(name), "cuda")
    gc, gd = [t.cuda() for t in scenes.cotangents(s)]
    rg = None
    if ref_harness.tet_seed_supported(seed):
        ref = ref_harness.ref_tet_forward(s, seed)
        rg = ref_harness.ref_tet_backward(s, ref, gc, gd)

    def grads(k=1.0):
        vc = s.verts_color.clone().requires_grad_()
        fo = s.faces_opacity.clone().requires_grad_()
        renderer = TetRenderer(TetRenderSettings(s.H, s.W, s.bg, seed), deterministic=True)
        color, depth, _ = renderer(s.verts, s.faces, vc, fo, s.mv_mats, s.proj_mats, s.verts_depth, s.faces_intense,
                                   s.tets, s.face_tets, s.tet_faces)
        torch.autograd.backward([color, depth], [gc * k, gd * k])
        return vc.grad, fo.grad

    lib.dmr_debug_set_tet_trail_cap(cap)
    try:
        runs = [grads() for _ in range(3)]
        for r in runs[1:]:
            assert torch.equal(r[0], runs[0][0]) and torch.equal(r[1], runs[0][1])
        if rg is None:
            ref_harness.check_grads(ref_harness.scene_key(s, seed), runs[0])
        for n, g, r in (("verts_color", runs[0][0], rg[0]), ("faces_opacity", runs[0][1], rg[1])) if rg else ():
            e = rel_l2(g, r)
            assert e <= GRAD_TOL, "%s: rel L2 %.3e" % (n, e)
        # max |cotangent| from near 2^-80 to 2^100: the binary point follows g (det.cuh)
        for k in (2.0 ** -80, 2.0 ** -30, 2.0 ** 20, 2.0 ** 100):
            a, b = grads(k)
            assert exactly_scaled(runs[0][0], a, k) and exactly_scaled(runs[0][1], b, k), k
        z = grads(0.0)
        assert float(z[0].abs().max()) == 0.0 and float(z[1].abs().max()) == 0.0
    finally:
        lib.dmr_debug_set_tet_trail_cap(0)


def _with_irregular_tets(s, nfaces=40, shift=2e-3, seed=5):
    """A copy of scene `s` (on the CPU) whose tables are INCONSISTENT for `nfaces` interior faces: the face's first
    vertex is replaced by a slightly shifted copy of it, so both tets next to the face have a side that is not made of
    their own four vertices.  The reference marches through such tets with the vertices it gathers through faces[];
    the compact adjacency records cannot present them (TetRec code 0xF) and take the out-of-line path."""
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


def test_tet_irregular_tets_follow_the_reference():
    """Tets whose sides are not made of their own vertices: same march decisions, images and gradients as the
    reference (which gathers every side through faces[] / verts[])."""
    s = scenes.to_device(_with_irregular_tets(scenes.config("small_tet")), "cuda")
    B, P, F, T = s.mv_mats.shape[0], s.verts.shape[0], s.faces.shape[0], s.tets.shape[0]
    ref = ref_harness.ref_tet_forward(s, 0)
    ri = ref_harness.ref_tet_intermediates(s, ref)
    color, depth, active, pb, fb, bb, ib = ours_forward(s, 0)
    dims = dict(B=B, P=P, F=F, W=s.W, H=s.H, R=ri["R"], T=T)
    np.testing.assert_array_equal(debug.view("tet", "first_face", ib, **dims), ri["first_face"])
    np.testing.assert_array_equal(debug.view("tet", "n_contrib", ib, **dims), ri["n_contrib"])
    assert torch.equal(active > 0.5, ref["active"] > 0.5)
    assert (color - ref["color"]).abs().max().item() <= IMG_TOL
    assert (depth - ref["depth"]).abs().max().item() <= IMG_TOL
    assert (active > 0.5).float().mean().item() > 0.3      # rays still get through the perturbed tets

    gc, gd = [t.cuda() for t in scenes.cotangents(s)]
    rg = ref_harness.ref_tet_backward(s, ref, gc, gd)
    vc = s.verts_color.clone().requires_grad_()
    fo = s.faces_opacity.clone().requires_grad_()
    renderer = TetRenderer(TetRenderSettings(s.H, s.W, s.bg, 0))
    c2, d2, _ = renderer(s.verts, s.faces, vc, fo, s.mv_mats, s.proj_mats, s.verts_depth, s.faces_intense, s.tets,
                         s.face_tets, s.tet_faces)
    torch.autograd.backward([c2, d2], [gc, gd])
    for n, g, r in (("verts_color", vc.grad, rg[0]), ("faces_opacity", fo.grad, rg[1])):
        e = rel_l2(g, r)
        assert e <= GRAD_TOL, "%s: rel L2 %.3e" % (n, e)
