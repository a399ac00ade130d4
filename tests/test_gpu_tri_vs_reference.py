"""GPU parity: CUDA tri path (through the public API -> _C shim -> C ABI) against
the reference renderer on identical seeded scenes: the UNMODIFIED reference extension (oracle/_ref) when it is
built, the CPU oracle (its port, pinned to the reference's stored outputs) otherwise -- tests/ref_harness.py.

Tolerances (BASELINE.json north_star):
  * integer / indexing work (tiles_touched, offsets, R, sorted keys + values,
    tile ranges, n_contrib): bit-exact
  * forward images: <= 1e-5 max-abs
  * gradients: <= 1e-4 relative L2 (atomic reordering allowed)
"""
import numpy as np
import pytest
import torch

import binning_checks
import ref_harness
from dmesh_renderer_b200 import TriRenderer, TriRenderSettings, _C, debug, scenes

pytestmark = pytest.mark.gpu

IMG_TOL = 1e-5
GRAD_TOL = 1e-4


def rel_l2(a, b):
    a, b = a.double(), b.double()
    return ((a - b).norm() / b.norm().clamp_min(1e-30)).item()


def exactly_scaled(a, b, k):
    """b == a * k bit for bit, except that a result below the fp32 normal range (2^-126) is rounded once from the
    exact value in b and twice in a * k: there the two may differ by one subnormal step."""
    ak = a.double() * k
    normal = ak.abs() >= 2.0 ** -126
    return torch.equal((a * k)[normal], b[normal]) and bool(((ak - b.double()).abs()[~normal] <= 2.0 ** -149).all())


def ours_forward(s):
    mv, pj = s.mv_mats.transpose(1, 2), s.proj_mats.transpose(1, 2)
    imv, ipj = torch.inverse(mv), torch.inverse(pj)
    out = _C.render_tris(s.bg, s.verts, s.faces, s.verts_color, s.faces_opacity, mv, pj, imv, ipj, s.verts_depth,
                         s.faces_intense, s.H, s.W)
    return out, (mv, pj, imv, ipj)


@pytest.mark.parametrize("name", ["tiny_tri", "small_tri", "C1", "C2"])
def test_tri_intermediates_and_images(name):
    s = scenes.to_device(scenes.config(name), "cuda")
    B, P, F = s.mv_mats.shape[0], s.verts.shape[0], s.faces.shape[0]
    ref = ref_harness.ref_tri_forward(s)
    ri = ref_harness.ref_tri_intermediates(s, ref)
    (R, color, depth, pb, fb, bb, ib), _ = ours_forward(s)

    dims = dict(B=B, P=P, F=F, W=s.W, H=s.H, R=R)
    vimg = debug.view("tri", "verts_image", pb, **dims)
    np.testing.assert_array_equal(vimg[:, :2].view(np.uint32), ri["verts_image"].view(np.uint32))
    np.testing.assert_array_equal(vimg[:, 2].view(np.uint32), ri["ndc_z"].view(np.uint32))
    tt = debug.view("tri", "tiles_touched", fb, **dims)
    np.testing.assert_array_equal(tt, ri["tiles_touched"])
    assert R == ref["R"]
    dk = debug.view("tri", "depth_keys", fb, **dims)
    live = tt > 0      # culled faces leave depths[] unwritten in the reference (SURVEY App. B)
    np.testing.assert_array_equal(dk[live], ri["depths"].view(np.uint32)[live])
    binning_checks.check_face_order_and_offsets(debug.view("tri", "face_order", fb, **dims), dk, tt,
                                                debug.view("tri", "offsets", fb, **dims), ri["offsets"])
    binning_checks.check_same_pairs(debug.view("tri", "keys_unsorted", bb, face_buffer=fb, **dims),
                                    debug.view("tri", "values_unsorted", bb, **dims),
                                    ri["keys_unsorted"], ri["values_unsorted"])
    np.testing.assert_array_equal(debug.view("tri", "keys_sorted", bb, face_buffer=fb, **dims), ri["keys_sorted"])
    np.testing.assert_array_equal(debug.view("tri", "values_sorted", bb, **dims), ri["values_sorted"])
    np.testing.assert_array_equal(debug.view("tri", "ranges", ib, **dims), ri["ranges"])
    np.testing.assert_array_equal(debug.view("tri", "n_contrib", ib, **dims), ri["n_contrib"])
    np.testing.assert_array_equal(debug.view("tri", "final_T", ib, **dims).view(np.uint32), ri["final_T"].view(np.uint32))

    assert (color - ref["color"]).abs().max().item() <= IMG_TOL
    assert (depth - ref["depth"]).abs().max().item() <= IMG_TOL


@pytest.mark.parametrize("name", ["tiny_tri", "small_tri", "C1", "C2"])
def test_tri_gradients(name):
    s = scenes.to_device(scenes.config(name), "cuda")
    gc, gd = [t.cuda() for t in scenes.cotangents(s)]
    ref = ref_harness.ref_tri_forward(s)
    rg = ref_harness.ref_tri_backward(s, ref, gc, gd)

    leaves = [s.verts.clone().requires_grad_(), s.verts_color.clone().requires_grad_(),
              s.faces_opacity.clone().requires_grad_(), s.verts_depth.clone().requires_grad_(),
              s.faces_intense.clone().requires_grad_()]
    renderer = TriRenderer(TriRenderSettings(s.H, s.W, s.bg))
    color, depth = renderer(leaves[0], s.faces, leaves[1], leaves[2], s.mv_mats, s.proj_mats, leaves[3], leaves[4])
    torch.autograd.backward([color, depth], [gc, gd])
    names = ["verts", "verts_color", "faces_opacity", "verts_depth", "faces_intense"]
    for n, leaf, r in zip(names, leaves, rg):
        e = rel_l2(leaf.grad, r)
        assert e <= GRAD_TOL, "%s: rel L2 %.3e" % (n, e)


def test_tri_empty_and_edge_cases():
    dev = "cuda"
    s = scenes.to_device(scenes.config("tiny_tri"), dev)
    mv, pj = s.mv_mats.transpose(1, 2), s.proj_mats.transpose(1, 2)
    imv, ipj = torch.inverse(mv), torch.inverse(pj)
    B = mv.shape[0]
    # P == 0: zero images, empty buffers (render.cu:88-89,105)
    e = torch.zeros
    out = _C.render_tris(s.bg, e(0, 3, device=dev), e(0, 3, dtype=torch.int32, device=dev), e(0, 3, device=dev),
                         e(0, device=dev), mv, pj, imv, ipj, e(B, 0, device=dev), e(B, 0, device=dev), s.H, s.W)
    assert out[0] == 0 and out[1].abs().max().item() == 0 and out[3].numel() == 0
    # everything behind the camera: background image, R == 0, zero gradients
    verts = s.verts.clone()
    verts[:, :] = s.verts * 0.01 + torch.tensor([3.0, 2.0, 10.0], device=dev) * 3
    R, color, depth, pb, fb, bb, ib = _C.render_tris(s.bg, verts, s.faces, s.verts_color, s.faces_opacity, mv, pj, imv, ipj,
                                                     s.verts_depth, s.faces_intense, s.H, s.W)
    assert R == 0
    assert torch.equal(color, torch.ones_like(color)) and torch.equal(depth, torch.ones_like(depth))
    g = _C.render_tris_backward(s.bg, verts, s.faces, s.verts_color, s.faces_opacity, mv, pj, imv, ipj, s.verts_depth,
                                s.faces_intense, torch.ones_like(color), torch.ones_like(depth), R, pb, fb, bb, ib)
    assert all(t.abs().max().item() == 0 for t in g)
    # validation errors carry the reference's messages (render.cu:49-79)
    with pytest.raises(RuntimeError, match="verts must have dimensions"):
        _C.render_tris(s.bg, s.verts[:, :2], s.faces, s.verts_color, s.faces_opacity, mv, pj, imv, ipj, s.verts_depth,
                       s.faces_intense, s.H, s.W)
    with pytest.raises(RuntimeError, match="faces_intense must have dimensions"):
        _C.render_tris(s.bg, s.verts, s.faces, s.verts_color, s.faces_opacity, mv, pj, imv, ipj, s.verts_depth,
                       s.faces_intense[:, :5], s.H, s.W)


def test_tri_non_multiple_of_16_image():
    s = scenes.random_tri_scene("odd", 21, 2000, 0.1, 100, 75, B=2)
    s = scenes.to_device(s, "cuda")
    ref = ref_harness.ref_tri_forward(s)
    (R, color, depth, *_), _ = ours_forward(s)
    assert R == ref["R"]
    assert (color - ref["color"]).abs().max().item() <= IMG_TOL
    assert (depth - ref["depth"]).abs().max().item() <= IMG_TOL


def test_inverses_on_gpu_are_torch_inverse_bits_and_singular_raises():
    from dmesh_renderer_b200 import TriRenderer, TriRenderSettings
    s = scenes.to_device(scenes.config("tiny_tri"), "cuda")
    mv, pj = s.mv_mats.transpose(1, 2), s.proj_mats.transpose(1, 2)
    inv = _C._Inverses(mv, pj)
    torch.cuda.synchronize()
    inv.check()
    assert torch.equal(inv.inv_mv, torch.inverse(mv)) and torch.equal(inv.inv_proj, torch.inverse(pj))
    assert inv.mv.is_contiguous() and torch.equal(inv.mv, mv) and torch.equal(inv.proj, pj)
    # csrc/inverse.cu against torch.inverse, bit for bit: random matrices, the cameras of every benchmark scene,
    # contiguous and transposed views, B = 1 and B > 1 (torch takes different library paths for the two)
    g = torch.Generator().manual_seed(5)
    stacks = [(torch.randn(4096, 4, 4, generator=g), torch.randn(4096, 4, 4, generator=g) * 100.0)]
    for name in ("C1", "C2", "C4", "C3"):
        c = scenes.config(name)
        stacks.append((c.mv_mats, c.proj_mats))
    for a, b in stacks:
        a, b = a.cuda(), b.cuda()
        for x, y in ((a, b), (a.transpose(1, 2), b.transpose(1, 2)), (a[:1], b[:1]), (a[:1].transpose(1, 2), b[:1].transpose(1, 2))):
            inv = _C._Inverses(x, y)
            torch.cuda.synchronize()
            inv.check()
            assert torch.equal(inv.inv_mv.view(torch.int32), torch.inverse(x).view(torch.int32))
            assert torch.equal(inv.inv_proj.view(torch.int32), torch.inverse(y).view(torch.int32))
    r = TriRenderer(TriRenderSettings(s.H, s.W, s.bg))
    bad = s.proj_mats.clone()
    bad[0] = 0
    with pytest.raises(RuntimeError, match="singular"):
        r(s.verts, s.faces, s.verts_color, s.faces_opacity, s.mv_mats, bad, s.verts_depth, s.faces_intense)


def test_speculative_binning_buffer_when_num_rendered_grows():
    """The binning buffer is pre-sized from the previous call with the same shapes; a call whose num_rendered
    outgrows it must fall back to an exact allocation (same shapes, camera far -> near)."""
    far = scenes.random_tri_scene("far", 11, 4000, 0.05, 160, 160, dist=8.0, far=12.0)
    near = scenes.random_tri_scene("near", 11, 4000, 0.12, 160, 160, dist=2.0)
    R = []
    for cpu in (far, near, far):
        s = scenes.to_device(cpu, "cuda")
        gc, gd = [t.cuda() for t in scenes.cotangents(cpu)]
        ref = ref_harness.ref_tri_forward(s)
        rg = ref_harness.ref_tri_backward(s, ref, gc, gd)
        leaves = [s.verts.clone().requires_grad_(), s.verts_color.clone().requires_grad_(),
                  s.faces_opacity.clone().requires_grad_(), s.verts_depth.clone().requires_grad_(),
                  s.faces_intense.clone().requires_grad_()]
        color, depth = TriRenderer(TriRenderSettings(s.H, s.W, s.bg))(leaves[0], s.faces, leaves[1], leaves[2], s.mv_mats,
                                                                      s.proj_mats, leaves[3], leaves[4])
        torch.autograd.backward([color, depth], [gc, gd])
        assert (color - ref["color"]).abs().max().item() <= IMG_TOL
        for leaf, r in zip(leaves, rg):
            assert rel_l2(leaf.grad, r) <= GRAD_TOL
        R.append(ref["R"])
    assert R[1] > 1.25 * R[0] + 1024      # the second call really outgrew the speculative buffer


def test_fused_vertex_depth_matches_the_upstream_torch_computation():
    """verts_depth=None (SURVEY 8f-1): the renderer's own NDC z + its chain rule into the vertex positions must
    equal passing verts_depth = ndc_z(proj @ mv @ p) computed (and differentiated) upstream in PyTorch."""
    cpu = scenes.random_tri_scene("fd", 21, 3000, 0.07, 144, 176, B=3)
    s = scenes.to_device(cpu, "cuda")
    gc, gd = [t.cuda() for t in scenes.cotangents(cpu)]
    renderer = TriRenderer(TriRenderSettings(s.H, s.W, s.bg))

    def leaves():
        return [s.verts.clone().requires_grad_(), s.verts_color.clone().requires_grad_(),
                s.faces_opacity.clone().requires_grad_(), s.faces_intense.clone().requires_grad_()]

    # upstream: depth computed by the caller, gradient flows back through torch
    a = leaves()
    vh = torch.cat([a[0], torch.ones_like(a[0][:, :1])], dim=1)
    clip = torch.einsum("bij,bjk,pk->bpi", s.proj_mats, s.mv_mats, vh)
    vdepth = (clip[..., 2] / clip[..., 3]).contiguous()
    c0, d0 = renderer(a[0], s.faces, a[1], a[2], s.mv_mats, s.proj_mats, vdepth, a[3])
    torch.autograd.backward([c0, d0], [gc, gd])
    # fused
    b = leaves()
    c1, d1 = renderer(b[0], s.faces, b[1], b[2], s.mv_mats, s.proj_mats, None, b[3])
    torch.autograd.backward([c1, d1], [gc, gd])
    assert (c1 - c0).abs().max().item() <= IMG_TOL and (d1 - d0).abs().max().item() <= IMG_TOL
    for n, x, y in zip(("verts", "verts_color", "faces_opacity", "faces_intense"), b, a):
        e = rel_l2(x.grad, y.grad)
        assert e <= GRAD_TOL, "%s: rel L2 %.3e" % (n, e)
    # the depth term really contributes to the vertex gradient (the test would be vacuous otherwise)
    c = leaves()
    c2, d2 = renderer(c[0], s.faces, c[1], c[2], s.mv_mats, s.proj_mats, vdepth.detach(), c[3])
    torch.autograd.backward([c2, d2], [gc, gd])
    assert rel_l2(c[0].grad, a[0].grad) > 1e-3


@pytest.mark.parametrize("fused_depth", [False, True])
def test_direct_gradient_sink_equals_autograd_accumulation(fused_depth):
    """PackedSceneGrads.direct(): the backward kernels add into the packed .grad buffer themselves; the result must
    equal what autograd's own accumulation produces, across several calls per step (views_per_call) and with the
    fused vertex depth, and a call on other tensors must not be redirected."""
    from dmesh_renderer_b200.multiview import PackedSceneGrads, multiview_step
    cpu = scenes.random_tri_scene("sink", 33, 2500, 0.08, 128, 160, B=4)
    s = scenes.to_device(cpu, "cuda")
    gc, gd = [t.cuda() for t in scenes.cotangents(cpu)]
    renderer = TriRenderer(TriRenderSettings(s.H, s.W, s.bg))
    vd = None if fused_depth else s.verts_depth

    # plain autograd, all views in one call
    ref = [s.verts.clone().requires_grad_(), s.verts_color.clone().requires_grad_(), s.faces_opacity.clone().requires_grad_()]
    fi0 = s.faces_intense.clone().requires_grad_()
    c0, d0 = renderer(ref[0], s.faces, ref[1], ref[2], s.mv_mats, s.proj_mats, vd, fi0)
    torch.autograd.backward([c0, d0], [gc, gd])

    class Render:   # multiview_step slices verts_depth; None stays None
        def __call__(self, v, f, vc, fo, mv, pj, vdep, fint):
            return renderer(v, f, vc, fo, mv, pj, None if fused_depth else vdep, fint)

    g = PackedSceneGrads(s.verts.clone(), s.verts_color.clone(), s.faces_opacity.clone())
    fi1 = s.faces_intense.clone().requires_grad_()
    launches = []
    orig = _C.render_tris_backward

    def spy(*a, **k):
        launches.append(k.get("accumulate_into") is not None)
        return orig(*a, **k)
    _C.render_tris_backward = spy
    try:
        def cotangents(c, d):   # call i renders views 2i, 2i+1; its backward has not run yet
            first = 2 * len(launches)
            return gc[first:first + c.shape[0]], gd[first:first + c.shape[0]]
        multiview_step(Render(), g, s.faces, s.mv_mats, s.proj_mats, s.verts_depth, fi1, cotangents, views_per_call=2)
        assert launches == [True, True]
        for n, leaf, r in zip(("verts", "verts_color", "faces_opacity"), g.leaves, ref):
            assert rel_l2(leaf.grad, r.grad) <= GRAD_TOL, n
            assert leaf.grad.data_ptr() >= g.flat.data_ptr() and leaf.grad.data_ptr() < g.flat.data_ptr() + 4 * g.flat.numel()
        assert rel_l2(fi1.grad, fi0.grad) <= GRAD_TOL
        # tensors that are not the sink's leaves: ordinary autograd path even while the sink is active
        other = [t.detach().clone().requires_grad_() for t in ref]
        with g.direct():
            c2, d2 = renderer(other[0], s.faces, other[1], other[2], s.mv_mats, s.proj_mats, vd, s.faces_intense)
            torch.autograd.backward([c2, d2], [gc, gd])
        assert launches[-1] is False
        for o, r in zip(other, ref):
            assert rel_l2(o.grad, r.grad) <= GRAD_TOL
        assert not _C._grad_sinks
    finally:
        _C.render_tris_backward = orig


def _tri_grads(s, gc, gd, deterministic, sink=False):
    leaves = [s.verts.clone().requires_grad_(), s.verts_color.clone().requires_grad_(),
              s.faces_opacity.clone().requires_grad_(), s.verts_depth.clone().requires_grad_(),
              s.faces_intense.clone().requires_grad_()]
    renderer = TriRenderer(TriRenderSettings(s.H, s.W, s.bg), deterministic=deterministic)
    color, depth = renderer(leaves[0], s.faces, leaves[1], leaves[2], s.mv_mats, s.proj_mats, leaves[3], leaves[4])
    torch.autograd.backward([color, depth], [gc, gd])
    return [leaf.grad for leaf in leaves]


@pytest.mark.parametrize("name", ["small_tri", "C1", "C2", "mv4"])
def test_deterministic_backward_is_reproducible_and_matches(name):
    """SURVEY 8f-3: TriRenderer(..., deterministic=True) must give bit-identical gradients on every run (64-bit
    fixed-point accumulation) that agree with the reference extension within the gradient tolerance, for any scale
    of the cotangents (the fixed-point format is relative to max |dL_dout|)."""
    cpu = scenes.random_tri_scene("mv4", 44, 3000, 0.09, 160, 144, B=4) if name == "mv4" else scenes.config(name)
    s = scenes.to_device(cpu, "cuda")
    gc, gd = [t.cuda() for t in scenes.cotangents(cpu)]
    ref = ref_harness.ref_tri_forward(s)
    rg = ref_harness.ref_tri_backward(s, ref, gc, gd)
    names = ["verts", "verts_color", "faces_opacity", "verts_depth", "faces_intense"]
    runs = [_tri_grads(s, gc, gd, True) for _ in range(4)]
    for r in runs[1:]:
        for n, a, b in zip(names, runs[0], r):
            assert torch.equal(a, b), "%s differs between two deterministic runs" % n
    for n, a, r in zip(names, runs[0], rg):
        e = rel_l2(a, r)
        assert e <= GRAD_TOL, "%s: rel L2 %.3e" % (n, e)
    # linear in the cotangent, at any magnitude: powers of two scale exactly, so even the bits must follow -- from
    # max |cotangent| near 2^-80 to 2^100 (the binary point follows g down to 2^-112, det.cuh)
    for k in (2.0 ** -80, 2.0 ** -30, 2.0 ** 20, 2.0 ** 100):
        scaled = _tri_grads(s, gc * k, gd * k, True)
        for n, a, b in zip(names, runs[0], scaled):
            assert exactly_scaled(a, b, k), "%s: not exactly linear under cotangent scale %g" % (n, k)
    zero = _tri_grads(s, gc * 0, gd * 0, True)
    assert all(float(z.abs().max()) == 0.0 for z in zero)


def test_deterministic_mode_default_switch_and_gradient_sink():
    """set_deterministic() flips the process-wide default; the deterministic kernels also serve the direct gradient
    sink (PackedSceneGrads.direct) -- there the result is reproducible as long as the sink starts from the same values."""
    import dmesh_renderer_b200 as pkg
    from dmesh_renderer_b200.multiview import PackedSceneGrads
    cpu = scenes.random_tri_scene("detsink", 45, 2000, 0.1, 128, 128, B=2)
    s = scenes.to_device(cpu, "cuda")
    gc, gd = [t.cuda() for t in scenes.cotangents(cpu)]
    base = _tri_grads(s, gc, gd, True)
    old = pkg.set_deterministic(True)
    try:
        assert old is False
        again = _tri_grads(s, gc, gd, None)          # None -> process default
        for a, b in zip(base, again):
            assert torch.equal(a, b)
        outs = []
        for _ in range(2):
            g = PackedSceneGrads(s.verts.clone(), s.verts_color.clone(), s.faces_opacity.clone())
            r = TriRenderer(TriRenderSettings(s.H, s.W, s.bg))
            with g.direct():
                c, d = r(g.leaves[0], s.faces, g.leaves[1], g.leaves[2], s.mv_mats, s.proj_mats, s.verts_depth, s.faces_intense)
                torch.autograd.backward([c, d], [gc, gd])
            outs.append(g.flat.clone())
        assert torch.equal(outs[0], outs[1])
        for a, leaf in zip(base[:3], g.leaves):
            assert torch.equal(a, leaf.grad)          # 0 + x == x
    finally:
        pkg.set_deterministic(old)


def test_speculative_phase2_when_the_scene_vanishes_and_two_calls_in_flight():
    """Round-2 host logic on the GPU: (1) a call whose instance count drops to ZERO while phase 2 was launched
    speculatively on a buffer sized from the previous call must give the background image and zero gradients;
    (2) two forward calls between their two phases own separate pinned num_rendered words (ADVICE r1): finishing
    them in the opposite order must give each its own result."""
    dev = "cuda"
    a = scenes.to_device(scenes.random_tri_scene("inflight_a", 51, 3000, 0.08, 128, 160, B=2), dev)
    b = scenes.to_device(scenes.random_tri_scene("inflight_b", 52, 3000, 0.03, 128, 160, B=2), dev)   # same shapes, fewer instances
    renderer = TriRenderer(TriRenderSettings(a.H, a.W, a.bg))
    # (1)
    leaves = [a.verts.clone().requires_grad_(), a.verts_color.clone().requires_grad_(), a.faces_opacity.clone().requires_grad_()]
    c0, d0 = renderer(leaves[0], a.faces, leaves[1], leaves[2], a.mv_mats, a.proj_mats, a.verts_depth, a.faces_intense)
    far = (a.verts * 0.01 + torch.tensor([3.0, 2.0, 10.0], device=dev) * 3).requires_grad_()      # behind the camera
    c1, d1 = renderer(far, a.faces, leaves[1], leaves[2], a.mv_mats, a.proj_mats, a.verts_depth, a.faces_intense)
    assert torch.equal(c1, torch.ones_like(c1)) and torch.equal(d1, torch.ones_like(d1))
    torch.autograd.backward([c1, d1], [torch.ones_like(c1), torch.ones_like(d1)])
    assert float(far.grad.abs().max()) == 0.0 and float(leaves[1].grad.abs().max()) == 0.0
    c2, d2 = renderer(leaves[0], a.faces, leaves[1], leaves[2], a.mv_mats, a.proj_mats, a.verts_depth, a.faces_intense)
    assert torch.equal(c2, c0) and torch.equal(d2, d0)       # and the next call grows back past the zero capacity
    # (2)
    def args(s):
        mv, pj = s.mv_mats.transpose(1, 2), s.proj_mats.transpose(1, 2)
        return (s.bg, s.verts, s.faces, s.verts_color, s.faces_opacity, mv, pj), (torch.inverse(mv), torch.inverse(pj)), \
               (s.verts_depth, s.faces_intense, s.H, s.W)
    outs = {}
    for name, s in (("a", a), ("b", b)):
        x, inv, y = args(s)
        outs[name] = _C.render_tris(*x, *inv, *y)
    xa, ia, ya = args(a)
    xb, ib, yb = args(b)
    pa = _C.tri_forward_begin(*xa, *ya)
    pb = _C.tri_forward_begin(*xb, *yb)
    assert pa.pinned is not pb.pinned and pa.pinned[2].value != pb.pinned[2].value
    rb = _C.tri_forward_finish(pb, *ib)
    ra = _C.tri_forward_finish(pa, *ia)
    assert ra[0] == outs["a"][0] and rb[0] == outs["b"][0] and ra[0] != rb[0]
    assert torch.equal(ra[1], outs["a"][1]) and torch.equal(rb[1], outs["b"][1])
    assert torch.equal(ra[2], outs["a"][2]) and torch.equal(rb[2], outs["b"][2])
