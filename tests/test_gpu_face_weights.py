"""Tri and tet renderers: per-(view, face) visibility statistics of the forward pass (return_face_weights=True).

face_weights[b, f] = sum over the pixels of view b where face f was composited of the blending weight T * alpha (the
factor the face's colour is multiplied by); face_hits[b, f] = the number of those pixels.  Yardsticks:
  * an fp64 scatter-add over the CPU oracle's fragments (tests/tri_fragments.py, tests/tet_fragments.py): hits bit for
    bit, weights <= 1e-5 relative L2;
  * sum over faces = alpha.sum() per view, without any reference;
  * dL/dfaces_intense of a render with white colours and the cotangent (1, 0, 0) on colour, 0 on depth;
  * reproducibility and bit-identical images and gradients with the switch on.
"""
import numpy as np
import pytest
import torch

from dmesh_renderer_b200 import TetRenderer, TetRenderSettings, TriRenderer, TriRenderSettings, _C, _lib, scenes
from test_gpu_tet_camera_grads import CASES as TET_CASES, SCENES as TET_SCENES, _stages, gpu_forward, trail_cap
from test_gpu_tet_camera_grads import oracle_fragments as tet_oracle_fragments
from test_gpu_tri_camera_grads import SCENES as TRI_SCENES, oracle_fragments as tri_oracle_fragments, rel_l2
from test_gpu_vs_oracle_and_golden import edge_scene
import tet_meshes
from test_face_weights_reference import scatter_reference

pytestmark = pytest.mark.gpu
f64 = torch.float64
W_TOL = 1e-5
TRI_ALL = dict(TRI_SCENES, edge=edge_scene)
TET_ALL = dict(TET_CASES, inside=("inside", 0, 0))
TET_BUILD = dict(TET_SCENES, inside=lambda: tet_meshes.delaunay_tet_scene("inside", 21, 400, 61, 83, 2, cameras="inside"))


# ---------------------------------------------------------------------------------------------- tri
def tri_run(cpu, det=False, alpha=True, grads=False, renderer_kw=None, fused=False):
    s = scenes.to_device(cpu, "cuda")
    leaves = [t.clone().requires_grad_(grads) for t in (s.verts, s.verts_color, s.faces_opacity, s.faces_intense)]
    out = TriRenderer(TriRenderSettings(s.H, s.W, s.bg), deterministic=det, return_alpha=alpha, **(renderer_kw or {}))(
        leaves[0], s.faces, leaves[1], leaves[2], s.mv_mats, s.proj_mats, None if fused else s.verts_depth, leaves[3])
    return out, leaves


def tri_stats(cpu, det=False):
    out, _ = tri_run(cpu, det=det, renderer_kw=dict(return_face_weights=True))
    return out[2], out[3], out[4]       # alpha, face_weights, face_hits


@pytest.mark.parametrize("name", list(TRI_ALL))
def test_tri_matches_oracle_fragments(name):
    cpu = TRI_ALL[name]()
    (counts, face, _), _ = tri_oracle_fragments(cpu)
    B, F = cpu.mv_mats.shape[0], cpu.faces.shape[0]
    pix_view = np.repeat(np.arange(B), cpu.H * cpu.W)
    rw, rh = scatter_reference(B, F, pix_view, counts.reshape(-1), face,
                               cpu.faces_opacity.to(f64)[torch.from_numpy(face.astype(np.int64))])
    alpha, fw, fh = tri_stats(cpu)
    assert fw.dtype == torch.float32 and fh.dtype == torch.int32 and tuple(fw.shape) == (B, F)
    assert torch.equal(fh.cpu().long(), rh)
    e = rel_l2(fw.cpu().numpy(), rw.numpy())
    assert e <= W_TOL, "face_weights rel L2 %.3e" % e
    assert rh.sum() > 0


def _identity(alpha, fw):
    a = alpha.double().sum((1, 2, 3))
    s = fw.double().sum(1)
    return ((s - a).abs() / a.clamp_min(1e-30)).max().item()


@pytest.mark.parametrize("name", ["small_tri", "C1", "cam4", "C2", "C4x8"])
def test_tri_weights_sum_to_alpha(name):
    cpu = scenes.config("C4", views=64, view_slice=slice(0, 8)) if name == "C4x8" else \
        TRI_ALL[name]() if name in TRI_ALL else scenes.config(name)
    alpha, fw, fh = tri_stats(cpu)
    assert _identity(alpha, fw) <= 1e-5
    assert ((fh > 0) | (fw == 0)).all()


@pytest.mark.parametrize("name", ["small_tri", "cam4", "edge"])
def test_tri_weights_equal_intensity_gradient_of_a_white_render(name):
    cpu = TRI_ALL[name]()
    _, fw, _ = tri_stats(cpu)
    white = cpu._replace(verts_color=torch.ones_like(cpu.verts_color))
    out, leaves = tri_run(white, alpha=False, grads=True)
    gc = torch.zeros_like(out[0])
    gc[:, 0] = 1
    torch.autograd.backward([out[0], out[1]], [gc, torch.zeros_like(out[1])])
    # the colour of a hit is intense * interp(colour) = intense: d colour / d intense = T * alpha.  The backward walk
    # recovers T by dividing by (1 - alpha) face by face, which loses more than the forward's product on the edge
    # scene's grazing triangles (measured 3.9e-5 there; the fragment test holds face_weights to 1e-5 of fp64)
    e = rel_l2(fw.cpu().numpy(), leaves[3].grad.cpu().numpy())
    assert e <= (1e-4 if name == "edge" else W_TOL), e


@pytest.mark.parametrize("deterministic", [False, True], ids=["default", "det"])
def test_tri_reproducible(deterministic):
    cpu = TRI_ALL["cam4"]()
    runs = [tri_stats(cpu, det=deterministic) for _ in range(3)]
    for r in runs[1:]:
        assert torch.equal(r[1], runs[0][1]) and torch.equal(r[2], runs[0][2])


def test_tri_speculative_rerun_counts_once():
    """A phase 2 that ran on a too-small speculative binning buffer and was repeated gives the statistics of a call
    that ran once."""
    cpu = TRI_ALL["C1"]()
    _C._last_R.clear()
    ref = tri_stats(cpu)
    # same shapes, a scene that binned into far fewer instances: the next call's speculative buffer is too small
    centre = cpu.verts.mean(0, keepdim=True)
    tiny = cpu._replace(verts=centre + (cpu.verts - centre) * 1e-3)
    tri_stats(tiny)
    key = [k for k in _C._last_R if k[0] == "tri"]
    small_R = max(_C._last_R[k] for k in key)
    again = tri_stats(cpu)
    assert max(_C._last_R[k] for k in key) > small_R + small_R // 4 + 1024   # phase 2 did run twice
    assert torch.equal(again[1], ref[1]) and torch.equal(again[2], ref[2])


@pytest.mark.parametrize("deterministic", [False, True], ids=["default", "det"])
@pytest.mark.parametrize("fused", [False, True], ids=["explicit_depth", "fused_depth"])
def test_tri_images_and_gradients_unchanged(fused, deterministic):
    cpu = TRI_ALL["cam4"]()
    gc, gd = scenes.cotangents(cpu)
    res = []
    for on in (False, True):
        out, leaves = tri_run(cpu, det=deterministic, grads=True, fused=fused, renderer_kw=dict(return_face_weights=on))
        torch.autograd.backward([out[0], out[1], out[2]], [gc.cuda(), gd.cuda(), gd.cuda() * 0.5])
        res.append([o.detach() for o in out[:3]] + [l.grad for l in leaves])
    for a, b in zip(*res):
        if deterministic or a.dim() == 4:          # default mode: gradients carry float-atomic noise run to run
            assert torch.equal(a, b)
        else:
            assert rel_l2(a.cpu().numpy(), b.cpu().numpy()) <= 1e-6


def test_tri_empty_scenes_give_zeros():
    cpu = TRI_ALL["tiny_tri"]()
    B, F = cpu.mv_mats.shape[0], cpu.faces.shape[0]
    # nothing on screen: every triangle collapsed to one point
    _, fw, fh = tri_stats(cpu._replace(verts=torch.zeros_like(cpu.verts)))
    assert not fw.any() and not fh.any() and tuple(fw.shape) == (B, F)
    # P == 0: zero images, zero statistics
    s = scenes.to_device(cpu, "cuda")
    out = TriRenderer(TriRenderSettings(s.H, s.W, s.bg), return_face_weights=True)(
        s.verts[:0], s.faces, s.verts_color[:0], s.faces_opacity, s.mv_mats, s.proj_mats, s.verts_depth[:, :0],
        s.faces_intense)
    assert len(out) == 4 and tuple(out[2].shape) == (B, F) and not out[2].any() and not out[3].any()


# ---------------------------------------------------------------------------------------------- tet
def tet_run(cpu, seed=0, det=False, stats=True, grads=False, intensity=False, alpha=True):
    s = scenes.to_device(cpu, "cuda")
    vc, fo = s.verts_color.clone().requires_grad_(grads), s.faces_opacity.clone().requires_grad_(grads)
    fi = s.faces_intense.clone().requires_grad_(intensity)
    out = TetRenderer(TetRenderSettings(s.H, s.W, s.bg, seed), deterministic=det, intensity_grads=intensity,
                      return_alpha=alpha, return_face_weights=stats)(
        s.verts, s.faces, vc, fo, s.mv_mats, s.proj_mats, s.verts_depth, fi, s.tets, s.face_tets, s.tet_faces)
    return out, (vc, fo, fi)


_tet_refs = {}


def tet_reference(case):
    """(cpu, fp64 weights, hits, parted pixels, all steps walked by the backward pass)."""
    if case not in _tet_refs:
        name, seed, _cap = TET_ALL[case]
        cpu = TET_BUILD[name]()
        fwd = gpu_forward(cpu, seed)
        frags, o = tet_oracle_fragments(cpu, fwd["coords"])
        assert o["mismatch"] == 0
        B, F, HW = cpu.mv_mats.shape[0], cpu.faces.shape[0], cpu.H * cpu.W
        parted = (fwd["first_face"] != o["first_face"]) | (fwd["n_contrib"] != frags["counts"]) | \
            (np.abs(fwd["color"] - o["color"]).max(1).reshape(-1) > 1e-5)
        counts = frags["counts"].astype(np.int64) * frags["active"]      # inactive pixels contribute nothing
        keep = np.repeat(frags["active"], frags["counts"].astype(np.int64))
        face, reach = frags["face"][keep], frags["reach"][keep]
        rw, rh = scatter_reference(B, F, np.arange(B * HW) // HW, counts, face,
                                   cpu.faces_opacity.to(f64)[torch.from_numpy(face.astype(np.int64))])
        # steps of the parted pixels on either side: at most this many (view, face) entries may differ; the entries the
        # parted pixels touch on the oracle's side are left out of the weight comparison
        slack = int(counts[parted].sum() + fwd["n_contrib"][parted].astype(np.int64).sum())
        pf = np.repeat(parted & frags["active"], counts)
        touched = np.zeros(B * F, bool)
        touched[(np.repeat(np.arange(B * HW) // HW, counts) * F + face)[pf]] = True
        _tet_refs[case] = (cpu, rw, rh, (slack, torch.from_numpy(touched).view(B, F)), bool(reach.all()), frags)
    return _tet_refs[case]


@pytest.mark.parametrize("deterministic", [False, True], ids=["default", "det"])
@pytest.mark.parametrize("case", list(TET_ALL))
def test_tet_matches_oracle_fragments(case, deterministic):
    name, seed, cap = TET_ALL[case]
    cpu, rw, rh, (slack, touched), _, frags = tet_reference(case)
    with trail_cap(cap):
        out, _ = tet_run(cpu, seed=seed, det=deterministic)
        torch.cuda.synchronize()
    alpha, fw, fh = out[3], out[4].cpu(), out[5].cpu()
    ok = fh.long() == rh
    assert int((~ok).sum()) <= slack, (int((~ok).sum()), slack)
    ok &= ~touched
    e = rel_l2(fw[ok].numpy(), rw[ok].numpy())
    assert e <= W_TOL, "face_weights rel L2 %.3e" % e
    assert _identity(alpha, out[4]) <= 1e-5


@pytest.mark.parametrize("case", list(TET_ALL))
def test_tet_weights_equal_intensity_gradient_of_a_white_render(case):
    name, seed, cap = TET_ALL[case]
    cpu, _, _, _, all_walked, _ = tet_reference(case)
    if not all_walked:
        pytest.skip("the reverse march gives up on some steps here: dL/dfaces_intense leaves them out")
    with trail_cap(cap):
        fw = tet_run(cpu, seed=seed)[0][4]
        white = cpu._replace(verts_color=torch.ones_like(cpu.verts_color))
        out, leaves = tet_run(white, seed=seed, stats=False, alpha=False, intensity=True)
        gc = torch.zeros_like(out[0])
        gc[:, 0] = 1
        torch.autograd.backward([out[0], out[1]], [gc, torch.zeros_like(out[1])])
    # the backward walk forms T by its own reverse recurrence (prev_log_T -= log1m), which parts from the forward's
    # by a little more than 1e-5 over the long rays of a camera inside the mesh (measured 1.1e-5)
    e = rel_l2(fw.cpu().numpy(), leaves[2].grad.cpu().numpy())
    assert e <= (2e-5 if case == "inside" else W_TOL), e


@pytest.mark.parametrize("deterministic", [False, True], ids=["default", "det"])
def test_tet_reproducible_and_trail_cap(deterministic):
    cpu = TET_BUILD["small_tet"]()
    runs = [tet_run(cpu, det=deterministic)[0] for _ in range(3)]
    for r in runs[1:]:
        assert torch.equal(r[4], runs[0][4]) and torch.equal(r[5], runs[0][5])
    with trail_cap(3):
        short = tet_run(cpu, det=deterministic)[0]
    # steps beyond a short trail are marched again with the forward's own arithmetic: the same bits
    assert torch.equal(short[5], runs[0][5]) and torch.equal(short[4], runs[0][4])


@pytest.mark.parametrize("name", ["C3"])
def test_tet_weights_sum_to_alpha_C3(name):
    out, _ = tet_run(scenes.config(name))
    assert _identity(out[3], out[4]) <= 1e-5


@pytest.mark.parametrize("deterministic", [False, True], ids=["default", "det"])
def test_tet_images_and_gradients_unchanged(deterministic):
    cpu = TET_BUILD["small_tet"]()
    gc, gd = scenes.cotangents(cpu)
    res = []
    for on in (False, True):
        out, leaves = tet_run(cpu, seed=7, det=deterministic, stats=on, grads=True, intensity=True)
        torch.autograd.backward([out[0], out[1], out[3]], [gc.cuda(), gd.cuda(), gd.cuda() * 0.5])
        res.append([out[0].detach(), out[1].detach(), out[2], out[3].detach()] + [l.grad for l in leaves])
    for i, (a, b) in enumerate(zip(*res)):
        if deterministic or i < 4:                 # default mode: gradients carry float-atomic noise run to run
            assert torch.equal(a, b)
        else:
            assert rel_l2(a.cpu().numpy(), b.cpu().numpy()) <= 1e-6


def test_tet_nothing_on_screen_gives_zeros():
    cpu = TET_BUILD["tiny_tet"]()
    out, _ = tet_run(cpu._replace(verts=torch.zeros_like(cpu.verts)))
    assert not out[4].any() and not out[5].any()


def test_tri_no_faces_renders_as_without_statistics():
    """Vertices but no faces (every face pruned): the images, alpha and dL/dbg are those of the switch off, and the
    statistics are [B,0]."""
    cpu = TRI_ALL["tiny_tri"]()
    s = scenes.to_device(cpu, "cuda")
    B = s.mv_mats.shape[0]
    gc, gd = [t.cuda() for t in scenes.cotangents(cpu)]
    res = []
    for on in (False, True):
        bg = (s.bg * 0.5 + 0.25).detach().clone().requires_grad_()
        out = TriRenderer(TriRenderSettings(s.H, s.W, bg), return_alpha=True, return_face_weights=on)(
            s.verts, s.faces[:0], s.verts_color, s.faces_opacity[:0], s.mv_mats, s.proj_mats, s.verts_depth,
            s.faces_intense[:, :0])
        torch.autograd.backward([out[0], out[1], out[2]], [gc, gd, gd * 0.5])
        res.append([o.detach() for o in out[:3]] + [bg.grad])
        if on:
            assert tuple(out[3].shape) == (B, 0) and tuple(out[4].shape) == (B, 0)
    for a, b in zip(*res):
        assert torch.equal(a, b)
    assert torch.equal(res[0][0], s.bg.view(1, 3, 1, 1).expand_as(res[0][0]) * 0.5 + 0.25)   # the background


def _forward_launches_and_stages(fn):
    """Kernel launches and profile stages of one call of fn (after a warm-up call with the same shapes)."""
    lib = _lib.load()
    fn()
    torch.cuda.synchronize()
    _lib.check(lib.dmr_profile_enable(1))
    try:
        _stages()
        n0 = lib.dmr_launch_count()
        fn()
        n1 = lib.dmr_launch_count()
        torch.cuda.synchronize()
        return n1 - n0, _stages()
    finally:
        _lib.check(lib.dmr_profile_enable(0))


def test_switch_off_launches_and_stages():
    """With the switch off the forward calls make no statistics launch and record no statistics stage; with it on they
    make exactly one more launch (tri: the conversion; its forward kernel replaces the plain one) or two (tet: the
    post-pass and the conversion) under a stage of their own."""
    tri = TRI_ALL["cam4"]()
    ts = scenes.to_device(tri, "cuda")
    tet = TET_BUILD["small_tet"]()
    es = scenes.to_device(tet, "cuda")
    tri_call = lambda on: lambda: TriRenderer(TriRenderSettings(ts.H, ts.W, ts.bg), return_face_weights=on)(
        ts.verts, ts.faces, ts.verts_color, ts.faces_opacity, ts.mv_mats, ts.proj_mats, ts.verts_depth, ts.faces_intense)
    tet_call = lambda on: lambda: TetRenderer(TetRenderSettings(es.H, es.W, es.bg, 0), return_face_weights=on)(
        es.verts, es.faces, es.verts_color, es.faces_opacity, es.mv_mats, es.proj_mats, es.verts_depth,
        es.faces_intense, es.tets, es.face_tets, es.tet_faces)
    for call, stage, extra in ((tri_call, "tri_face_weights", 1), (tet_call, "tet_face_weights", 2)):
        n_off, st_off = _forward_launches_and_stages(call(False))
        n_on, st_on = _forward_launches_and_stages(call(True))
        assert not (st_off & {"tri_face_weights", "tet_face_weights"})
        assert st_on == st_off | {stage}
        assert n_on == n_off + extra


def test_stages_and_argument_checks():
    lib = _lib.load()
    names = [lib.dmr_profile_stage_name(i).decode() for i in range(lib.dmr_profile_stage_count())]
    assert names[-2:] == ["tri_face_weights", "tet_face_weights"]
    assert lib.dmr_tri_face_weights_bytes(3, 5) == 180 and lib.dmr_tet_face_weights_bytes(2, 7) == 168
    # a missing or too small workspace is refused before anything is enqueued
    null, some = _C.ctypes.c_void_p(0), _C.ctypes.c_void_p(256)
    assert lib.dmr_tet_face_weights(1, 4, 4, 1, 8, 8, 0, *([some] * 8), null, 0, null) != 0
    assert b"workspace" in lib.dmr_last_error()
    assert lib.dmr_tri_forward_render_face_weights(1, 4, 4, 8, 8, 0, *([some] * 11), some, 47, null) != 0
    assert b"workspace" in lib.dmr_last_error()
