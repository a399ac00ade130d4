"""GPU: the tet renderer on Delaunay meshes with tables in arbitrary order, and with cameras inside the mesh.

The scenes (tests/tet_meshes.py) reach what the Kuhn grids of the other tet tests never do: all 24 (side, vertex
order) codes of the adjacency records, the -1 of a boundary face in column 0 of face_tets, faces straddling the camera
plane (the preprocessing's "no pixel bounding box" fallback, and the first-intersection search over faces whose depth
range comes from vertices behind the camera), a vertex exactly in the camera plane, and image sizes that leave partial
8x8 march CTAs (and partial 16x16 tiles) on both edges.  Nothing is recorded: every comparison is with the CPU oracle
(or its fragments, for jittered rays and the fp64 references) on the same scene at run time.

  * binning integers, first_face / first_tet, n_contrib, active mask: bit-exact; images <= 1e-5 max-abs
  * colour and opacity gradients: <= 1e-4 relative L2 against TetOracle.backward
  * camera and vertex gradients: <= 1e-3, intensity gradients <= 1e-4, against the fp64 fragment reference
"""
import numpy as np
import pytest
import torch

import binning_checks
import tet_fragments
import tet_meshes
from dmesh_renderer_b200 import TetRenderer, TetRenderSettings, _C, _lib, debug, scenes
from test_gpu_tet_camera_grads import MAX_PARTED, rel_l2, trail_cap
from test_gpu_vs_oracle_and_golden import dev_mats, oracle, run_tet
from test_tet_vertex_grads_reference import reference_grads_verts, rigid_residual

pytestmark = pytest.mark.gpu

IMG_TOL, GRAD_TOL, CAM_TOL, VERT_TOL, INT_TOL = 1e-5, 1e-4, 1e-3, 1e-3, 1e-4
H, W = 61, 83
BUILD = {
    "outside": lambda: tet_meshes.delaunay_tet_scene("outside", 21, 400, H, W, 2, cameras="outside"),
    "canonical": lambda: tet_meshes.delaunay_tet_scene("canonical", 21, 400, H, W, 2, cameras="outside", shuffle=False),
    "inside": lambda: tet_meshes.delaunay_tet_scene("inside", 21, 400, H, W, 2, cameras="inside"),
    "on_plane": lambda: tet_meshes.delaunay_tet_scene("on_plane", 21, 400, H, W, 3, cameras="on_plane"),
    # tile lists of up to ~5800 faces: many first-intersection rounds of 256
    "mid_inside": lambda: tet_meshes.delaunay_tet_scene("mid_inside", 22, 6000, 161, 203, 2, cameras="inside"),
}
SMALL = ["outside", "canonical", "inside", "on_plane"]

_cases = {}


def case(name):
    """(cpu scene, cuda scene, device matrices [mv, proj, inv_mv, inv_proj], oracle, oracle outputs), built once: the
    oracle gets the matrices the GPU gets, inverses included."""
    if name not in _cases:
        cpu = BUILD[name]()
        s = scenes.to_device(cpu, "cuda")
        mats = dev_mats(s)
        o = oracle.TetOracle(cpu, mats=[m.contiguous().cpu().numpy() for m in mats])   # torch.inverse: column-major
        _cases[name] = (cpu, s, mats, o, o.outputs())
    return _cases[name]


def dims(s, R=0):
    return dict(B=s.mv_mats.shape[0], P=s.verts.shape[0], F=s.faces.shape[0], W=s.W, H=s.H, R=R, T=s.tets.shape[0])


# ---------------------------------------------------------------------------------------------- forward parity
@pytest.mark.parametrize("name", list(BUILD))
def test_forward_matches_oracle(name):
    cpu, s, mats, o, ref = case(name)
    (color, depth, active, pb, fb, bb, ib), _ = run_tet(s, mats)
    d = dims(s, ref["R"])
    tt = debug.view("tet", "tiles_touched", fb, **d)
    np.testing.assert_array_equal(tt, ref["tiles_touched"])
    live = tt > 0
    dk = debug.view("tet", "depth_keys", fb, **d)
    np.testing.assert_array_equal(dk[live], ref["depth_keys"][live])
    binning_checks.check_face_order_and_offsets(debug.view("tet", "face_order", fb, **d), dk, tt,
                                                debug.view("tet", "offsets", fb, **d), ref["offsets"])
    np.testing.assert_array_equal(debug.view("tet", "keys_sorted", bb, face_buffer=fb, **d), ref["keys_sorted"])
    np.testing.assert_array_equal(debug.view("tet", "values_sorted", bb, **d), ref["values_sorted"])
    np.testing.assert_array_equal(debug.view("tet", "ranges", ib, **d), ref["ranges"])
    np.testing.assert_array_equal(debug.view("tet", "first_face", ib, **d), ref["first_face"])
    np.testing.assert_array_equal(debug.view("tet", "first_tet", ib, **d), ref["first_tet"])
    np.testing.assert_array_equal(debug.view("tet", "n_contrib", ib, **d), ref["n_contrib"])
    assert np.array_equal(active.cpu().numpy() > 0.5, ref["active"] > 0.5)
    assert np.abs(color.cpu().numpy() - ref["color"]).max() <= IMG_TOL
    assert np.abs(depth.cpu().numpy() - ref["depth"]).max() <= IMG_TOL
    assert (ref["active"] > 0.5).mean() > 0.3
    if name == "mid_inside":                              # several rounds of the face-parallel first intersection
        r = ref["ranges"].astype(np.int64)
        assert (r[:, 1] - r[:, 0]).max() > 4 * 256


@pytest.mark.parametrize("split", [1, 2, 3])
@pytest.mark.parametrize("name", ["inside", "on_plane"])
def test_first_intersection_split_matches_oracle(name, split):
    """Split mode: several CTAs per tile meet in a per-pixel atomicMin and close each other's search with the
    smallest max depth of any hit (fi_close) -- here with depth ranges that come from vertices behind the camera."""
    cpu, s, mats, o, ref = case(name)
    lib = _lib.load()
    lib.dmr_debug_set_tet_first_split(split)
    try:
        out, _ = run_tet(s, mats)
        torch.cuda.synchronize()
    finally:
        lib.dmr_debug_set_tet_first_split(0)
    d = dims(s, ref["R"])
    np.testing.assert_array_equal(debug.view("tet", "first_face", out[6], **d), ref["first_face"])
    np.testing.assert_array_equal(debug.view("tet", "first_tet", out[6], **d), ref["first_tet"])
    np.testing.assert_array_equal(debug.view("tet", "n_contrib", out[6], **d), ref["n_contrib"])


# ---------------------------------------------------------------------------------------------- colour, opacity
@pytest.mark.parametrize("cap", [0, 3], ids=["auto_trail", "trail3"])
@pytest.mark.parametrize("deterministic", [False, True], ids=["default", "det"])
@pytest.mark.parametrize("name", SMALL)
def test_gradients_match_oracle(name, deterministic, cap):
    """trail_cap(3): the steps beyond the third face of a ray are re-marched through the adjacency records in the
    backward pass, i.e. through the decoded side codes once more."""
    cpu, s, mats, o, ref = case(name)
    gc, gd = [t.cuda() for t in scenes.cotangents(cpu)]
    og = o.backward(gc.cpu(), gd.cpu())

    def grads():
        out, _ = run_tet(s, mats)
        g = _C.render_tets_backward(s.bg, s.verts, s.faces, s.verts_color, s.faces_opacity, *mats, s.verts_depth,
                                    s.faces_intense, s.tets, s.face_tets, s.tet_faces, gc, gd, *out[3:], 0,
                                    deterministic=deterministic)
        torch.cuda.synchronize()
        assert np.abs(out[0].cpu().numpy() - ref["color"]).max() <= IMG_TOL
        return [x.clone() for x in g[:2]]

    with trail_cap(cap):
        runs = [grads() for _ in range(2 if deterministic else 1)]
    if deterministic:
        assert torch.equal(runs[0][0], runs[1][0]) and torch.equal(runs[0][1], runs[1][1])
    assert (ref["n_contrib"] > 3).mean() > 0.2                 # the trail cap bites on many rays
    for n, g, r in (("verts_color", runs[0][0], og[0]), ("faces_opacity", runs[0][1], og[1])):
        e = rel_l2(g.cpu().numpy(), r)
        assert e <= GRAD_TOL, "%s: rel L2 %.3e" % (n, e)


# ---------------------------------------------------------------------------------------------- jittered rays
def fragments(name, seed):
    """GPU forward with ray_random_seed `seed`, the oracle's fragments on the GPU's own pixel coordinates, and the
    pixels whose march parts from the oracle's (fp-level ties of a grazing ray)."""
    cpu, s, mats, o, ref = case(name)
    out, _ = run_tet(s, mats, seed=seed)
    d = dims(s)
    fw = dict(color=out[0].cpu().numpy(), depth=out[1].cpu().numpy(), active=out[2].cpu().numpy().reshape(-1) > 0.5,
              first_face=debug.view("tet", "first_face", out[6], **d),
              n_contrib=debug.view("tet", "n_contrib", out[6], **d),
              coords=debug.view("tet", "tet_jitter", out[6], **d).copy() if seed > 0 else None)
    frags, fo = tet_fragments.tet_fragments(cpu, [m.cpu().numpy() for m in mats], fw["coords"])
    assert fo["mismatch"] == 0
    parted = (fw["first_face"] != fo["first_face"]) | (fw["n_contrib"] != frags["counts"]) | \
        (np.abs(fw["color"] - fo["color"]).max(1).reshape(-1) > IMG_TOL) | \
        (np.abs(fw["depth"] - fo["depth"]).reshape(-1) > IMG_TOL)
    return cpu, fw, frags, fo, parted


@pytest.mark.parametrize("name", ["outside", "inside"])
def test_jittered_rays_match_oracle_fragments(name):
    cpu, fw, frags, fo, parted = fragments(name, 7)
    print("\n[tet general meshes] %s, ray_random_seed 7: %d pixel(s) parted from the oracle's march" % (
        name, int(parted.sum())))
    assert fw["coords"] is not None and not np.array_equal(fw["coords"] % 1.0, np.full_like(fw["coords"], 0.5))
    assert parted.sum() <= MAX_PARTED
    assert np.array_equal(fw["active"][~parted], frags["active"][~parted])
    assert frags["active"].mean() > 0.3


# ---------------------------------------------------------------------------------------------- fp64 references
_refs = {}


def reference_for(name):
    """Cotangents zero at pixels whose GPU march parts from the oracle's, and the fp64 fragment reference."""
    if name not in _refs:
        cpu, fw, frags, fo, parted = fragments(name, 0)
        assert parted.sum() <= MAX_PARTED, parted.sum()
        gc, gd = scenes.cotangents(cpu)
        B = gd.shape[0]
        keep = torch.from_numpy(~parted).view(B, 1, H, W).float()
        gc, gd = gc * keep, gd * keep
        _refs[name] = (cpu, gc, gd, frags, torch.from_numpy(~parted).view(B, H, W),
                       reference_grads_verts(cpu, frags, gc, gd))
        print("\n[tet general meshes] %s: %d pixel(s) parted from the oracle's march" % (name, int(parted.sum())))
    return _refs[name]


def gpu_grads(cpu, gc, gd, deterministic, vertex=True, intensity=True, camera=True):
    s = scenes.to_device(cpu, "cuda")
    v = s.verts.clone().requires_grad_(vertex)
    mv = s.mv_mats.clone().requires_grad_(camera)
    pj = s.proj_mats.clone().requires_grad_(camera)
    vc, fo = s.verts_color.clone().requires_grad_(), s.faces_opacity.clone().requires_grad_()
    fi = s.faces_intense.clone().requires_grad_(intensity)
    color, depth, active = TetRenderer(TetRenderSettings(s.H, s.W, s.bg, 0), deterministic=deterministic,
                                       vertex_grads=vertex, intensity_grads=intensity)(
        v, s.faces, vc, fo, mv, pj, s.verts_depth, fi, s.tets, s.face_tets, s.tet_faces)
    torch.autograd.backward([color, depth], [gc.cuda(), gd.cuda()])
    torch.cuda.synchronize()
    return color.detach().cpu(), depth.detach().cpu(), active.cpu(), dict(
        verts=v.grad, verts_color=vc.grad, faces_opacity=fo.grad, mv_mats=mv.grad, proj_mats=pj.grad,
        faces_intense=fi.grad)


@pytest.mark.parametrize("combo", ["camera", "all"])
@pytest.mark.parametrize("deterministic", [False, True], ids=["default", "det"])
@pytest.mark.parametrize("name", ["outside", "inside", "on_plane"])
def test_extension_gradients_match_fp64_reference(name, deterministic, combo):
    """Camera gradients alone, and camera + vertex + intensity gradients in one backward pass (another instantiation
    of the backward march)."""
    cpu, gc, gd, frags, same, (rc, rdp, rg, grazing) = reference_for(name)
    everything = combo == "all"
    color, depth, active, g = gpu_grads(cpu, gc, gd, deterministic, vertex=everything, intensity=everything)
    act = torch.from_numpy(frags["active"]).view(active.shape)
    assert torch.equal(active[same], act[same])
    m = (act & same)[:, None]
    # the reference reproduces the GPU's images and its colour and opacity gradients
    assert (color.double() - rc).abs().masked_select(m).max().item() <= 1e-4
    assert (depth.double() - rdp).abs().masked_select(m).max().item() <= 1e-4
    for k in ("verts_color", "faces_opacity"):
        assert rel_l2(g[k].cpu().numpy(), rg[k].numpy()) <= GRAD_TOL, k
    B = cpu.mv_mats.shape[0]
    errs = {k: [rel_l2(g[k][b].cpu().numpy(), rg[k][b].numpy()) for b in range(B)] for k in ("mv_mats", "proj_mats")}
    msg = "mv %.2e proj %.2e" % (max(errs["mv_mats"]), max(errs["proj_mats"]))
    for k in errs:
        assert max(errs[k]) <= CAM_TOL, (k, errs[k])
    if everything:
        gv, rv = g["verts"].cpu().numpy(), rg["verts"].numpy()
        # vertices of faces walked at a grazing angle are left out on both sides (test_gpu_tet_vertex_grads.py)
        keep = np.ones(gv.shape[0], bool)
        keep[cpu.faces.long()[grazing].reshape(-1).numpy()] = False
        ev = rel_l2(gv[keep], rv[keep])
        gi, ri = g["faces_intense"].cpu().numpy(), rg["faces_intense"].numpy()
        ei = [rel_l2(gi[b], ri[b]) for b in range(B)]
        msg += ", verts %.2e (%d grazing faces, %.1f %% of vertices kept), intensity %.2e" % (
            ev, grazing.numel(), 100 * keep.mean(), max(ei))
        assert np.abs(rv).max() > 0 and keep.mean() > 0.9
        assert ev <= VERT_TOL
        assert all(np.abs(ri[b]).max() > 0 for b in range(B))
        assert max(ei) <= INT_TOL, ei
    print("\n[tet general meshes] %s %s %s: max rel L2 %s" % (name, "det" if deterministic else "default", combo, msg))


@pytest.mark.parametrize("deterministic", [False, True], ids=["default", "det"])
def test_rigid_motion_identity_with_the_camera_inside(deterministic):
    cpu = case("inside")[0]
    gc, gd = scenes.cotangents(cpu)
    g = gpu_grads(cpu, gc, gd, deterministic, intensity=False)[3]
    gv, gm = g["verts"].cpu(), g["mv_mats"].cpu()
    r, sc, sv = rigid_residual(cpu.verts, cpu.mv_mats, gv, gm)
    r0, s0, _ = rigid_residual(cpu.verts, cpu.mv_mats, torch.zeros_like(gv), gm)   # negative control
    print("\n[tet general meshes] rigid motion, inside %s: residual %.2e of %.2e (without dL/dverts: %.2e)" % (
        "det" if deterministic else "default", r / sc, sc, r0 / s0))
    assert sv > 0.01 * sc
    assert r <= 1e-5 * sc
    assert r0 >= 1e-2 * s0
