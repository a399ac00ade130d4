"""Deterministic backward passes at the limits of their fixed-point format (csrc/det.cuh).

The deterministic mode accumulates every gradient term as a fixed-point integer whose binary point is placed relative
to g = max |dL_dout|.  Its failure modes are a sum beyond the accumulator's range (which a single 64-bit word with the
binary point 38 bits below g reached at 2^(25+e) -- between 2^25 g and 2^26 g, 2^(35+e) for the vertex-position
statistics -- and then wrapped to a finite, reproducible, wrong value) and a loss of resolution when a few cotangents
are far larger than the rest.  Each case here is compared three ways: deterministic mode, default mode (fp32 atomics)
and the fp64 fragment references of test_gpu_tri_camera_grads.py / test_gpu_tet_camera_grads.py.  The reference first
has to reproduce the GPU's images; then every gradient has to agree at the suite's 1e-4 relative L2 (vertex positions
with the default mode, which uses the same formula; the reference uses the exact derivative), and two deterministic
runs have to be bit-identical.

Every range case asserts, on the fp64 reference and before any GPU run, where its largest accumulator lies in units
of g, so that a change to a scene cannot quietly move a case off the boundary it is meant to exercise:
test_range_cases_reach_their_targets runs those checks without a GPU.
"""
import math

import numpy as np
import pytest
import torch

from dmesh_renderer_b200 import TetRenderer, TetRenderSettings, TriRenderer, TriRenderSettings, scenes
from dmesh_renderer_b200.multiview import PackedSceneGrads

import test_gpu_tet_camera_grads as tetref
import test_gpu_tri_camera_grads as triref

GRAD_TOL, IMG_TOL = 1e-4, 1e-4
TRI_KEYS = ("verts", "verts_color", "faces_opacity", "verts_depth", "faces_intense")
VALUE_KEYS = ("verts_color", "faces_opacity", "verts_depth", "faces_intense")


def rel_l2(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return float(np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-30))


def old_limit(g, bits):
    """|sum| at which a single 64-bit word with the binary point `bits` below g wraps: 2^63 / 2^(bits - e)."""
    e = math.frexp(g)[1]
    return 2.0 ** (63 - bits + e)


# ---------------------------------------------------------------------------------------------- scenes
def sheet_scene(H=256, W=256, B=1, layers=2):
    """A screen-covering triangle (edge_scene's verts[0:3]) with alpha 0.5, optionally a second full-screen layer
    behind it; black background; B copies of the same camera, so each view's sums are those of view 0."""
    base = scenes.random_tri_scene("sheet", 90, 8, 0.1, H, W, B=1)
    verts = torch.tensor([[-4.0, -4.0, 0.0], [4.0, -4.0, 0.0], [0.0, 5.0, 0.2],
                          [-7.0, -7.0, -0.6], [7.0, -7.0, -0.6], [0.0, 8.0, -0.4]])[:3 * layers].contiguous()
    faces = torch.arange(3 * layers, dtype=torch.int32).reshape(layers, 3)
    g = torch.Generator().manual_seed(91)
    verts_color = (torch.rand(3 * layers, 3, generator=g) * 0.5 + 0.5).contiguous()
    mv, pj = base.mv_mats.expand(B, 4, 4).contiguous(), base.proj_mats.expand(B, 4, 4).contiguous()
    return scenes.Scene("sheet", "tri", H, W, verts, faces, verts_color, torch.full((layers,), 0.5), mv, pj,
                        scenes.ndc_depth(verts, mv, pj).contiguous(), torch.ones(B, layers), torch.zeros(3))


def scaled(cpu, param, s):
    if param == "depth":
        return cpu._replace(verts_depth=(cpu.verts_depth * s).contiguous())
    if param == "color":
        return cpu._replace(verts_color=(cpu.verts_color * s).contiguous())
    if param == "intense":
        return cpu._replace(faces_intense=(cpu.faces_intense * s).contiguous())
    raise KeyError(param)


def tri_cotangents(cpu, kind):
    B = cpu.mv_mats.shape[0]
    gc, gd = torch.ones(B, 3, cpu.H, cpu.W), torch.ones(B, 1, cpu.H, cpu.W)
    if kind == "sign":                     # the cotangent of an L1 loss: |dL_dout| = g everywhere, random signs
        gen = torch.Generator().manual_seed(92)
        gc = gc * (torch.randint(0, 2, gc.shape, generator=gen) * 2 - 1)
        gd = gd * (torch.randint(0, 2, gd.shape, generator=gen) * 2 - 1)
    return gc, gd


def g_of(gc, gd):
    return max(float(gc.abs().max()), float(gd.abs().max()))


_tri_refs = {}


def tri_reference(cpu, gc, gd, key=None):
    """(fragments, (color, depth, grads)) of the fp64 reference; cached by `key`."""
    if key is not None and key in _tri_refs:
        return _tri_refs[key]
    frags, _ = triref.oracle_fragments(cpu)
    out = (frags, triref.reference_grads(cpu, frags, gc, gd, False))
    if key is not None:
        _tri_refs[key] = out
    return out


def value_peak(grads, keys=VALUE_KEYS):
    """Largest |gradient| over the fixed-point value accumulators (one view, one face per vertex: the per-(view, face)
    records and the per-vertex / per-face accumulators hold the gradients themselves)."""
    return max(float(grads[k].abs().max()) for k in keys)


# Range sweep (a): scale one input so that the largest value accumulator lands at 2^target g.
# inside: well within the old range; below: just below it (2^25 g <= old limit 2^26 g at g = 1); past: >= 2^28 g.
# Explicit depths drive faces_opacity, vertex colours faces_intense and faces_opacity, intensities verts_color (and
# faces_opacity, which is then the largest).
TARGETS = {"inside": 22.0, "below": 25.5, "past": 29.0}
DRIVES = ("depth", "color", "intense")


def sweep_case(param, target, cot):
    """The scene, cotangents and reference of one sweep point; asserts where its largest accumulator lies."""
    key = ("sweep", param, target, cot)
    if key in _tri_refs:
        return _tri_refs[key]
    cpu0 = sheet_scene()
    gc, gd = tri_cotangents(cpu0, cot)
    g = g_of(gc, gd)
    s = 1.0
    for _ in range(3):                     # the driven gradient is affine in the scale: a few secant steps
        cpu = scaled(cpu0, param, s)
        _, (_, _, rg) = tri_reference(cpu, gc, gd)
        peak = value_peak(rg)
        if abs(math.log2(peak / g) - TARGETS[target]) < 0.25:
            break
        s *= 2.0 ** TARGETS[target] * g / peak
    frags, ref = tri_reference(cpu, gc, gd)
    assert (frags[0] == cpu.faces.shape[0]).all(), "the sheet must cover every pixel with every layer"
    peak = value_peak(ref[2])
    lim = old_limit(g, 38)
    if target == "inside":
        assert peak <= 2.0 ** 23 * g
    elif target == "below":
        assert 0.5 * lim <= peak < lim and peak >= 2.0 ** 25 * g
    else:
        assert peak >= 2.0 ** 28 * g and peak >= 4 * lim
    _tri_refs[key] = (cpu, gc, gd, frags, ref)
    return _tri_refs[key]


def cross_view_case(B):
    """(b): the same face in B views, each view below the old range, the call total (det_fopa, det_vert) above it."""
    key = ("cross", B)
    if key in _tri_refs:
        return _tri_refs[key]
    one, _, _, _, (_, _, r1) = sweep_case("depth", "below", "ones")
    per_view = value_peak(r1)
    cpu = sheet_scene(B=B)._replace(verts_depth=one.verts_depth.expand(B, -1).contiguous())
    gc, gd = tri_cotangents(cpu, "ones")
    frags, ref = tri_reference(cpu, gc, gd)
    lim = old_limit(g_of(gc, gd), 38)
    assert per_view < lim <= float(ref[2]["faces_opacity"].abs().max())
    _tri_refs[key] = (cpu, gc, gd, frags, ref)
    return _tri_refs[key]


def position_case():
    """(d): the vertex-position statistics past the old 28-bit range, 2^(35+e) g, through explicit depths scaled
    until |dL/dverts| (det_vert, and the S1 / S24 / S3 sums behind it) passes 2^37 g; fp32 stays finite."""
    key = ("position",)
    if key in _tri_refs:
        return _tri_refs[key]
    cpu0 = sheet_scene()
    gc, gd = tri_cotangents(cpu0, "ones")
    g = g_of(gc, gd)
    _, (_, _, r0) = tri_reference(cpu0, gc, gd)
    s = 2.0 ** 37.5 * g / float(r0["verts"].abs().max())
    cpu = scaled(cpu0, "depth", s)
    frags, ref = tri_reference(cpu, gc, gd)
    assert float(ref[2]["verts"].abs().max()) >= 2.0 * old_limit(g, 28)
    assert float(cpu.verts_depth.abs().max()) < 1e30
    _tri_refs[key] = (cpu, gc, gd, frags, ref)
    return _tri_refs[key]


_tet_refs = {}


def tet_range_scene(B):
    return scenes.tet_grid_scene("bigtets", 14, 2, 256, 256, B=B, opacity=(0.3, 0.6))


def tet_case(B):
    """(e): a 2x2x2 tet grid (few big tets over much of the screen), colours scaled so that the opacity accumulator
    of one view passes 2^28 g (and in a 4-view call, 2^30 g)."""
    if B in _tet_refs:
        return _tet_refs[B]
    cpu0 = tet_range_scene(B)
    gc, gd = tri_cotangents(cpu0, "ones")
    g = g_of(gc, gd)
    frags0 = tetref.oracle_fragments(cpu0)[0]
    r0 = tetref.reference_grads(cpu0, frags0, gc, gd)[2]
    s = 2.0 ** 29 * g / float(r0["faces_opacity"].abs().max()) * (B if B > 1 else 1)
    cpu = cpu0._replace(verts_color=(cpu0.verts_color * s).contiguous())
    frags = tetref.oracle_fragments(cpu)[0]
    ref = tetref.reference_grads(cpu, frags, gc, gd)
    assert float(ref[2]["faces_opacity"].abs().max()) >= 2.0 ** 28 * g * B
    assert 1e3 <= s <= 1e6               # colours of order 1e5: finite in fp32 throughout
    _tet_refs[B] = (cpu, gc, gd, frags, ref)
    return _tet_refs[B]


# ---------------------------------------------------------------------------------------------- CPU check of the cases
@pytest.mark.parametrize("cot", ["ones", "sign"])
def test_range_cases_reach_their_targets(cot):
    """No GPU: every range case lands where it is meant to (the asserts are inside the case builders)."""
    for param in DRIVES:
        for target in TARGETS:
            sweep_case(param, target, cot)
    if cot == "ones":
        for B in (4, 8):
            cross_view_case(B)
        position_case()
        for B in (1, 4):
            tet_case(B)


# ---------------------------------------------------------------------------------------------- GPU side
def tri_run(cpu, gc, gd, deterministic, exact=False):
    s = scenes.to_device(cpu, "cuda")
    leaves = [t.clone().requires_grad_() for t in (s.verts, s.verts_color, s.faces_opacity, s.verts_depth,
                                                   s.faces_intense)]
    color, depth = TriRenderer(TriRenderSettings(s.H, s.W, s.bg), deterministic=deterministic,
                               exact_vertex_grads=exact)(leaves[0], s.faces, leaves[1], leaves[2], s.mv_mats,
                                                         s.proj_mats, leaves[3], leaves[4])
    torch.autograd.backward([color, depth], [gc.cuda(), gd.cuda()])
    return color.detach().cpu(), depth.detach().cpu(), {k: t.grad.cpu() for k, t in zip(TRI_KEYS, leaves)}


def tri_sink_run(cpu, gc, gd, exact=False):
    """The deterministic kernels into PackedSceneGrads.direct() (the convert kernel adds into the sink)."""
    s = scenes.to_device(cpu, "cuda")
    pg = PackedSceneGrads(s.verts.clone(), s.verts_color.clone(), s.faces_opacity.clone())
    r = TriRenderer(TriRenderSettings(s.H, s.W, s.bg), deterministic=True, exact_vertex_grads=exact)
    with pg.direct():
        c, d = r(pg.leaves[0], s.faces, pg.leaves[1], pg.leaves[2], s.mv_mats, s.proj_mats, s.verts_depth,
                 s.faces_intense)
        torch.autograd.backward([c, d], [gc.cuda(), gd.cuda()])
    return {k: t.grad.cpu() for k, t in zip(("verts", "verts_color", "faces_opacity"), pg.leaves)}


def check_tri(cpu, gc, gd, ref, exact=False, sink=False, verts_vs_ref=False):
    rc, rd, rg = ref
    det = tri_run(cpu, gc, gd, True, exact)
    det2 = tri_run(cpu, gc, gd, True, exact)
    dflt = tri_run(cpu, gc, gd, False, exact)
    scale = max(float(rc.abs().max()), float(rd.abs().max()), 1.0)
    assert float((det[0].double() - rc).abs().max()) <= IMG_TOL * scale
    assert float((det[1].double() - rd).abs().max()) <= IMG_TOL * scale
    errs = {}
    for k in TRI_KEYS:
        assert torch.equal(det[2][k], det2[2][k]), "%s differs between two deterministic runs" % k
        assert torch.isfinite(dflt[2][k]).all(), k
        if k == "verts" and not verts_vs_ref:
            errs[k] = rel_l2(det[2][k], dflt[2][k])
        else:
            errs[k] = rel_l2(det[2][k], rg[k])
            assert rel_l2(dflt[2][k], rg[k]) <= GRAD_TOL, "default mode %s: %.3e" % (k, rel_l2(dflt[2][k], rg[k]))
        assert errs[k] <= GRAD_TOL, "deterministic %s: rel L2 %.3e" % (k, errs[k])
    if sink:
        sg = tri_sink_run(cpu, gc, gd, exact)
        for k, v in sg.items():
            assert torch.equal(v, det[2][k]), "%s through the direct sink" % k
    return errs


@pytest.mark.gpu
@pytest.mark.parametrize("exact", [False, True], ids=["reference_formula", "exact"])
@pytest.mark.parametrize("cot", ["ones", "sign"])
@pytest.mark.parametrize("target", list(TARGETS))
@pytest.mark.parametrize("param", list(DRIVES))
def test_tri_one_view_range_sweep(param, target, cot, exact):
    """(a), (c): explicit depths, vertex colours or intensities scaled until faces_opacity / faces_intense /
    verts_color reach 2^22 g, just below the old range and 2^29 g.  verts_depth's per-view accumulator is bounded by
    the pixel count (its terms are weights times the cotangent) and stays in range here.  exact: slots 21 and 22 of
    the statistics record take the position scale."""
    cpu, gc, gd, _, ref = sweep_case(param, target, cot)
    check_tri(cpu, gc, gd, ref, exact=exact, verts_vs_ref=exact)


@pytest.mark.gpu
@pytest.mark.parametrize("B", [4, 8])
def test_tri_cross_view_range(B):
    """(b): below the old range in every view, above it over the call (det_fopa sums over the views), also through
    the direct gradient sink."""
    cpu, gc, gd, _, ref = cross_view_case(B)
    check_tri(cpu, gc, gd, ref, sink=True)


@pytest.mark.gpu
def test_tri_position_statistics_range():
    """(d): vertex-position statistics (S1 / S24 / S3, the 1/det-carrying sums) and det_vert past 2^37 g, with exact
    vertex gradients compared with the fp64 reference."""
    cpu, gc, gd, _, ref = position_case()
    check_tri(cpu, gc, gd, ref, exact=True, verts_vs_ref=True)


def tet_check(cpu, gc, gd, frags, ref, deterministic_runs=2):
    fw = tetref.gpu_forward(cpu, 0)
    B, H, W = gd.shape[0], cpu.H, cpu.W
    _, out = tetref.oracle_fragments(cpu)
    parted = (fw["first_face"] != out["first_face"]) | (fw["n_contrib"] != frags["counts"])
    assert parted.sum() <= tetref.MAX_PARTED
    if parted.any():                       # compare on the same fragments only (test_gpu_tet_camera_grads.py)
        keep = torch.from_numpy(~parted).view(B, 1, H, W).float()
        gc, gd = gc * keep, gd * keep
        ref = tetref.reference_grads(cpu, frags, gc, gd)
    rc, rdp, rg = ref
    runs = [tetref.gpu_run(cpu, gc, gd, deterministic=True, mv_grad=False, pj_grad=False)
            for _ in range(deterministic_runs)]
    dflt = tetref.gpu_run(cpu, gc, gd, deterministic=False, mv_grad=False, pj_grad=False)
    act = torch.from_numpy(frags["active"]).view(runs[0][2].shape) & torch.from_numpy(~parted).view(B, H, W)
    m = act[:, None]
    scale = max(float(rc.abs().max()), 1.0)
    assert (runs[0][0].cpu().double() - rc).abs().masked_select(m).max().item() <= IMG_TOL * scale
    errs = {}
    for k in ("verts_color", "faces_opacity"):
        for r in runs[1:]:
            assert torch.equal(r[3][k], runs[0][3][k]), k
        assert rel_l2(dflt[3][k].cpu(), rg[k]) <= GRAD_TOL, "default mode %s" % k
        errs[k] = rel_l2(runs[0][3][k].cpu(), rg[k])
        assert errs[k] <= GRAD_TOL, "deterministic %s: rel L2 %.3e" % (k, errs[k])
    return errs


@pytest.mark.gpu
@pytest.mark.parametrize("B", [1, 4])
def test_tet_range(B):
    """(e): the tet accumulators det_vert / det_fopa past 2^28 g (one view) and 2^30 g (a 4-view call)."""
    tet_check(*tet_case(B))


# ---------------------------------------------------------------------------------------------- resolution (f)
def resolution_cotangents(cpu, kind, k):
    gc, gd = scenes.cotangents(cpu)
    if kind == "color_small":
        gc = gc * 2.0 ** -k
    elif kind == "depth_small":
        gd = gd * 2.0 ** -k
    else:                                  # one spike pixel at 2^k times the rest, in the colour cotangent
        gc = gc.clone()
        gc[0, 1, cpu.H // 2, cpu.W // 2] = 2.0 ** k
    return gc, gd


RES_KINDS = ["color_small", "depth_small", "spike"]


@pytest.mark.gpu
@pytest.mark.parametrize("k", [10, 20])
@pytest.mark.parametrize("kind", RES_KINDS)
@pytest.mark.parametrize("name", ["small_tri", "C1"])
def test_tri_resolution(name, kind, k):
    """(f): a cotangent image 2^-k below the other, or one pixel 2^k above the rest, moves the binary point k bits
    up for every gradient of the call; with 48 (values) and 40 (positions) fractional bits below g both k = 10 and
    k = 20 stay at the suite's tolerance."""
    cpu = triref.SCENES[name]()
    gc, gd = resolution_cotangents(cpu, kind, k)
    _, ref = tri_reference(cpu, gc, gd, key=("res", name, kind, k))
    check_tri(cpu, gc, gd, ref)


@pytest.mark.gpu
@pytest.mark.parametrize("k", [10, 20])
@pytest.mark.parametrize("kind", RES_KINDS)
def test_tet_resolution(kind, k):
    cpu = scenes.config("small_tet")
    gc, gd = resolution_cotangents(cpu, kind, k)
    frags = tetref.oracle_fragments(cpu)[0]
    tet_check(cpu, gc, gd, frags, tetref.reference_grads(cpu, frags, gc, gd))


# ---------------------------------------------------------------------------------------------- non-finite (g)
POISON = [("color", float("inf")), ("color", float("-inf")), ("color", float("nan")),
          ("depth", float("inf")), ("depth", float("-inf")), ("depth", float("nan"))]


def poisoned_cotangents(cpu, image, value):
    gc, gd = [t.clone() for t in scenes.cotangents(cpu)]
    (gc[0, 2] if image == "color" else gd[0, 0])[cpu.H // 3, cpu.W // 4] = value
    return gc, gd


@pytest.mark.gpu
@pytest.mark.parametrize("image,value", POISON, ids=["%s_%s" % (i, v) for i, v in POISON])
def test_tri_nonfinite_cotangent_poisons(image, value):
    """(g): the fixed-point format has no inf / NaN; every fixed-point output is NaN instead of a finite value."""
    cpu = scenes.config("small_tri")
    gc, gd = poisoned_cotangents(cpu, image, value)
    g = tri_run(cpu, gc, gd, True)[2]
    for k in TRI_KEYS:
        assert torch.isnan(g[k]).all(), k
    for k, v in tri_sink_run(cpu, gc, gd).items():
        assert torch.isnan(v).all(), "%s through the direct sink" % k


@pytest.mark.gpu
@pytest.mark.parametrize("image,value", POISON, ids=["%s_%s" % (i, v) for i, v in POISON])
def test_tet_nonfinite_cotangent_poisons(image, value):
    cpu = scenes.config("small_tet")
    gc, gd = poisoned_cotangents(cpu, image, value)
    g = tetref.gpu_run(cpu, gc, gd, deterministic=True, mv_grad=False, pj_grad=False)[3]
    for k in ("verts_color", "faces_opacity"):
        assert torch.isnan(g[k]).all(), k


@pytest.mark.gpu
def test_term_beyond_the_range_poisons():
    """A single term past the two-word format's per-term range (2^62 high-word units, more than 2^46 g) cannot be
    added exactly: the call is poisoned with NaN rather than returning a saturated value.  Default mode stays finite."""
    cpu = sheet_scene(layers=1)._replace(faces_intense=torch.full((1, 1), 2.0 ** 60))
    gc, gd = tri_cotangents(cpu, "ones")
    dflt = tri_run(cpu, gc, gd, False)[2]
    assert all(torch.isfinite(dflt[k]).all() for k in TRI_KEYS)
    det = tri_run(cpu, gc, gd, True)[2]
    for k in ("verts", "verts_color", "faces_opacity", "verts_depth", "faces_intense"):
        assert torch.isnan(det[k]).all(), k


# ---------------------------------------------------------------------------------------------- exponent edges (h)
@pytest.mark.gpu
def test_det_scales_edges():
    """det_scales at its two ends.  Below g = 2^-112 the binary point stops following g: at g ~ 2^-118 the gradients
    keep 42 of their 48 fractional bits and still match the default mode instead of vanishing.  A finite g in
    (3.0e38, FLT_MAX] scales like any other finite g instead of giving all-zero gradients."""
    cpu = scenes.config("small_tri")
    gc, gd = scenes.cotangents(cpu)
    base = tri_run(cpu, gc, gd, False)[2]
    k = 2.0 ** -118
    tiny = tri_run(cpu, gc * k, gd * k, True)[2]
    for n in VALUE_KEYS:
        assert rel_l2(tiny[n].double() / k, base[n]) <= GRAD_TOL, n
    # g = 3.3e38 in one colour pixel of the sheet, everything else zero: every gradient stays within fp32 (a scene
    # whose intermediate products overflow would be poisoned as a whole, which is allowed but not what is tested here)
    cpu = sheet_scene()
    gc, gd = tri_cotangents(cpu, "ones")
    gc, gd = torch.zeros_like(gc), torch.zeros_like(gd)
    gc[0, 0, cpu.H // 2, cpu.W // 2] = 3.3e38
    dflt = tri_run(cpu, gc, gd, False)[2]
    det = tri_run(cpu, gc, gd, True)[2]
    for n in TRI_KEYS:
        assert torch.isfinite(dflt[n]).all(), n
        assert n == "verts_depth" or torch.count_nonzero(det[n]) > 0, n      # no depth cotangent here
        assert rel_l2(det[n], dflt[n]) <= GRAD_TOL, n
