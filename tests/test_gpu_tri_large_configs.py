"""GPU parity at the LARGE configs of BASELINE.json: CUDA tri path (public API -> _C shim -> C ABI) against the
reference renderer on identical seeded scenes (the UNMODIFIED reference extension oracle/_ref when it is built, the
CPU oracle otherwise -- tests/ref_harness.py).

  C5      configs[4]: 4 M triangles, 2048x2048, R = 32 M instances (binning / sort dominated)
  C4x8    configs[3], one rank's share at 8 GPUs: 1 M triangles, 8 views at 1024x1024 in ONE call (multi-view
          batch: per-vertex vector accumulators in backward (use_vacc), R = 16.8 M)
  mv64    64 views in one call: B * tiles = 65536 -> 17 tile bits -> the THREE-pass tile sort (and the reference's
          7-pass 64-bit sort, cuda_rasterizer/rasterizer_impl.cu:316-324)

Same tolerances as test_gpu_tri_vs_reference.py (BASELINE.json north_star): integer / indexing work bit-exact,
images <= 1e-5 max-abs, gradients <= 1e-4 relative L2.  All comparisons run on the device (torch), so that the
test time is the two renderers' time, not host copies of 32 M-element intermediates.
"""
import numpy as np
import pytest
import torch

import ref_harness
from dmesh_renderer_b200 import TriRenderer, TriRenderSettings, _C, debug, scenes

pytestmark = pytest.mark.gpu

IMG_TOL = 1e-5
GRAD_TOL = 1e-4


def _A(x):
    return (x + 127) // 128 * 128


def rel_l2(a, b):
    a, b = a.double(), b.double()
    return ((a - b).norm() / b.norm().clamp_min(1e-30)).item()


def scene(name):
    if name == "C5":
        return scenes.config("C5")
    if name == "C4x8":
        return scenes.config("C4", views=8)
    if name == "mv64":
        return scenes.random_tri_scene("mv64", 64, 20_000, 0.05, 512, 512, B=64)
    raise KeyError(name)


def ref_views(s, fwd):
    """Device views into the reference's state buffers (layouts: SURVEY.md App. B), or the oracle's arrays on the
    device with the same dtypes."""
    if "bufs" not in fwd:
        it = ref_harness.ref_tri_intermediates(s, fwd)
        dev = lambda a, dt: torch.from_numpy(np.ascontiguousarray(a).view(dt)).to(s.verts.device)
        return {"tiles_touched": dev(it["tiles_touched"], np.int32), "values_sorted": dev(it["values_sorted"], np.int32),
                "keys_sorted": dev(it["keys_sorted"], np.int64), "final_T": dev(it["final_T"], np.int32),
                "n_contrib": dev(it["n_contrib"], np.int32), "ranges": dev(it["ranges"], np.int32)}
    B, P, F = s.mv_mats.shape[0], s.verts.shape[0], s.faces.shape[0]
    BF, BI, R = B * F, B * s.H * s.W, fwd["R"]
    pb, fb, bb, ib = fwd["bufs"]
    i32 = torch.int32
    out = {}
    out["tiles_touched"] = fb[_A(4 * BF):_A(4 * BF) + 4 * BF].view(i32)
    o = 0
    out["values_sorted"] = bb[o:o + 4 * R].view(i32); o = _A(o + 4 * R)
    o = _A(o + 4 * R)
    out["keys_sorted"] = bb[o:o + 8 * R].view(torch.int64)
    o = 0
    out["final_T"] = ib[o:o + 4 * BI].view(i32); o = _A(o + 4 * BI)
    o = _A(o + 4 * BI)
    out["n_contrib"] = ib[o:o + 4 * BI].view(i32); o = _A(o + 4 * BI)
    tiles = B * ((s.W + 15) // 16) * ((s.H + 15) // 16)
    out["ranges"] = ib[o:o + 8 * tiles].view(i32).view(tiles, 2)
    return out


@pytest.mark.parametrize("name", ["C5", "C4x8", "mv64"])
def test_tri_large_forward_and_backward_match_reference(name):
    cpu = scene(name)
    s = scenes.to_device(cpu, "cuda")
    gc, gd = [t.cuda() for t in scenes.cotangents(cpu)]
    B, P, F = s.mv_mats.shape[0], s.verts.shape[0], s.faces.shape[0]

    # ---- forward: integer intermediates bit-exact, images within 1e-5
    ref = ref_harness.ref_tri_forward(s)
    rv = ref_views(s, ref)
    mv, pj = s.mv_mats.transpose(1, 2), s.proj_mats.transpose(1, 2)
    R, color, depth, pb, fb, bb, ib = _C.render_tris(s.bg, s.verts, s.faces, s.verts_color, s.faces_opacity, mv, pj,
                                                     torch.inverse(mv), torch.inverse(pj), s.verts_depth, s.faces_intense,
                                                     s.H, s.W)
    assert R == ref["R"]
    dims = dict(B=B, P=P, F=F, W=s.W, H=s.H, R=R)
    assert torch.equal(debug.view_torch("tri", "tiles_touched", fb, **dims), rv["tiles_touched"])
    assert torch.equal(debug.view_torch("tri", "values_sorted", bb, **dims), rv["values_sorted"])
    assert torch.equal(debug.view_torch("tri", "keys_sorted", bb, face_buffer=fb, **dims), rv["keys_sorted"])
    assert torch.equal(debug.view_torch("tri", "ranges", ib, **dims), rv["ranges"])
    assert torch.equal(debug.view_torch("tri", "n_contrib", ib, **dims), rv["n_contrib"])
    assert torch.equal(debug.view_torch("tri", "final_T", ib, **dims).view(torch.int32), rv["final_T"])
    assert (color - ref["color"]).abs().max().item() <= IMG_TOL
    assert (depth - ref["depth"]).abs().max().item() <= IMG_TOL
    if name == "mv64":   # the case exists for the three-pass tile sort
        tiles = B * ((s.W + 15) // 16) * ((s.H + 15) // 16)
        assert tiles.bit_length() > 16

    # ---- backward through the public API: gradients within 1e-4 relative L2
    rg = ref_harness.ref_tri_backward(s, ref, gc, gd)
    del ref, rv, pb, fb, bb, ib
    leaves = [s.verts.clone().requires_grad_(), s.verts_color.clone().requires_grad_(),
              s.faces_opacity.clone().requires_grad_(), s.verts_depth.clone().requires_grad_(),
              s.faces_intense.clone().requires_grad_()]
    renderer = TriRenderer(TriRenderSettings(s.H, s.W, s.bg))
    color2, depth2 = renderer(leaves[0], s.faces, leaves[1], leaves[2], s.mv_mats, s.proj_mats, leaves[3], leaves[4])
    assert torch.equal(color2, color) and torch.equal(depth2, depth)      # same bits through either entry point
    torch.autograd.backward([color2, depth2], [gc, gd])
    for n, leaf, r in zip(["verts", "verts_color", "faces_opacity", "verts_depth", "faces_intense"], leaves, rg):
        e = rel_l2(leaf.grad, r)
        assert e <= GRAD_TOL, "%s: rel L2 %.3e" % (n, e)
