"""Forward and backward time with and without the alpha image and the background gradient (_C level).

    python tools/alpha_bg_timing.py [--configs C2 C4x8 C3] [--runs 30] [--warmup 5] [--out FILE]

Per config: the forward call alone (_C.render_tris / _C.render_tets) without and with the alpha image (tri_alpha /
tet_alpha right behind it), then the backward call alone without and with an alpha cotangent and the background
gradient (dL_dout_alpha=..., background_grad=True), in default and deterministic mode -- timed with CUDA events,
alternating the variants, the L2 cache overwritten (a 256 MB buffer is cleared) before every timed run; median and
spread of --runs runs after --warmup untimed ones.  C2 is the tri renderer's single-view 1024^2 config, C4x8 eight views
of C4 in one call, C3 the tet renderer's single-view 512^2 config.  Prints one JSON object with the card's name and
power limit.
"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

import torch  # noqa: E402

from camera_grad_timing import card  # noqa: E402
from dmesh_renderer_b200 import _C, scenes  # noqa: E402

SCENES = {"C2": lambda: scenes.config("C2"), "C4x8": lambda: scenes.config("C4", views=64, view_slice=slice(0, 8)),
          "C3": lambda: scenes.config("C3")}


def variants_for(s, dev):
    """{(phase, variant): callable} of one config."""
    gc, gd = [t.to(dev) for t in scenes.cotangents(s)]
    ga = gd * 0.5
    B, H, W = gd.shape[0], s.H, s.W
    mv, pj = s.mv_mats.transpose(1, 2).contiguous(), s.proj_mats.transpose(1, 2).contiguous()
    imv, ipj = torch.inverse(mv), torch.inverse(pj)
    if s.kind == "tri":
        args = (s.bg, s.verts, s.faces, s.verts_color, s.faces_opacity, mv, pj, imv, ipj, s.verts_depth, s.faces_intense)
        fwd = lambda: _C.render_tris(*args, H, W)
        out = fwd()
        bargs = args + (gc, gd) + tuple(out[:1]) + tuple(out[3:])
        alpha = lambda: _C.tri_alpha(out[6], B, H, W, dev)
        bwd = lambda det, **kw: _C.render_tris_backward(*bargs, deterministic=det, **kw)
    else:
        args = (s.bg, s.verts, s.faces, s.verts_color, s.faces_opacity, mv, pj, imv, ipj, s.verts_depth, s.faces_intense,
                s.tets, s.face_tets, s.tet_faces)
        fwd = lambda: _C.render_tets(*args, H, W, 0)
        out = fwd()
        bargs = args + (gc, gd) + tuple(out[3:]) + (0,)
        alpha = lambda: _C.tet_alpha(out[6], B, H, W, dev)
        bwd = lambda det, **kw: _C.render_tets_backward(*bargs, deterministic=det, **kw)
    v = {("forward", "off"): fwd, ("forward", "alpha"): lambda: (fwd(), alpha())}
    for det in (False, True):
        m = "det" if det else "default"
        v[("backward_" + m, "off")] = lambda det=det: bwd(det)
        v[("backward_" + m, "alpha_bg")] = lambda det=det: bwd(det, dL_dout_alpha=ga, background_grad=True)
    return v, out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--configs", nargs="+", default=list(SCENES))
    ap.add_argument("--runs", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("alpha_bg_timing.py needs a CUDA device")
    dev = torch.device("cuda", 0)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    name, power = card()
    res = {"gpu": name, "power_limit": power, "lib": os.environ.get("DMESH_B200_LIB", "in-tree"), "runs": a.runs,
           "configs": {}}
    for cfg in a.configs:
        s = scenes.to_device(SCENES[cfg](), dev)
        variants, out = variants_for(s, dev)
        times = {k: [] for k in variants}
        for it in range(a.warmup + a.runs):
            for k, fn in variants.items():
                flush.zero_()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                fn()
                e1.record()
                torch.cuda.synchronize()
                if it >= a.warmup:
                    times[k].append(e0.elapsed_time(e1))
        r = {}
        for (phase, v), t in times.items():
            t = sorted(t)
            r["%s_%s" % (phase, v)] = {"median_ms": t[len(t) // 2], "min_ms": t[0], "max_ms": t[-1]}
        for phase, on in (("forward", "alpha"), ("backward_default", "alpha_bg"), ("backward_det", "alpha_bg")):
            r["%s_ratio" % phase] = r["%s_%s" % (phase, on)]["median_ms"] / r["%s_off" % phase]["median_ms"]
        res["configs"][cfg] = r
        del s, out, variants
        torch.cuda.empty_cache()
    line = json.dumps(res)
    print(line)
    if a.out:
        with open(a.out, "a") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
