"""Backward time of the tet renderer with and without face-intensity gradients (_C level).

    python tools/tet_intensity_grad_timing.py [--configs C3 C3x4] [--runs 30] [--warmup 5] [--out FILE]

Per config: one forward (_C.render_tets), then the backward alone -- _C.render_tets_backward with the intensity path
off, on (intensity_grads=True), and on together with camera and vertex-position gradients (compared with camera and
vertex-position gradients alone), in default and deterministic mode -- timed with CUDA events, alternating the
variants, the L2 cache overwritten (a 256 MB buffer is cleared) before every timed run; median and spread of --runs
runs after --warmup untimed ones.  C3 is the single-view 512^2 config; C3x4 the same geometry seen by four cameras in
one 512^2 call.  Prints one JSON object with the card's name and power limit.
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
from tet_camera_grad_timing import scene  # noqa: E402

ALL = dict(camera_grads=True, vertex_grads=True)
VARIANTS = {"off": dict(), "intensity": dict(intensity_grads=True), "camera_vertex": ALL,
            "intensity_camera_vertex": dict(ALL, intensity_grads=True)}
# (variant, the mode it modifies)
RATIOS = (("intensity", "off"), ("intensity_camera_vertex", "camera_vertex"))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--configs", nargs="+", default=["C3", "C3x4"])
    ap.add_argument("--runs", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("tet_intensity_grad_timing.py needs a CUDA device")
    dev = torch.device("cuda", 0)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    name, power = card()
    res = {"gpu": name, "power_limit": power, "lib": os.environ.get("DMESH_B200_LIB", "in-tree"), "runs": a.runs,
           "configs": {}}
    for cfg in a.configs:
        s = scenes.to_device(scene(cfg), dev)
        gc, gd = [t.to(dev) for t in scenes.cotangents(s)]
        mv, pj = s.mv_mats.transpose(1, 2).contiguous(), s.proj_mats.transpose(1, 2).contiguous()
        imv, ipj = torch.inverse(mv), torch.inverse(pj)
        args = (s.bg, s.verts, s.faces, s.verts_color, s.faces_opacity, mv, pj, imv, ipj, s.verts_depth, s.faces_intense,
                s.tets, s.face_tets, s.tet_faces)
        out = _C.render_tets(*args, s.H, s.W, 0)
        bargs = args + (gc, gd) + tuple(out[3:]) + (0,)
        variants = {(det, v): (lambda det=det, kw=kw: _C.render_tets_backward(*bargs, deterministic=det, **kw))
                    for det in (False, True) for v, kw in VARIANTS.items()}
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
        for (det, v), t in times.items():
            t = sorted(t)
            r["%s_%s" % ("det" if det else "default", v)] = {"median_ms": t[len(t) // 2], "min_ms": t[0], "max_ms": t[-1]}
        for mode in ("default", "det"):
            for v, base in RATIOS:
                r["%s_%s_ratio" % (mode, v)] = r["%s_%s" % (mode, v)]["median_ms"] / r["%s_%s" % (mode, base)]["median_ms"]
        res["configs"][cfg] = r
        del s, out, bargs, variants
        torch.cuda.empty_cache()
    line = json.dumps(res)
    print(line)
    if a.out:
        with open(a.out, "a") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
