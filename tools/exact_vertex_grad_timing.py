"""Backward time of the tri renderer with the reference's and with exact vertex-position gradients (_C level, one call
of 8 views at 1024^2).

    python tools/exact_vertex_grad_timing.py [--configs C2 C4] [--runs 30] [--warmup 5] [--out FILE]

Per config: one forward (_C.render_tris), then the backward alone -- _C.render_tris_backward with
exact_vertex_grads=False and True, default and deterministic mode -- timed with CUDA events, alternating the variants,
the L2 cache overwritten (a 256 MB buffer is cleared) before every timed run; median and spread of --runs runs after
--warmup untimed ones.  C2 is rendered with its single camera repeated to 8 views, C4 with 8 of its views.  Prints one
JSON object with the card's name and power limit.
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

from dmesh_renderer_b200 import _C, scenes  # noqa: E402


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power = [x.strip() for x in q.split(",")]
    except Exception:
        name, power = torch.cuda.get_device_name(0), "unknown"
    return name, power


def scene8(name):
    if name == "C4":
        return scenes.config("C4", views=64, view_slice=slice(0, 8))
    s = scenes.config(name)
    r = lambda t: t.repeat(8, *([1] * (t.dim() - 1))).contiguous()
    return s._replace(mv_mats=r(s.mv_mats), proj_mats=r(s.proj_mats), verts_depth=r(s.verts_depth),
                      faces_intense=r(s.faces_intense))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--configs", nargs="+", default=["C2", "C4"])
    ap.add_argument("--runs", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("exact_vertex_grad_timing.py needs a CUDA device")
    dev = torch.device("cuda", 0)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    name, power = card()
    res = {"gpu": name, "power_limit": power, "lib": os.environ.get("DMESH_B200_LIB", "in-tree"), "runs": a.runs,
           "configs": {}}
    for cfg in a.configs:
        s = scenes.to_device(scene8(cfg), dev)
        gc, gd = [t.to(dev) for t in scenes.cotangents(s)]
        mv, pj = s.mv_mats.transpose(1, 2).contiguous(), s.proj_mats.transpose(1, 2).contiguous()
        imv, ipj = torch.inverse(mv), torch.inverse(pj)
        args = (s.bg, s.verts, s.faces, s.verts_color, s.faces_opacity, mv, pj, imv, ipj, s.verts_depth, s.faces_intense)
        out = _C.render_tris(*args, s.H, s.W)
        bargs = args + (gc, gd, out[0]) + tuple(out[3:])
        variants = {(det, ex): (lambda det=det, ex=ex: _C.render_tris_backward(*bargs, deterministic=det,
                                                                                exact_vertex_grads=ex))
                    for det in (False, True) for ex in (False, True)}
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
        for (det, ex), t in times.items():
            t = sorted(t)
            r["%s_%s" % ("det" if det else "default", "exact" if ex else "reference")] = {
                "median_ms": t[len(t) // 2], "min_ms": t[0], "max_ms": t[-1]}
        for mode in ("default", "det"):
            r[mode + "_ratio"] = r[mode + "_exact"]["median_ms"] / r[mode + "_reference"]["median_ms"]
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
