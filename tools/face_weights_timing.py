"""Forward time with and without the face visibility statistics (_C level).

    python tools/face_weights_timing.py [--configs C2 C4x8 C3] [--runs 30] [--warmup 5] [--out FILE]

Per config: the forward call (_C.render_tris with tri_forward_finish(face_weights=...), or _C.render_tets followed by
_C.tet_face_weights) without and with the statistics -- timed with CUDA events, alternating the two variants, the L2
cache overwritten (a 256 MB buffer is cleared) before every timed run; median and spread of --runs runs after --warmup
untimed ones.  C2 is the tri renderer's single-view 1024^2 config, C4x8 eight views of C4 in one call, C3 the tet
renderer's single-view 512^2 config.  Prints one JSON object with the card's name and power limit.
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


def variants_for(s):
    """{variant: callable} of one config."""
    B, H, W = s.mv_mats.shape[0], s.H, s.W
    mv, pj = s.mv_mats.transpose(1, 2).contiguous(), s.proj_mats.transpose(1, 2).contiguous()
    imv, ipj = torch.inverse(mv), torch.inverse(pj)
    if s.kind == "tri":
        def fwd(stats):
            st = _C.tri_forward_begin(s.bg, s.verts, s.faces, s.verts_color, s.faces_opacity, mv, pj, s.verts_depth,
                                      s.faces_intense, H, W)
            return _C.tri_forward_finish(st, imv, ipj, face_weights=stats)
    else:
        args = (s.bg, s.verts, s.faces, s.verts_color, s.faces_opacity, mv, pj, imv, ipj, s.verts_depth, s.faces_intense,
                s.tets, s.face_tets, s.tet_faces)

        def fwd(stats):
            out = _C.render_tets(*args, H, W, 0)
            if stats:
                out += _C.tet_face_weights(B, s.verts.shape[0], s.faces.shape[0], s.tets.shape[0], H, W, 0, imv, ipj,
                                           out[3], out[4], out[6])
            return out
    return {"off": lambda: fwd(False), "face_weights": lambda: fwd(True)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--configs", nargs="+", default=list(SCENES))
    ap.add_argument("--runs", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("face_weights_timing.py needs a CUDA device")
    dev = torch.device("cuda", 0)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    name, power = card()
    res = {"gpu": name, "power_limit": power, "lib": os.environ.get("DMESH_B200_LIB", "in-tree"), "runs": a.runs,
           "configs": {}}
    for cfg in a.configs:
        s = scenes.to_device(SCENES[cfg](), dev)
        variants = variants_for(s)
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
        for v, t in times.items():
            t = sorted(t)
            r["forward_%s" % v] = {"median_ms": t[len(t) // 2], "min_ms": t[0], "max_ms": t[-1]}
        r["forward_ratio"] = r["forward_face_weights"]["median_ms"] / r["forward_off"]["median_ms"]
        res["configs"][cfg] = r
        del s, variants
        torch.cuda.empty_cache()
    line = json.dumps(res)
    print(line)
    if a.out:
        with open(a.out, "a") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
