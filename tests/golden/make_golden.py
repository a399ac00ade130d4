"""Generate the golden fixtures of tests/golden/*.npz from the UNMODIFIED reference
CUDA extension (oracle/_ref, built by oracle/build_ref.py from /root/reference).

Run on a B200 box (the reference has no CPU path):

    gpurun -- 'python tests/golden/make_golden.py gpurun_out/golden'
    cp gpurun_out/golden/*.npz tests/golden/

Scene inputs are NOT stored: they are regenerated from the seeded scene definitions
in dmesh_renderer_b200/scenes.py (a checksum of the inputs is stored and verified
by the tests).  The four matrix stacks handed to the `_C` entry points ARE stored:
the inverses come from torch.inverse on the GPU (reference __init__.py:62-63),
whose last bits differ from a CPU inverse, and the ray/triangle barycentrics are
ill-conditioned enough to amplify that above the 1e-5 image tolerance.  Stored per scene: forward images, the integer intermediates unpacked
from the reference's state buffers (tests/ref_harness.py, SURVEY.md App. B) and
the gradients for seeded cotangents.
"""
import hashlib
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import ref_harness  # noqa: E402
from dmesh_renderer_b200 import scenes  # noqa: E402

TRI = ["tiny_tri", "small_tri"]
TET = ["tiny_tet", "small_tet"]


def input_checksum(s):
    h = hashlib.sha256()
    for v in s:
        if isinstance(v, torch.Tensor):
            h.update(v.detach().cpu().contiguous().numpy().tobytes())
    return h.hexdigest()


def main(out_dir):
    if ref_harness.ref_module() is None:   # the harness would answer with the CPU oracle, which these fixtures pin
        raise SystemExit("the reference extension oracle/_ref is not built (oracle/build_ref.py)")
    os.makedirs(out_dir, exist_ok=True)
    for name in TRI:
        cpu = scenes.config(name)
        s = scenes.to_device(cpu, "cuda")
        gc, gd = [t.cuda() for t in scenes.cotangents(cpu)]
        fwd = ref_harness.ref_tri_forward(s)
        it = ref_harness.ref_tri_intermediates(s, fwd)
        g = ref_harness.ref_tri_backward(s, fwd, gc, gd)
        live = it["tiles_touched"] > 0
        np.savez_compressed(
            os.path.join(out_dir, name + ".npz"), checksum=input_checksum(cpu), R=fwd["R"],
            mats=np.stack([m.contiguous().cpu().numpy() for m in fwd["mats"]]),
            color=fwd["color"].cpu().numpy(), depth=fwd["depth"].cpu().numpy(),
            verts_image=it["verts_image"], ndc_z=it["ndc_z"], tiles_touched=it["tiles_touched"], offsets=it["offsets"],
            depth_keys=np.where(live, it["depths"].view(np.uint32), 0).astype(np.uint32),
            keys_sorted=it["keys_sorted"], values_sorted=it["values_sorted"], ranges=it["ranges"],
            n_contrib=it["n_contrib"], final_T=it["final_T"],
            g_verts=g[0].cpu().numpy(), g_verts_color=g[1].cpu().numpy(), g_faces_opacity=g[2].cpu().numpy(),
            g_verts_depth=g[3].cpu().numpy(), g_faces_intense=g[4].cpu().numpy())
        print("wrote", name, "R =", fwd["R"])
    for name in TET:
        cpu = scenes.config(name)
        s = scenes.to_device(cpu, "cuda")
        gc, gd = [t.cuda() for t in scenes.cotangents(cpu)]
        fwd = ref_harness.ref_tet_forward(s, 0)
        it = ref_harness.ref_tet_intermediates(s, fwd)
        g = ref_harness.ref_tet_backward(s, fwd, gc, gd)
        live = it["tiles_touched"] > 0
        np.savez_compressed(
            os.path.join(out_dir, name + ".npz"), checksum=input_checksum(cpu), R=it["R"],
            mats=np.stack([m.contiguous().cpu().numpy() for m in fwd["mats"]]),
            color=fwd["color"].cpu().numpy(), depth=fwd["depth"].cpu().numpy(), active=fwd["active"].cpu().numpy(),
            tiles_touched=it["tiles_touched"], offsets=it["offsets"],
            depth_keys=np.where(live, it["min_depths"].view(np.uint32), 0).astype(np.uint32),
            keys_sorted=it["keys_sorted"], values_sorted=it["values_sorted"], ranges=it["ranges"],
            first_face=it["first_face"], first_tet=it["first_tet"], n_contrib=it["n_contrib"],
            g_verts_color=g[0].cpu().numpy(), g_faces_opacity=g[1].cpu().numpy())
        print("wrote", name, "R =", it["R"], "active", float(fwd["active"].mean()))


if __name__ == "__main__":
    main(sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "gpurun_out", "golden"))
