"""Record what the reference renderer returns for every scene the parity tests use (tests/golden/parity_record.npz).

    python tests/golden/make_parity_record.py [--renderer-verified-at REVISION]

Run on a B200.  With the reference extension built (oracle/_ref), the record holds the extension's outputs.  Without
it, the record can only be taken from this repository's CUDA renderer, and only with --renderer-verified-at naming a
revision whose native code is the code under test and whose parity tests passed against the extension; the
provenance is stored in the file.

Per scene (key: kind, sha256 of the scene inputs, ray seed; tests/ref_harness.py): R, sha256 digests of the full
integer intermediates and of the bits of final_T, a fixed sample of SAMPLE elements of each image and gradient, for
the seeded cotangents of scenes.cotangents.  tests/ref_harness.py checks the CPU oracle against it, and the CUDA
output directly where the oracle has no counterpart (jittered tet rays).
"""
import argparse
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import ref_harness as rh  # noqa: E402
import test_gpu_tet_vs_reference as tet_tests  # noqa: E402
import test_gpu_tri_large_configs as large_tests  # noqa: E402
from dmesh_renderer_b200 import _C, scenes  # noqa: E402


def tri_scenes():
    """Every tri scene the parity tests hand to the reference (same constructors, same seeds)."""
    yield from (scenes.config(n) for n in ("tiny_tri", "small_tri", "C1", "C2"))
    yield scenes.random_tri_scene("odd", 21, 2000, 0.1, 100, 75, B=2)
    yield scenes.random_tri_scene("far", 11, 4000, 0.05, 160, 160, dist=8.0, far=12.0)
    yield scenes.random_tri_scene("near", 11, 4000, 0.12, 160, 160, dist=2.0)
    yield scenes.random_tri_scene("mv4", 44, 3000, 0.09, 160, 144, B=4)
    yield from (large_tests.scene(n) for n in ("C5", "C4x8", "mv64"))


def tet_scenes():
    """(scene, ray seed) of every tet parity test."""
    yield from ((scenes.config(n), 0) for n in ("tiny_tet", "small_tet", "C3"))
    yield scenes.config("small_tet"), 7
    yield tet_tests._with_irregular_tets(scenes.config("small_tet")), 0


def record_tri(s, gc, gd, use_ref):
    if use_ref:
        fwd = rh.ref_tri_forward(s)
        it = dict(rh.ref_tri_intermediates(s, fwd))
        it["depth_keys"] = it["depths"].view(np.uint32)
        return (rh.record_entry(fwd["R"], rh.tri_ints(it), fwd["color"], fwd["depth"]),
                rh.grads_entry(rh.ref_tri_backward(s, fwd, gc, gd)))
    mv, pj = s.mv_mats.transpose(1, 2), s.proj_mats.transpose(1, 2)
    a = (s.bg, s.verts, s.faces, s.verts_color, s.faces_opacity, mv, pj, torch.inverse(mv), torch.inverse(pj),
         s.verts_depth, s.faces_intense)
    out = _C.render_tris(*a, s.H, s.W)
    grads = _C.render_tris_backward(*a, gc, gd, out[0], out[3], out[4], out[5], out[6])
    return rh.record_entry(out[0], rh.cuda_tri_ints(s, out), out[1], out[2]), rh.grads_entry(grads)


def record_tet(s, seed, gc, gd, use_ref):
    if use_ref:
        fwd = rh.ref_tet_forward(s, seed)
        it = dict(rh.ref_tet_intermediates(s, fwd), active=fwd["active"].cpu().numpy())
        it["depth_keys"] = it["min_depths"].view(np.uint32)
        return (rh.record_entry(it["R"], rh.tet_ints(it), fwd["color"], fwd["depth"]),
                rh.grads_entry(rh.ref_tet_backward(s, fwd, gc, gd)))
    mv, pj = s.mv_mats.transpose(1, 2), s.proj_mats.transpose(1, 2)
    a = (s.bg, s.verts, s.faces, s.verts_color, s.faces_opacity, mv, pj, torch.inverse(mv), torch.inverse(pj),
         s.verts_depth, s.faces_intense, s.tets, s.face_tets, s.tet_faces)
    out = _C.render_tets(*a, s.H, s.W, seed)
    grads = _C.render_tets_backward(*a, gc, gd, out[3], out[4], out[5], out[6], seed)
    R, ints = rh.cuda_tet_ints(s, out)
    return rh.record_entry(R, ints, out[0], out[1]), rh.grads_entry(grads)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--renderer-verified-at", metavar="REVISION",
                    help="record this repository's CUDA renderer (reference extension not built)")
    ap.add_argument("--out", default=rh.RECORD)
    args = ap.parse_args()
    use_ref = rh.ref_module() is not None
    if use_ref:
        provenance = "the reference CUDA extension (oracle/_ref)"
    elif args.renderer_verified_at:
        provenance = ("this repository's CUDA renderer at revision %s, whose parity tests passed against the reference "
                      "CUDA extension (integer intermediates and final_T bit for bit, images within 1e-5, gradients "
                      "within 1e-4 relative L2)" % args.renderer_verified_at)
    else:
        raise SystemExit("the reference extension oracle/_ref is not built; see the module doc")
    rec = {"provenance": np.array(provenance)}
    work = [(s, 0) for s in tri_scenes()] + list(tet_scenes())
    for cpu, seed in work:
        s = scenes.to_device(cpu, "cuda")
        gc, gd = [t.cuda() for t in scenes.cotangents(cpu)]
        fwd, grads = (record_tri(s, gc, gd, use_ref) if s.kind == "tri" else record_tet(s, seed, gc, gd, use_ref))
        key = rh.scene_key(s, seed)
        rec.update({key + "__" + k: v for k, v in {**fwd, **grads}.items()})
        print("recorded", s.name, "seed", seed, key, "R =", int(fwd["R"]), flush=True)
        del s, gc, gd
        torch.cuda.empty_cache()
    np.savez_compressed(args.out, **rec)
    print("wrote", args.out, os.path.getsize(args.out), "bytes;", provenance)


if __name__ == "__main__":
    main()
