"""ctypes wrapper of tests/tri_fragments.cpp: the fragments the CPU oracle's tri renderer composites.

Test infrastructure only.  The library is compiled (g++, the oracle's flags) into the system temporary directory,
named after a hash of its sources, so that the repository tree is never written to.
"""
import ctypes
import hashlib
import os
import subprocess
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "tri_fragments.cpp")
ORACLE_SRC = os.path.join(os.path.dirname(HERE), "oracle", "oracle.cpp")

_lib = None


def lib():
    global _lib
    if _lib is not None:
        return _lib
    h = hashlib.sha256()
    for p in (SRC, ORACLE_SRC):
        with open(p, "rb") as f:
            h.update(f.read())
    path = os.path.join(tempfile.gettempdir(), "dmesh_tri_fragments_%s_%d.so" % (h.hexdigest()[:16], os.getuid()))
    if not os.path.exists(path):
        tmp = "%s.%d.tmp" % (path, os.getpid())
        cmd = ["g++", "-O2", "-std=c++17", "-fopenmp", "-ffp-contract=off", "-fPIC", "-shared", SRC, "-o", tmp]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError("tri_fragments build failed:\n" + r.stderr[-4000:])
        os.replace(tmp, path)
    L = ctypes.CDLL(path)
    L.oracle_tri_forward.restype = ctypes.c_void_p
    L.oracle_tri_free.argtypes = [ctypes.c_void_p]
    L.oracle_tri_fragments.restype = ctypes.c_size_t
    L.oracle_tri_fragments.argtypes = [ctypes.c_void_p] * 4 + [ctypes.c_size_t]
    L.oracle_tri_get.restype = None
    _lib = L
    return L


def _p(a):
    return a.ctypes.data_as(ctypes.c_void_p)


def tri_fragments(scene, mats):
    """Fragments of `scene` rendered by the CPU oracle with the column-major matrices `mats` = [mv, proj, inv_mv,
    inv_proj] (fp32 arrays [B,4,4]).  Returns (counts[B,H,W] uint32, face[N] int32, clamp code[N] int32, color[B,3,H,W]
    of the oracle, n_contrib[B*H*W])."""
    L = lib()
    B, P, F = scene.mv_mats.shape[0], scene.verts.shape[0], scene.faces.shape[0]
    W, H = scene.W, scene.H
    f32 = lambda t: np.ascontiguousarray(t.detach().cpu().numpy() if hasattr(t, "detach") else t, np.float32)
    a = [f32(scene.verts), np.ascontiguousarray(scene.faces.cpu().numpy(), np.int32), f32(scene.verts_color),
         f32(scene.faces_opacity)] + [f32(m) for m in mats] + [f32(scene.verts_depth), f32(scene.faces_intense),
                                                              f32(scene.bg)]
    h = ctypes.c_void_p(L.oracle_tri_forward(B, P, F, W, H, *[_p(x) for x in a]))
    try:
        counts = np.zeros((B, H, W), np.uint32)
        n = int(L.oracle_tri_fragments(h, _p(counts), None, None, 0))
        face, code = np.zeros(max(n, 1), np.int32), np.zeros(max(n, 1), np.int32)
        L.oracle_tri_fragments(h, _p(counts), _p(face), _p(code), n)
        color = np.zeros((B, 3, H, W), np.float32)
        depth = np.zeros((B, 1, H, W), np.float32)
        n_contrib = np.zeros(B * H * W, np.uint32)
        null = ctypes.c_void_p(0)
        # oracle_tri_get(h, color, depth, verts_image, ndc_z, tiles_touched, offsets, depth_key, keys_unsorted,
        #                vals_unsorted, keys_sorted, vals_sorted, ranges, n_contrib, final_T)
        L.oracle_tri_get(h, _p(color), _p(depth), *([null] * 10), _p(n_contrib), null)
    finally:
        L.oracle_tri_free(h)
    return counts, face[:n], code[:n], dict(color=color, depth=depth, n_contrib=n_contrib)
