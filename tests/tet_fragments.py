"""ctypes wrapper of tests/tet_fragments.cpp: the fragments the CPU oracle's tet renderer composites, and which of
them its backward pass walks.

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
SRC = os.path.join(HERE, "tet_fragments.cpp")
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
    path = os.path.join(tempfile.gettempdir(), "dmesh_tet_fragments_%s_%d.so" % (h.hexdigest()[:16], os.getuid()))
    if not os.path.exists(path):
        tmp = "%s.%d.tmp" % (path, os.getpid())
        cmd = ["g++", "-O2", "-std=c++17", "-fopenmp", "-ffp-contract=off", "-fPIC", "-shared", SRC, "-o", tmp]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError("tet_fragments build failed:\n" + r.stderr[-4000:])
        os.replace(tmp, path)
    L = ctypes.CDLL(path)
    L.oracle_tet_forward.restype = ctypes.c_void_p
    L.oracle_tet_free.argtypes = [ctypes.c_void_p]
    L.oracle_tet_get.restype = None
    L.oracle_tet_backward.restype = None
    L.oracle_tet_last_face.restype = None
    L.oracle_tet_fragments.restype = ctypes.c_size_t
    L.oracle_tet_fragments.argtypes = [ctypes.c_void_p] * 10 + [ctypes.c_size_t, ctypes.c_void_p]
    _lib = L
    return L


def _p(a):
    return a.ctypes.data_as(ctypes.c_void_p) if a is not None else ctypes.c_void_p(0)


def tet_fragments(scene, mats, coords=None, gradients=None):
    """Fragments of tet scene `scene` marched by the CPU oracle with the column-major matrices `mats` = [mv, proj, inv_mv,
    inv_proj] (fp32 arrays [B,4,4]) and the ray pixel coordinates `coords` (float32 [B*H*W, 2], None = pixel centres).
    Returns (frags, out): frags = dict(counts[B*H*W] uint32, face[N] int32, reach[N] bool, active[B*H*W] bool,
    coords[B*H*W, 2] float32); out = the exporter's own images and integers (color, depth, first_face, last_face,
    mismatch) and the oracle's tet_render results (oracle_color, oracle_depth, oracle_active, oracle_first_face,
    oracle_last_face, oracle_n_contrib).  `gradients` = (dL_dcolor, dL_ddepth): also the oracle's tet_backward gradients (float64
    verts_color [P,3], faces_opacity [F]) as out["oracle_grads"]."""
    L = lib()
    B, P, F, T = scene.mv_mats.shape[0], scene.verts.shape[0], scene.faces.shape[0], scene.tets.shape[0]
    W, H = scene.W, scene.H
    BI = B * H * W
    f32 = lambda t: np.ascontiguousarray(t.detach().cpu().numpy() if hasattr(t, "detach") else t, np.float32)
    i32 = lambda t: np.ascontiguousarray(t.detach().cpu().numpy() if hasattr(t, "detach") else t, np.int32)
    a = [f32(scene.verts), i32(scene.faces), f32(scene.verts_color), f32(scene.faces_opacity)] + [f32(m) for m in mats] + \
        [f32(scene.faces_intense), i32(scene.tets), i32(scene.face_tets), i32(scene.tet_faces), f32(scene.bg)]
    if coords is None:
        ys, xs = np.meshgrid(np.arange(H), np.arange(W), indexing="ij")
        coords = np.stack([xs + 0.5, ys + 0.5], -1).astype(np.float32).reshape(1, H * W, 2).repeat(B, 0).reshape(BI, 2)
    coords = np.ascontiguousarray(coords, np.float32).reshape(BI, 2)
    h = ctypes.c_void_p(L.oracle_tet_forward(B, P, F, T, W, H, *[_p(x) for x in a]))
    try:
        counts = np.zeros(BI, np.uint32)
        ff, lf = np.zeros(BI, np.int32), np.zeros(BI, np.int32)
        act = np.zeros(BI, np.uint8)
        color, depth = np.zeros((B, 3, H, W), np.float32), np.zeros((B, 1, H, W), np.float32)
        mism = np.zeros(1, np.uint32)
        args = (_p(coords), _p(counts), _p(ff), _p(lf), _p(act), _p(color), _p(depth))
        n = int(L.oracle_tet_fragments(h, *args, None, None, 0, _p(mism)))
        face, reach = np.zeros(max(n, 1), np.int32), np.zeros(max(n, 1), np.uint8)
        L.oracle_tet_fragments(h, *args, _p(face), _p(reach), n, _p(mism))
        o = dict(oracle_color=np.zeros((B, 3, H, W), np.float32), oracle_depth=np.zeros((B, 1, H, W), np.float32),
                 oracle_active=np.zeros((B, H, W), np.float32), oracle_first_face=np.zeros(BI, np.int32),
                 oracle_n_contrib=np.zeros(BI, np.uint32), oracle_last_face=np.zeros(BI, np.int32))
        null = ctypes.c_void_p(0)
        # oracle_tet_get(h, color, depth, active, tiles_touched, offsets, depth_key, keys_sorted, vals_sorted, ranges,
        #                first_face, first_tet, n_contrib)
        L.oracle_tet_get(h, _p(o["oracle_color"]), _p(o["oracle_depth"]), _p(o["oracle_active"]), *([null] * 6),
                         _p(o["oracle_first_face"]), null, _p(o["oracle_n_contrib"]))
        L.oracle_tet_last_face(h, _p(o["oracle_last_face"]))
        if gradients is not None:
            gc, gd = (f32(g) for g in gradients)
            g = [np.zeros((P, 3)), np.zeros(F)]
            L.oracle_tet_backward(h, _p(gc), _p(gd), _p(g[0]), _p(g[1]))
            o["oracle_grads"] = g
    finally:
        L.oracle_tet_free(h)
    frags = dict(counts=counts, face=face[:n], reach=reach[:n].astype(bool), active=act.astype(bool), coords=coords)
    o.update(color=color, depth=depth, first_face=ff, last_face=lf, mismatch=int(mism[0]))
    return frags, o
