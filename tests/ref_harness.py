"""Test-side harness around the reference renderer.

Two sources, one interface:
  * the UNMODIFIED reference extension (oracle/_ref, built by oracle/build_ref.py from a checkout of
    SonSang/dmesh_renderer): the four `_C` entry points are called exactly the way the reference's Python wrapper
    calls them (its dmesh_renderer/__init__.py:62-88, 124-149, 298-328, 373-401) and its opaque state buffers are
    unpacked with the layouts of its fromChunk functions (cuda_rasterizer/rasterizer_impl.cu:127-171,
    cuda_renderer/renderer_impl.cu:129-190; SURVEY.md App. B);
  * when that extension is not built (a plain checkout of this repository): the CPU oracle (oracle/oracle.cpp), the
    repository's port of the reference, handed the same device-computed matrices and inverses.  Every oracle result
    is first checked against the RECORD (tests/golden/parity_record.npz) of the scene: what the reference returned
    for it, as recorded by tests/golden/make_parity_record.py.  Integer intermediates and final_T are recorded as
    digests of the full arrays (compared bit for bit), images and gradients as a fixed sample of SAMPLE elements
    (1e-5 max-abs, 1e-4 relative L2).  A scene without a record fails.  The oracle casts unjittered rays only, so
    for tet calls with ray_random_seed > 0 the tests compare the CUDA output with the record directly.

Test infrastructure only -- never imported by dmesh_renderer_b200.
"""
import hashlib
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "oracle"))
import build_ref  # noqa: E402
import oracle  # noqa: E402

RECORD = os.path.join(ROOT, "tests", "golden", "parity_record.npz")
SAMPLE = 512
IMG_TOL, GRAD_TOL = 1e-5, 1e-4

_ref = None


def ref_module():
    global _ref
    if _ref is None:
        _ref = build_ref.load()
    return _ref


def _A(x):
    return (x + 127) // 128 * 128


def _view(buf, off, count, dtype):
    nbytes = count * np.dtype(dtype).itemsize
    return buf[off:off + nbytes].cpu().numpy().view(dtype)


def _host_mats(mats):
    return [m.contiguous().cpu().numpy() for m in mats]


def _dev(a, like):
    return torch.from_numpy(np.ascontiguousarray(a)).to(like.device)


def tet_seed_supported(seed):
    """Jittered tet rays (seed > 0) are compared with the reference extension itself, or with the record."""
    return seed == 0 or ref_module() is not None


# ------------------------------------------------------------------ the record of the reference's outputs
def scene_key(s, seed=0):
    h = hashlib.sha256()
    for v in s:
        if isinstance(v, torch.Tensor):
            h.update(v.detach().cpu().contiguous().numpy().tobytes())
    return "%s_%s_seed%d" % (s.kind, h.hexdigest()[:24], seed)


def _np64(a):
    return np.asarray(a.detach().cpu() if isinstance(a, torch.Tensor) else a, dtype=np.float64)


def digest(a):
    """sha256 of an integer array, or of the bit pattern of a float32 array, independent of the integer dtype."""
    a = np.ascontiguousarray(a.detach().cpu().numpy() if isinstance(a, torch.Tensor) else a)
    if a.dtype.kind == "f":
        a = a.view(np.uint32)
    return hashlib.sha256(a.astype(np.int64).tobytes()).hexdigest()


def sample(a):
    """A fixed sample of SAMPLE elements of the flattened array (all of them if it is smaller)."""
    a = _np64(a).reshape(-1)
    if a.size <= SAMPLE:
        return a
    return a[(np.arange(SAMPLE, dtype=np.int64) * 2654435761) % a.size]


def tri_ints(o):
    """The recorded integer fields from a dict with the oracle's tri output names."""
    live = np.asarray(o["tiles_touched"]) > 0
    return dict(tiles_touched=o["tiles_touched"], depth_keys_live=np.asarray(o["depth_keys"])[live],
                keys_sorted=o["keys_sorted"], values_sorted=o["values_sorted"], ranges=o["ranges"],
                n_contrib=o["n_contrib"], final_T=o["final_T"], verts_image=o["verts_image"], ndc_z=o["ndc_z"])


def tet_ints(o):
    """The recorded integer fields from a dict with the oracle's tet output names."""
    live = np.asarray(o["tiles_touched"]) > 0
    return dict(tiles_touched=o["tiles_touched"], depth_keys_live=np.asarray(o["depth_keys"])[live],
                keys_sorted=o["keys_sorted"], values_sorted=o["values_sorted"], ranges=o["ranges"],
                n_contrib=o["n_contrib"], first_face=o["first_face"], first_tet=o["first_tet"],
                active=np.asarray(o["active"]) > 0.5)


def cuda_tri_ints(s, out):
    """tri_ints of the CUDA renderer's _C.render_tris result `out`."""
    from dmesh_renderer_b200 import debug
    B, P, F = s.mv_mats.shape[0], s.verts.shape[0], s.faces.shape[0]
    d = dict(B=B, P=P, F=F, W=s.W, H=s.H, R=out[0])
    vimg = debug.view("tri", "verts_image", out[3], **d)
    o = {k: debug.view("tri", k, out[4], **d) for k in ("tiles_touched", "depth_keys")}
    o.update({k: debug.view("tri", k, out[5], face_buffer=out[4], **d) for k in ("keys_sorted", "values_sorted")})
    o.update({k: debug.view("tri", k, out[6], **d) for k in ("ranges", "n_contrib", "final_T")})
    o.update(verts_image=vimg[:, :2], ndc_z=vimg[:, 2])
    return tri_ints(o)


def cuda_tet_ints(s, out):
    """(R, tet_ints) of the CUDA renderer's _C.render_tets result `out`."""
    from dmesh_renderer_b200 import debug
    B, P, F, T = s.mv_mats.shape[0], s.verts.shape[0], s.faces.shape[0], s.tets.shape[0]
    d = dict(B=B, P=P, F=F, W=s.W, H=s.H, R=0, T=T)
    o = {k: debug.view("tet", k, out[4], **d) for k in ("tiles_touched", "depth_keys")}
    d["R"] = R = int(np.asarray(o["tiles_touched"], np.int64).sum())
    o.update({k: debug.view("tet", k, out[5], face_buffer=out[4], **d) for k in ("keys_sorted", "values_sorted")})
    o.update({k: debug.view("tet", k, out[6], **d) for k in ("ranges", "n_contrib", "first_face", "first_tet")})
    o["active"] = out[2].cpu().numpy()
    return R, tet_ints(o)


def record_entry(R, ints, color, depth):
    """What the record keeps of a forward result."""
    e = {"R": np.int64(R), "color": sample(color).astype(np.float32), "depth": sample(depth).astype(np.float32)}
    e.update({"digest_" + k: np.array(digest(v)) for k, v in ints.items()})
    return e


def grads_entry(grads):
    return {"grad%d" % i: sample(g).astype(np.float32) for i, g in enumerate(grads)}


_record = None


def recorded(key):
    global _record
    if _record is None:
        with np.load(RECORD) as z:
            _record = {k: z[k] for k in z.files}
    e = {k[len(key) + 2:]: v for k, v in _record.items() if k.startswith(key + "__")}
    assert e, ("no recorded reference output for scene %s: record it with tests/golden/make_parity_record.py on a "
               "revision whose parity tests pass against the reference extension" % key)
    return e


def check_forward(key, R, ints, color, depth):
    """A forward result (R, integer fields, images) against the record of scene `key`."""
    e = recorded(key)
    assert int(R) == int(e["R"]), "R %d, recorded %d" % (R, e["R"])
    for k, v in ints.items():
        assert digest(v) == str(e["digest_" + k]), "%s differs from the record" % k
    for k, v in (("color", color), ("depth", depth)):
        err = np.abs(sample(v) - e[k]).max()
        assert err <= IMG_TOL, "%s: max abs %.3e from the record" % (k, err)


def check_grads(key, grads):
    """Gradients against the record of scene `key` (relative L2 over the recorded sample)."""
    e = recorded(key)
    for i, g in enumerate(grads):
        r = e["grad%d" % i].astype(np.float64)
        err = np.linalg.norm(sample(g) - r) / max(np.linalg.norm(r), 1e-30)
        assert err <= GRAD_TOL, "gradient %d: rel L2 %.3e from the record" % (i, err)


def ref_tri_forward(s):
    """s: Scene on cuda.  Returns dict with outputs, num_rendered and the raw buffers (or the oracle's outputs)."""
    C = ref_module()
    mv = s.mv_mats.transpose(1, 2)
    pj = s.proj_mats.transpose(1, 2)
    imv, ipj = torch.inverse(mv), torch.inverse(pj)
    if C is None:
        o = oracle.TriOracle(s, mats=_host_mats((mv, pj, imv, ipj)))
        out = o.outputs()
        key = scene_key(s)
        check_forward(key, out["R"], tri_ints(out), out["color"], out["depth"])
        return dict(R=out["R"], color=_dev(out["color"], s.verts), depth=_dev(out["depth"], s.verts), oracle=o,
                    outputs=out, mats=(mv, pj, imv, ipj), key=key)
    R, color, depth, pb, fb, bb, ib = C.render_tris(s.bg, s.verts, s.faces, s.verts_color, s.faces_opacity, mv, pj, imv,
                                                    ipj, s.verts_depth, s.faces_intense, s.H, s.W)
    return dict(R=R, color=color, depth=depth, bufs=(pb, fb, bb, ib), mats=(mv, pj, imv, ipj))


def ref_tri_backward(s, fwd, gc, gd):
    if "oracle" in fwd:
        grads = fwd["oracle"].backward(gc, gd)
        check_grads(fwd["key"], grads)
        return [_dev(g, s.verts) for g in grads]
    C = ref_module()
    mv, pj, imv, ipj = fwd["mats"]
    pb, fb, bb, ib = fwd["bufs"]
    return C.render_tris_backward(s.bg, s.verts, s.faces, s.verts_color, s.faces_opacity, mv, pj, imv, ipj,
                                  s.verts_depth, s.faces_intense, gc, gd, fwd["R"], pb, fb, bb, ib)


def ref_tri_intermediates(s, fwd):
    if "oracle" in fwd:
        o = fwd["outputs"]
        out = {k: o[k] for k in ("verts_image", "ndc_z", "tiles_touched", "offsets", "values_sorted", "values_unsorted",
                                 "keys_sorted", "keys_unsorted", "final_T", "n_contrib", "ranges")}
        out["depths"] = o["depth_keys"].view(np.float32)    # a live face's depth key is the bit pattern of its depth
        return out
    B, P, F = s.mv_mats.shape[0], s.verts.shape[0], s.faces.shape[0]
    BP, BF, BI = B * P, B * F, B * s.H * s.W
    R = fwd["R"]
    pb, fb, bb, ib = fwd["bufs"]
    out = {}
    ndc = _view(pb, 0, 3 * BP, np.float32).reshape(BP, 3)
    out["ndc_z"] = ndc[:, 2].copy()
    out["verts_image"] = _view(pb, _A(12 * BP), 2 * BP, np.float32).reshape(BP, 2)
    out["depths"] = _view(fb, 0, BF, np.float32)
    out["tiles_touched"] = _view(fb, _A(4 * BF), BF, np.uint32)
    out["offsets"] = _view(fb, fb.numel() - 128 - 4 * BF, BF, np.uint32)
    o = 0
    out["values_sorted"] = _view(bb, o, R, np.uint32); o = _A(o + 4 * R)
    out["values_unsorted"] = _view(bb, o, R, np.uint32); o = _A(o + 4 * R)
    out["keys_sorted"] = _view(bb, o, R, np.uint64); o = _A(o + 8 * R)
    out["keys_unsorted"] = _view(bb, o, R, np.uint64)
    o = 0
    out["final_T"] = _view(ib, o, BI, np.float32); o = _A(o + 4 * BI)
    out["final_prev_T"] = _view(ib, o, BI, np.float32); o = _A(o + 4 * BI)
    out["n_contrib"] = _view(ib, o, BI, np.uint32); o = _A(o + 4 * BI)
    tiles = B * ((s.W + 15) // 16) * ((s.H + 15) // 16)
    out["ranges"] = _view(ib, o, 2 * tiles, np.uint32).reshape(tiles, 2)
    return out


def ref_tet_forward(s, seed=0):
    C = ref_module()
    mv = s.mv_mats.transpose(1, 2)
    pj = s.proj_mats.transpose(1, 2)
    imv, ipj = torch.inverse(mv), torch.inverse(pj)
    if C is None:
        if not tet_seed_supported(seed):
            raise ValueError("the CPU oracle casts unjittered rays only (ray_random_seed 0), got seed %d: compare "
                             "with the record (check_forward / check_grads)" % seed)
        o = oracle.TetOracle(s, mats=_host_mats((mv, pj, imv, ipj)))
        out = o.outputs()
        key = scene_key(s, seed)
        check_forward(key, out["R"], tet_ints(out), out["color"], out["depth"])
        return dict(color=_dev(out["color"], s.verts), depth=_dev(out["depth"], s.verts),
                    active=_dev(out["active"], s.verts), oracle=o, outputs=out, mats=(mv, pj, imv, ipj), key=key)
    color, depth, active, pb, fb, bb, ib = C.render_tets(s.bg, s.verts, s.faces, s.verts_color, s.faces_opacity, mv, pj,
                                                         imv, ipj, s.verts_depth, s.faces_intense, s.tets, s.face_tets,
                                                         s.tet_faces, s.H, s.W, seed)
    return dict(color=color, depth=depth, active=active, bufs=(pb, fb, bb, ib), mats=(mv, pj, imv, ipj))


def ref_tet_backward(s, fwd, gc, gd):
    if "oracle" in fwd:
        grads = fwd["oracle"].backward(gc, gd)
        check_grads(fwd["key"], grads)
        return [_dev(g, s.verts) for g in grads]
    C = ref_module()
    mv, pj, imv, ipj = fwd["mats"]
    pb, fb, bb, ib = fwd["bufs"]
    return C.render_tets_backward(s.bg, s.verts, s.faces, s.verts_color, s.faces_opacity, mv, pj, imv, ipj,
                                  s.verts_depth, s.faces_intense, s.tets, s.face_tets, s.tet_faces, gc, gd, pb, fb, bb,
                                  ib)


def ref_tet_intermediates(s, fwd):
    if "oracle" in fwd:
        o = fwd["outputs"]
        out = {k: o[k] for k in ("R", "tiles_touched", "offsets", "values_sorted", "keys_sorted", "ranges", "n_contrib",
                                 "first_face", "first_tet")}
        out["min_depths"] = o["depth_keys"].view(np.float32)  # a live face's depth key is the bit pattern of its min depth
        return out
    B, P, F = s.mv_mats.shape[0], s.verts.shape[0], s.faces.shape[0]
    BP, BF, BI = B * P, B * F, B * s.H * s.W
    pb, fb, bb, ib = fwd["bufs"]
    out = {}
    out["verts_image"] = _view(pb, _A(12 * BP), 2 * BP, np.float32).reshape(BP, 2)
    o = 0
    out["depths"] = _view(fb, o, BF, np.float32); o = _A(o + 4 * BF)
    out["min_depths"] = _view(fb, o, BF, np.float32); o = _A(o + 4 * BF)
    out["max_depths"] = _view(fb, o, BF, np.float32); o = _A(o + 4 * BF)
    out["tiles_touched"] = _view(fb, o, BF, np.uint32)
    out["offsets"] = _view(fb, fb.numel() - 128 - 4 * BF, BF, np.uint32)
    R = int(out["offsets"][-1]) if BF else 0
    out["R"] = R
    o = 0
    out["values_sorted"] = _view(bb, o, R, np.uint32); o = _A(o + 4 * R)
    out["values_unsorted"] = _view(bb, o, R, np.uint32); o = _A(o + 4 * R)
    out["keys_sorted"] = _view(bb, o, R, np.uint64); o = _A(o + 8 * R)
    out["keys_unsorted"] = _view(bb, o, R, np.uint64)
    tiles = B * ((s.W + 15) // 16) * ((s.H + 15) // 16)
    o = 0
    out["n_contrib"] = _view(ib, o, BI, np.uint32); o = _A(o + 4 * BI)
    out["ranges"] = _view(ib, o, 2 * tiles, np.uint32).reshape(tiles, 2); o = _A(o + 8 * BI)
    out["final_log_T"] = _view(ib, o, BI, np.float32); o = _A(o + 4 * BI)
    out["final_prev_log_T"] = _view(ib, o, BI, np.float32); o = _A(o + 4 * BI)
    o = _A(o + 12 * BI)   # ray_o
    o = _A(o + 12 * BI)   # ray_d
    out["first_face"] = _view(ib, o, BI, np.int32); o = _A(o + 4 * BI)
    out["first_tet"] = _view(ib, o, BI, np.int32); o = _A(o + 4 * BI)
    out["last_face"] = _view(ib, o, BI, np.int32); o = _A(o + 4 * BI)
    out["last_tet"] = _view(ib, o, BI, np.int32)
    return out
