"""CPU: the Delaunay tet scenes of tests/tet_meshes.py reach the inputs the Kuhn grids never produce.

Kept separately from the GPU comparison (tests/test_gpu_tet_general_meshes.py) so that the coverage those tests rely
on -- every (side, vertex order) code of the adjacency records, the -1 of a boundary face in either column of
face_tets, faces straddling the camera plane, a vertex exactly in it -- cannot erode without a failure on a machine
without a GPU.
"""
import os
import sys

import numpy as np
import pytest
import torch

import tet_meshes
from dmesh_renderer_b200 import scenes

sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "oracle"))
import oracle  # noqa: E402

H, W = 61, 83
SCENES = {
    "outside": lambda: tet_meshes.delaunay_tet_scene("outside", 21, 400, H, W, 2, cameras="outside"),
    "canonical": lambda: tet_meshes.delaunay_tet_scene("canonical", 21, 400, H, W, 2, cameras="outside", shuffle=False),
    "inside": lambda: tet_meshes.delaunay_tet_scene("inside", 21, 400, H, W, 2, cameras="inside"),
    "on_plane": lambda: tet_meshes.delaunay_tet_scene("on_plane", 21, 400, H, W, 3, cameras="on_plane"),
}
W_EPS = 1e-4          # clip w below which the renderer's preprocessing gives up on a face's screen bounding box


def pairs(s):
    c = tet_meshes.side_codes(s)
    return {(k, int(v)) for k in range(4) for v in np.unique(c[:, k])}


@pytest.mark.parametrize("name", ["outside", "canonical"])
def test_tables_are_consistent(name):
    s = SCENES[name]()
    tets, faces, ft, tf = (x.long().numpy() for x in (s.tets, s.faces, s.face_tets, s.tet_faces))
    T, F = tets.shape[0], faces.shape[0]
    # every side of a tet is made of the tet's own vertices, and the four sides are four different faces
    side = np.sort(faces[tf], axis=2)                                        # [T,4,3]
    own = np.sort(tets, axis=1)
    assert all(np.isin(side[t], own[t]).all() for t in range(T))
    assert (np.sort(tf, axis=1)[:, 1:] != np.sort(tf, axis=1)[:, :-1]).all()
    assert (tet_meshes.side_codes(s) >= 0).all()
    # face_tets lists exactly the tets whose tet_faces name the face
    owners = [[] for _ in range(F)]
    for t in range(T):
        for f in tf[t]:
            owners[f].append(t)
    for f in range(F):
        assert sorted(x for x in ft[f] if x >= 0) == sorted(owners[f])
    n = (ft >= 0).sum(1)
    assert ((n == 1) | (n == 2)).all() and (n == 1).any()
    # interior faces have two different tets; boundary faces one, its -1 in column 0 for some faces and 1 for others
    assert (ft[n == 2, 0] != ft[n == 2, 1]).all()
    if name == "canonical":
        assert (ft[:, 0] >= 0).all()
        assert (np.diff(faces, axis=1) > 0).all() and (np.diff(tets, axis=1) > 0).all()
    else:
        assert (ft[:, 0] == -1).sum() >= 10 and (ft[:, 1] == -1).sum() >= 10
        assert (np.diff(faces, axis=1) < 0).any() and (np.diff(tets, axis=1) < 0).any()


def test_canonical_and_shuffled_tables_are_the_same_mesh():
    a, b = SCENES["canonical"](), SCENES["outside"]()
    assert torch.equal(a.verts, b.verts)
    key = lambda s: {tuple(sorted(r)) for r in s.tets.tolist()}
    assert key(a) == key(b)
    fa = {tuple(sorted(r)): (o, tuple(i)) for r, o, i in zip(a.faces.tolist(), a.faces_opacity.tolist(),
                                                               a.faces_intense.T.tolist())}
    fb = {tuple(sorted(r)): (o, tuple(i)) for r, o, i in zip(b.faces.tolist(), b.faces_opacity.tolist(),
                                                               b.faces_intense.T.tolist())}
    assert fa == fb                  # same opacity and intensities on each geometric face


def test_every_side_and_order_code_occurs():
    """tet_build_tetrec_kernel encodes, per side k of a tet, the order of the face's vertices against the tet's cyclic
    order (6 codes); tet_step decodes it.  The shuffled scene has all 24 (side, code) pairs; a Kuhn grid has 4."""
    codes = {a | (b << 2) for a in range(3) for b in range(3) if a != b}       # {1, 2, 4, 6, 8, 9}
    everything = {(k, c) for k in range(4) for c in codes}
    assert pairs(SCENES["outside"]()) == everything
    assert pairs(scenes.config("small_tet")) == {(0, 6), (1, 1), (2, 8), (3, 6)}
    assert pairs(scenes.config("tiny_tet")) == {(0, 6), (1, 1), (2, 8), (3, 6)}
    assert len(pairs(SCENES["canonical"]())) == 4


def straddling(s):
    w = tet_meshes.clip_w(s)[:, s.faces.long()]                               # [B,F,3]
    return ((w.min(2).values <= W_EPS) & (w.max(2).values > W_EPS)).sum(1)


def test_inside_cameras_put_faces_across_the_camera_plane():
    assert (straddling(SCENES["inside"]()) >= 100).all()
    assert (straddling(SCENES["outside"]()) == 0).all()
    assert (tet_meshes.clip_w(SCENES["outside"]()) > 1.0).all()


def test_on_plane_cameras_hold_a_vertex_in_the_camera_plane():
    s = SCENES["on_plane"]()
    w = tet_meshes.clip_w(s)
    v = tet_meshes.plane_vertex(s.verts.numpy())
    assert float(w[0, v]) == 0.0
    assert 0.0 < float(w[1, v].abs()) < W_EPS and 0.0 < float(w[2, v].abs()) < W_EPS
    assert float(w[1, v]) * float(w[2, v]) < 0                                  # one on each side
    assert (straddling(s) >= 100).all()
    assert (s.mv_mats[:, :3, :3] == torch.eye(3)).all()                         # translation only


@pytest.mark.parametrize("name,floor", [("outside", 0.3), ("canonical", 0.3), ("inside", 0.9), ("on_plane", 0.9)])
def test_oracle_renders_nontrivial_images(name, floor):
    s = SCENES[name]()
    out = oracle.TetOracle(s).outputs()
    act = out["active"] > 0.5
    assert act.mean() > floor, act.mean()
    assert out["n_contrib"].max() >= 10
    assert np.isfinite(out["color"]).all() and np.isfinite(out["depth"]).all()
    if name != "outside" and name != "canonical":
        assert act.reshape(s.mv_mats.shape[0], -1).mean(1).min() > floor             # in every view


def test_shuffled_and_canonical_tables_render_the_same_image():
    """Relabelling the mesh changes the order of every Moeller-Trumbore evaluation, not the picture -- except at rays
    through an edge, where the fp32 hit tests of the two sides may decide differently (measured: 1 pixel)."""
    a, b = (oracle.TetOracle(SCENES[n]()).outputs() for n in ("canonical", "outside"))
    assert np.array_equal(a["active"], b["active"])
    differ = (a["n_contrib"] != b["n_contrib"]) | (np.abs(a["color"] - b["color"]).max(1).reshape(-1) > 1e-5)
    assert differ.sum() <= 4, differ.sum()
