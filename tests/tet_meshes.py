"""Seeded Delaunay tet scenes with tables in arbitrary order and cameras inside the mesh (test helper, CPU only).

scenes.kuhn_tet_grid builds its tables one way only: every row of faces[] and tets[] ascending, tet_faces[t][k] the
face opposite tet vertex 3 - k, the -1 of a boundary face always in column 1 of face_tets, and the camera outside the
mesh.  DMesh passes a Delaunay tetrahedralisation with tables in whatever order the caller built them.  The scenes
here randomise everything the API lets vary -- tet ids and the vertex order within a tet, face ids and the vertex
order within a face, the column order of tet_faces and of face_tets -- so that the adjacency records of the tet
renderer take every (side, vertex order) code, and they put cameras inside the hull, some with a mesh vertex exactly
in the camera plane (clip w = 0).

Nothing is recorded: the tests compare the CUDA path with the CPU oracle on the same scene at run time, so another
qhull version changes the mesh, never the verdict.  scipy is a test dependency only; the package does not import it.
"""
import itertools

import numpy as np
import torch
from scipy.spatial import Delaunay

from dmesh_renderer_b200 import scenes

SIDES = np.array([[0, 1, 2], [0, 1, 3], [0, 2, 3], [1, 2, 3]])   # canonical side k: the face opposite tet vertex 3 - k
PERMS3 = np.array(list(itertools.permutations(range(3))))        # every vertex order of a face: rotations, reflections
INSIDE_FOV, INSIDE_NEAR = 60.0, 0.05
PLANE_SHIFT = 5e-5                                                # eye z - vertex z of the on-plane views 1 and 2


def _canonical_tables(verts):
    """Delaunay tets of `verts` [P,3] with sorted rows in lexicographic order, faces = the unique vertex triples
    (sorted), tet_faces[t][k] = the face opposite tet vertex 3 - k, face_tets with the lower tet id in column 0."""
    tets = np.sort(Delaunay(verts.astype(np.float64)).simplices.astype(np.int64), axis=1)
    tets = tets[np.lexsort(tets.T[::-1])]
    T = tets.shape[0]
    faces, inv = np.unique(tets[:, SIDES].reshape(-1, 3), axis=0, return_inverse=True)
    inv = inv.reshape(-1)
    tet_faces = inv.reshape(T, 4)
    face_tets = np.full((faces.shape[0], 2), -1, np.int64)
    order = np.argsort(inv, kind="stable")
    inv_s, tet_s = inv[order], np.repeat(np.arange(T), 4)[order]
    first = np.ones(inv_s.shape[0], bool)
    first[1:] = inv_s[1:] != inv_s[:-1]
    face_tets[inv_s[first], 0] = tet_s[first]
    face_tets[inv_s[~first], 1] = tet_s[~first]
    return tets, faces, tet_faces, face_tets


def _shuffle_tables(rng, tets, faces, tet_faces, face_tets):
    """The same mesh with randomised ids and orders.  Returns the tables and `fp`: new face i is canonical face fp[i]."""
    T, F = tets.shape[0], faces.shape[0]
    tp = rng.permutation(T)                                       # new tet i is old tet tp[i]
    new_tet = np.empty(T, np.int64)
    new_tet[tp] = np.arange(T)
    tets, tet_faces = tets[tp], tet_faces[tp]
    tets = np.take_along_axis(tets, np.argsort(rng.random((T, 4)), axis=1), 1)           # vertex order within a tet
    tet_faces = np.take_along_axis(tet_faces, np.argsort(rng.random((T, 4)), axis=1), 1)  # side order of a tet
    fp = rng.permutation(F)                                       # new face i is old face fp[i]
    new_face = np.empty(F, np.int64)
    new_face[fp] = np.arange(F)
    faces, face_tets, tet_faces = faces[fp], face_tets[fp], new_face[tet_faces]
    faces = np.take_along_axis(faces, PERMS3[rng.integers(0, 6, F)], 1)                  # vertex order within a face
    face_tets = np.where(face_tets >= 0, new_tet[np.maximum(face_tets, 0)], -1)
    swap = rng.random(F) < 0.5                                    # the -1 of a boundary face lands in either column
    face_tets[swap] = face_tets[swap][:, ::-1]
    return tets, faces, tet_faces, face_tets, fp


def _inside_cameras(g, B, W, H, near, far):
    """look_at from points within 0.3 of the origin (inside the hull of the mesh) in random directions."""
    mv = []
    for _ in range(B):
        eye = (torch.rand(3, generator=g, dtype=torch.float64) - 0.5) * 0.6
        d = torch.randn(3, generator=g, dtype=torch.float64)
        d[1] = d[1].clamp(-0.5, 0.5)                              # keeps the up vector (0, 1, 0) well conditioned
        mv.append(scenes.look_at(eye.tolist(), (eye + d / d.norm()).tolist()))
    pj = scenes.perspective(INSIDE_FOV, W / H, near, far).unsqueeze(0).repeat(B, 1, 1)
    return torch.stack(mv).float().contiguous(), pj.float().contiguous()


def plane_vertex(verts):
    """The vertex that the on-plane cameras put into their camera plane: the one nearest the origin."""
    return int(np.argmin(np.linalg.norm(verts.astype(np.float64), axis=1)))


def _on_plane_cameras(verts, B, W, H, near, far):
    """Translation-only view matrices (looking along -z) whose eye z is that of vertex `plane_vertex` exactly (view 0:
    the vertex gets clip w = 0.0), then that z + 5e-5 and - 5e-5 (|w| < 1e-4), cyclically.  The eye sits next to the
    vertex, inside the hull."""
    v = verts[plane_vertex(verts)]
    mv = torch.eye(4).repeat(B, 1, 1)
    for b in range(B):
        ez = np.float32(v[2]) + np.float32((0.0, PLANE_SHIFT, -PLANE_SHIFT)[b % 3])      # fp32 sum, exact negation below
        mv[b, 0, 3] = -(float(v[0]) + 0.05)
        mv[b, 1, 3] = -(float(v[1]) + 0.03)
        mv[b, 2, 3] = -float(ez)
    pj = scenes.perspective(INSIDE_FOV, W / H, near, far).float().unsqueeze(0).repeat(B, 1, 1)
    return mv.contiguous(), pj.contiguous()


def delaunay_tet_scene(name, seed, n_points, H, W, B, cameras="outside", near=None, far=8.0, shuffle=True,
                       opacity=(0.0, 0.2)):
    """A scenes.Scene of kind "tet": `n_points` random points in [-1,1]^3 (numpy default_rng(seed)) tetrahedralised by
    scipy.spatial.Delaunay.  shuffle=True randomises ids and orders of every table (seeded); shuffle=False gives the
    canonical tables of the same mesh, with the same colour, opacity and intensity on each geometric face, so the two
    scenes render the same image.  `cameras`: "outside" (fibonacci directions at distance 4, near 0.5), "inside"
    (look_at from inside the hull, fov 60, near 0.05) or "on_plane" (see _on_plane_cameras; fov 60, near 0.05)."""
    rng = np.random.default_rng(seed)
    verts = rng.uniform(-1.0, 1.0, (n_points, 3)).astype(np.float32)
    tets, faces, tet_faces, face_tets = _canonical_tables(verts)
    P, F = verts.shape[0], faces.shape[0]
    fp = np.arange(F)
    if shuffle:
        tets, faces, tet_faces, face_tets, fp = _shuffle_tables(rng, tets, faces, tet_faces, face_tets)
    fp = torch.from_numpy(fp)
    g = torch.Generator().manual_seed(seed + 1000)
    verts_color = torch.rand(P, 3, generator=g)
    faces_opacity = (torch.rand(F, generator=g) * (opacity[1] - opacity[0]) + opacity[0])[fp].contiguous()
    faces_intense = (torch.rand(B, F, generator=g) * 0.5 + 0.5)[:, fp].contiguous()
    if cameras == "outside":
        mv, pj = scenes.cameras(scenes.fibonacci_dirs(B, g), 4.0, W, H, near or 0.5, far)
    elif cameras == "inside":
        mv, pj = _inside_cameras(g, B, W, H, near or INSIDE_NEAR, far)
    elif cameras == "on_plane":
        mv, pj = _on_plane_cameras(verts, B, W, H, near or INSIDE_NEAR, far)
    else:
        raise ValueError(cameras)
    vt = torch.from_numpy(verts)
    i32 = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(torch.int32)
    return scenes.Scene(name, "tet", H, W, vt, i32(faces), verts_color, faces_opacity, mv, pj,
                        scenes.ndc_depth(vt, mv, pj), faces_intense, torch.ones(3), i32(tets), i32(face_tets),
                        i32(tet_faces))


def side_codes(s):
    """[T,4] order code of each side of each tet, as tet_build_tetrec_kernel (csrc/tet_kernels.cu) writes it: with
    cyc = the vertices opposite sides k+1, k+2, k+3 (mod 4) -- the vertices of side k --, code = a | b << 2 where a and
    b are the positions of the face's first and second vertex in cyc.  -1 where the side is not made of the tet's own
    vertices."""
    tets, faces, tet_faces = (np.asarray(x, np.int64) for x in (s.tets, s.faces, s.tet_faces))
    fv = faces[tet_faces]                                          # [T,4,3]
    loc = (fv[..., None] == tets[:, None, None, :])                # [T,4,3,4]: face vertex j is tet vertex i
    ok = (loc.sum(-1) == 1).all(-1)
    loc = loc.argmax(-1)                                           # [T,4,3]
    opp = 6 - loc.sum(-1)                                          # [T,4]: tet vertex opposite side k
    k = np.arange(4)
    cyc = np.stack([opp[:, (k + j) % 4] for j in (1, 2, 3)], -1)   # [T,4,3]
    a = (cyc == loc[..., 0:1]).argmax(-1)
    b = (cyc == loc[..., 1:2]).argmax(-1)
    return np.where(ok, a | (b << 2), -1)


def clip_w(s):
    """[B,P] clip-space w of every vertex in every view (fp32, like the renderer's preprocessing)."""
    P = s.verts.shape[0]
    vh = torch.cat([s.verts, torch.ones(P, 1)], 1)
    return torch.einsum("bj,bjk,pk->bp", s.proj_mats[:, 3, :], s.mv_mats, vh)
