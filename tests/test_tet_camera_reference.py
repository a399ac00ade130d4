"""CPU: the fragment exporter of the tet camera-gradient tests (tests/tet_fragments.cpp) walks exactly the oracle's own
tet march, and the fp64 reference evaluated on its fragments (tests/test_gpu_tet_camera_grads.py) reproduces the
oracle's images and its colour and opacity gradients -- the reference is validated without a GPU."""
import numpy as np
import pytest
import torch

from dmesh_renderer_b200 import scenes
from test_gpu_tet_camera_grads import GRAD_TOL, IMG_TOL, SCENES, oracle_fragments, reference_grads, rel_l2


@pytest.mark.parametrize("name", ["tiny_tet", "small_tet", "irregular"])
def test_exporter_reproduces_the_oracle_march(name):
    cpu = SCENES[name]()
    frags, out = oracle_fragments(cpu)
    assert out["mismatch"] == 0
    np.testing.assert_array_equal(frags["counts"], out["oracle_n_contrib"])
    np.testing.assert_array_equal(out["first_face"], out["oracle_first_face"])
    np.testing.assert_array_equal(out["last_face"], out["oracle_last_face"])
    np.testing.assert_array_equal(frags["active"], out["oracle_active"].reshape(-1) > 0.5)
    np.testing.assert_array_equal(out["color"].view(np.uint32), out["oracle_color"].view(np.uint32))
    np.testing.assert_array_equal(out["depth"].view(np.uint32), out["oracle_depth"].view(np.uint32))
    # the fragments of a pixel end with its last face
    ends = np.cumsum(frags["counts"].astype(np.int64)) - 1
    has = frags["counts"] > 0
    np.testing.assert_array_equal(frags["face"][ends[has]], out["last_face"][has])
    assert frags["active"].mean() > 0.3 and frags["reach"].sum() > 0


@pytest.mark.parametrize("name", ["tiny_tet", "small_tet", "irregular"])
def test_reference_reproduces_oracle_images_and_gradients(name):
    cpu = SCENES[name]()
    gc, gd = scenes.cotangents(cpu)
    frags, out = oracle_fragments(cpu, gradients=(gc, gd))
    color, depth, g = reference_grads(cpu, frags, gc, gd)
    act = torch.from_numpy(out["oracle_active"] > 0.5)[:, None]
    assert (color - torch.from_numpy(out["oracle_color"]).double()).abs().masked_select(act).max().item() <= IMG_TOL
    assert (depth - torch.from_numpy(out["oracle_depth"]).double()).abs().masked_select(act).max().item() <= IMG_TOL
    ovc, ofo = out["oracle_grads"]
    assert rel_l2(g["verts_color"].numpy(), ovc) <= GRAD_TOL
    assert rel_l2(g["faces_opacity"].numpy(), ofo) <= GRAD_TOL
    for k in ("mv_mats", "proj_mats"):
        assert torch.isfinite(g[k]).all() and g[k].abs().max() > 0
