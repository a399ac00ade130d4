"""CPU: the fp64 reference of the camera-gradient tests (tests/test_gpu_tri_camera_grads.py), evaluated on the
fragments taken from the CPU oracle (tests/tri_fragments.cpp), reproduces the oracle's images -- the reference is
validated without a GPU."""
import numpy as np
import pytest
import torch

from test_gpu_tri_camera_grads import SCENES, IMG_TOL, oracle_fragments, reference_render


@pytest.mark.parametrize("name", ["tiny_tri", "cam4"])
def test_reference_forward_reproduces_oracle_images(name):
    cpu = SCENES[name]()
    frags, ref = oracle_fragments(cpu)
    counts = frags[0]
    assert counts.sum() == len(frags[1]) > 0
    # every pixel's fragment count is at most its n_contrib
    assert (counts.reshape(-1) <= ref["n_contrib"]).all()
    f64 = torch.float64
    color, depth = reference_render(frags, cpu.faces, cpu.H, cpu.W, cpu.bg, cpu.verts.to(f64), cpu.verts_color.to(f64),
                                    cpu.faces_opacity.to(f64), cpu.mv_mats.to(f64), cpu.proj_mats.to(f64),
                                    cpu.faces_intense.to(f64), cpu.verts_depth.to(f64))
    assert np.abs(color.numpy() - ref["color"]).max() <= IMG_TOL
    assert np.abs(depth.numpy() - ref["depth"]).max() <= IMG_TOL
