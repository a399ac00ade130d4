"""GPU: bench.py --dump-outputs writes the outputs of the last timed step, and --steps sets the number of timed steps."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.timeout(600)
def test_bench_dumps_the_outputs_of_the_timed_step(tmp_path):
    out = tmp_path / "outputs"
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", "2", "--warmup", "1",
                        "--workload", "C1", "--no-per-config", "--dump-outputs", str(out)],
                       capture_output=True, text=True, timeout=540)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-3000:]
    result = json.loads(r.stdout.strip().splitlines()[-1])
    assert result["steps"] == 2
    # C1: 10 000 triangles (30 000 vertices), one 256 x 256 view per step -- every array fits and is stored whole
    shapes = {"grad_verts": (30_000, 3), "grad_verts_color": (30_000, 3), "grad_faces_opacity": (10_000,),
              "grad_verts_depth": (1, 30_000), "grad_faces_intense": (1, 10_000), "color": (1, 3, 256, 256),
              "depth": (1, 1, 256, 256)}
    assert sorted(os.listdir(out)) == sorted(n + ".npy" for n in shapes)
    assert sum(os.path.getsize(out / f) for f in os.listdir(out)) <= 64 << 20
    for name, shape in shapes.items():
        a = np.load(out / (name + ".npy"))
        assert a.dtype == np.float32 and a.shape == shape, (name, a.dtype, a.shape)
        assert np.isfinite(a).all() and np.abs(a).max() > 0, name
    color = np.load(out / "color.npy")
    assert color.min() >= -1e-5 and color.max() <= 1 + 1e-4

    # the same step, computed here: C1's view rendered through the public API (forward is deterministic: exact),
    # backward with the image-loss cotangent of bench.py's seeded targets (atomics: 1e-4 relative L2)
    import torch
    from dmesh_renderer_b200 import TriRenderer, TriRenderSettings, scenes
    s = scenes.to_device(scenes.config("C1"), "cuda")
    gen = torch.Generator().manual_seed(1234)
    tc, td = [torch.rand(1, c, s.H, s.W, generator=gen).cuda() for c in (3, 1)]
    leaves = [t.clone().requires_grad_() for t in (s.verts, s.verts_color, s.faces_opacity, s.verts_depth, s.faces_intense)]
    c, d = TriRenderer(TriRenderSettings(s.H, s.W, s.bg))(leaves[0], s.faces, leaves[1], leaves[2], s.mv_mats,
                                                          s.proj_mats, leaves[3], leaves[4])
    assert np.array_equal(np.load(out / "color.npy"), c.detach().cpu().numpy())
    assert np.array_equal(np.load(out / "depth.npy"), d.detach().cpu().numpy())
    torch.autograd.backward([c, d], [c.detach() - tc, d.detach() - td])
    for name, leaf in zip(("grad_verts", "grad_verts_color", "grad_faces_opacity", "grad_verts_depth",
                           "grad_faces_intense"), leaves):
        a, r = np.load(out / (name + ".npy")).astype(np.float64), leaf.grad.double().cpu().numpy()
        assert np.linalg.norm(a - r) / np.linalg.norm(r) <= 1e-4, name
