"""CPU: host logic of the tet renderer's camera-sharded step -- which calls a PackedSceneGrads buffer serves (with
and without the verts slot), re-binding after zero_grad(set_to_none=True), tet_multiview_step's argument checks, and
the C ABI's rejection of a negative first_view before any CUDA call."""
import ctypes

import pytest
import torch

from dmesh_renderer_b200 import _C
from dmesh_renderer_b200.multiview import PackedSceneGrads, tet_multiview_step


def _leaves(P=5, F=7):
    return torch.randn(P, 3), torch.rand(P, 3), torch.rand(F)


def test_buffer_without_positions_has_the_tet_layout():
    v, c, o = _leaves()
    g = PackedSceneGrads(None, c, o)
    assert g.flat.numel() == 3 * 5 + 7 and g.leaves == [c, o]
    assert c.grad.data_ptr() == g.flat.data_ptr() and o.grad.data_ptr() == g.flat[15:].data_ptr()
    full = PackedSceneGrads(*_leaves())
    assert full.flat.numel() == 6 * 5 + 7 and len(full.leaves) == 3
    with pytest.raises(ValueError):
        PackedSceneGrads(v, None, o)


def test_tri_call_never_matches_a_buffer_without_positions():
    v, c, o = _leaves()
    g = PackedSceneGrads(None, c, o)
    with g.direct():
        assert _C.grad_sink_for(v, c, o) is None                     # a tri call
        assert _C.grad_sink_for(v, c, o, tet=True) is g              # a tet call
        assert _C.grad_sink_for(None, c, o, tet=True) is g           # verts plays no part in this layout
    assert not _C._grad_sinks


def test_tet_call_matches_both_layouts_only_for_the_sinks_own_fp32_leaves():
    v, c, o = _leaves()
    full = PackedSceneGrads(v, c, o)
    v2, c2, o2 = [t.detach().clone() for t in _leaves()]
    part = PackedSceneGrads(None, c2, o2)
    with full.direct(), part.direct():
        assert _C.grad_sink_for(v, c, o, tet=True) is full
        assert _C.grad_sink_for(v2, c2, o2, tet=True) is part
        assert _C.grad_sink_for(v.clone(), c, o, tet=True) is None    # with a verts slot, verts must be the leaf too
        assert _C.grad_sink_for(v2, c2.clone(), o2, tet=True) is None  # a copy is not the leaf
        assert _C.grad_sink_for(v2, c2 * 1.0, o2, tet=True) is None    # neither is a function of it
        assert _C.grad_sink_for(v2, o2, c2, tet=True) is None           # order matters
        assert _C.grad_sink_for(v2, c2.double(), o2, tet=True) is None  # nor another dtype
        saved = c2.grad
        c2.grad = torch.zeros(3, 5).t()                                  # a .grad that is not contiguous
        assert _C.grad_sink_for(v2, c2, o2, tet=True) is None
        c2.grad = None                                                   # or none at all
        assert _C.grad_sink_for(v2, c2, o2, tet=True) is None
        c2.grad = saved
        assert _C.grad_sink_for(v2, c2, o2, tet=True) is part
    assert not _C._grad_sinks


def test_bind_reattaches_after_zero_grad_set_to_none():
    g = PackedSceneGrads(None, torch.zeros(5, 3), torch.zeros(7))
    assert g.bind() == 0
    opt = torch.optim.SGD(g.leaves, lr=0.1)
    g.leaves[0].grad.fill_(1.0)
    opt.zero_grad()                                   # set_to_none=True
    assert all(leaf.grad is None for leaf in g.leaves)
    with g.direct():                                  # re-attaches
        assert _C.grad_sink_for(None, *g.leaves, tet=True) is g
    for leaf in g.leaves:
        assert g.flat.data_ptr() <= leaf.grad.data_ptr() < g.flat.data_ptr() + 4 * g.flat.numel()
    g.leaves[1].grad = torch.full((7,), 2.5)          # a foreign tensor is moved into the buffer, not lost
    assert g.bind() == 1
    assert torch.equal(g.flat[15:], torch.full((7,), 2.5))
    g.zero_()
    assert float(g.flat.abs().sum()) == 0.0


def test_tet_multiview_step_needs_the_sinks_verts_when_the_buffer_holds_positions():
    v, c, o = _leaves()
    g = PackedSceneGrads(v, c, o)
    with pytest.raises(ValueError, match="verts leaf"):
        tet_multiview_step(None, g, v.detach().clone(), None, None, None, None, torch.zeros(1, 4, 4),
                           torch.zeros(1, 4, 4), None, None, None)


def test_c_abi_rejects_a_negative_first_view_without_a_gpu():
    from dmesh_renderer_b200 import _lib
    lib = _lib.load()
    null = ctypes.c_void_p(0)
    rc = lib.dmr_tet_forward_render_views(1, 4, 4, 1, 16, 16, 0, 1, -1, *([null] * 14), null)
    assert rc == 1                                    # DMR_EINVAL
    assert b"first_view" in lib.dmr_last_error()
