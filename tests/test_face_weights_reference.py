"""CPU: the fp64 reference of the face visibility statistics (tests/test_gpu_face_weights.py) on hand-made fragments.

For view b and face f, weights[b, f] = sum over the pixels of b where f was composited of T_before * alpha_f and
hits[b, f] = the number of those pixels; per pixel the weights telescope to 1 - prod (1 - alpha).
"""
import numpy as np
import torch

f64 = torch.float64


def scatter_reference(B, F, pix_view, counts, face, opacity):
    """fp64 (weights, hits) [B,F] from fragments in compositing order: counts [pixels], face [N], opacity [N] (fp64);
    pix_view [pixels] = the view of each pixel."""
    cnt = torch.from_numpy(np.asarray(counts).astype(np.int64))
    n = cnt.numel()
    N = int(cnt.sum())
    pix = torch.repeat_interleave(torch.arange(n), cnt)
    rank = torch.arange(N) - (torch.cumsum(cnt, 0) - cnt)[pix]
    K = max(int(cnt.max()) if N else 1, 1)
    one_minus = torch.ones(n, K, dtype=f64).index_put((pix, rank), 1 - opacity)
    T_before = torch.cumprod(torch.cat([torch.ones(n, 1, dtype=f64), one_minus[:, :-1]], 1), 1)
    w = T_before[pix, rank] * opacity
    idx = torch.from_numpy(np.asarray(pix_view).astype(np.int64))[pix] * F + torch.from_numpy(np.asarray(face).astype(np.int64))
    weights = torch.zeros(B * F, dtype=f64).index_add_(0, idx, w)
    hits = torch.zeros(B * F, dtype=torch.int64).index_add_(0, idx, torch.ones(N, dtype=torch.int64))
    return weights.view(B, F), hits.view(B, F)


def test_hand_computed_example():
    # view 0: pixel 0 composites faces 2 (0.5) then 0 (0.25); pixel 1 composites face 0 (0.25); view 1: pixel 2 nothing,
    # pixel 3 composites face 1 (1.0) then face 2 (0.5) (after an opaque face T = 0)
    counts = [2, 1, 0, 2]
    face = [2, 0, 0, 1, 2]
    op = torch.tensor([0.5, 0.25, 0.25, 1.0, 0.5], dtype=f64)
    w, h = scatter_reference(2, 3, [0, 0, 1, 1], counts, face, op)
    assert torch.allclose(w, torch.tensor([[0.5 * 0.25 + 0.25, 0.0, 0.5], [0.0, 1.0, 0.0]], dtype=f64))
    assert torch.equal(h, torch.tensor([[2, 0, 1], [0, 1, 1]]))


def test_weights_telescope_to_alpha():
    g = torch.Generator().manual_seed(4)
    B, HW, F = 3, 50, 20
    counts = torch.randint(0, 9, (B * HW,), generator=g).numpy()
    N = int(counts.sum())
    face = torch.randint(0, F, (N,), generator=g).numpy()
    opacity = torch.rand(F, generator=g, dtype=f64)
    w, h = scatter_reference(B, F, np.arange(B * HW) // HW, counts, face, opacity[torch.from_numpy(face)])
    pix = np.repeat(np.arange(B * HW), counts)
    T = torch.ones(B * HW, dtype=f64)
    for i in range(N):
        T[pix[i]] *= 1 - opacity[face[i]]
    alpha = (1 - T).view(B, HW).sum(1)
    assert torch.allclose(w.sum(1), alpha, rtol=1e-12, atol=1e-12)
    assert h.sum().item() == N and h.view(-1).tolist() == np.bincount(
        (pix // HW) * F + face, minlength=B * F).tolist()
