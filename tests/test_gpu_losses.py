"""SURVEY.md 8f-3: the identity-space training losses (reference loss_functions.py:20-110) evaluated natively - SDF values and
spatial gradients from nphm_ensemble_backward_inputs, no autograd graph - against the UNMODIFIED reference function running on
its own modules with autograd, same weights, same batch (its losses are stored in golden/losses.npz,
tests/golden/make_golden_reference.py)."""
import numpy as np
import pytest
import torch

from conftest import load_golden, make_ensemble

pytestmark = pytest.mark.gpu


def _batch(rng, B, n, dev):
    def pts(scale):
        return torch.from_numpy((rng.randn(B, n, 3) * scale + np.array([0.0, 0.05, -0.1])).astype(np.float32)).to(dev)

    def unit():
        v = rng.randn(B, n, 3).astype(np.float32)
        return torch.from_numpy(v / np.linalg.norm(v, axis=-1, keepdims=True)).to(dev)
    return {'points_face': pts(0.12), 'points_non_face': pts(0.2), 'sup_grad_near': pts(0.15), 'sup_grad_far': pts(0.4),
            'normals_face': unit(), 'normals_non_face': unit(),
            'gt_anchors': torch.from_numpy((rng.randn(B, 39, 3) * 0.1).astype(np.float32)).to(dev)}


def test_native_training_losses_match_the_reference_function(cuda_device):
    from nphm_b200.models import loss_functions as L
    gold = load_golden('losses.npz')
    ours = make_ensemble(0, device=cuda_device).train()
    rng = np.random.RandomState(5)
    B, n = 3, 700
    batch = _batch(rng, B, n, cuda_device)
    cond = torch.from_numpy((rng.randn(B, 1, 1344) * 0.3).astype(np.float32)).to(cuda_device)
    want = {k: float(gold['gpu_' + k]) for k in gold['gpu_keys']}
    with torch.no_grad():
        got = L.actual_compute_loss(batch, ours, cond)                      # native: no graph
    got_graph = L.actual_compute_loss(batch, ours, cond)                    # composite: autograd, what training uses
    assert set(got) == set(want) == set(got_graph)
    for k, w in want.items():
        for name, g in (('native', got[k]), ('composite', got_graph[k])):
            g = float(g.detach())
            assert abs(g - w) <= 2e-5 * max(1.0, abs(w)), (k, name, g, w)
        print('%-12s reference %.7f  native %.7f  composite %.7f' % (k, w, float(got[k].detach()), float(got_graph[k].detach())))
    assert not got['grad'].requires_grad and got_graph['grad'].requires_grad
