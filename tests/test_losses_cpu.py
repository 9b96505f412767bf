"""CPU check of the composite (autograd) path of nphm_b200.models.loss_functions against the reference's
actual_compute_loss (loss_functions.py:20-110) - same weights, same batch; the reference's losses and its gradient with
respect to lin1.weight (sampled: the 1024 largest entries and a seeded set) are stored in golden/losses.npz
(tests/golden/make_golden_reference.py).  The native path needs a GPU (test_gpu_losses.py)."""
import numpy as np
import torch

from conftest import load_golden, make_ensemble


def test_composite_training_losses_match_the_reference_function_on_cpu():
    from nphm_b200.models import loss_functions as L
    g = load_golden('losses.npz')
    ours = make_ensemble(0).train()
    rng = np.random.RandomState(11)
    B, n = 2, 40

    def pts(scale):
        return torch.from_numpy((rng.randn(B, n, 3) * scale).astype(np.float32))
    batch = {'points_face': pts(0.12), 'points_non_face': pts(0.2), 'sup_grad_near': pts(0.15), 'sup_grad_far': pts(0.4),
             'normals_face': pts(1.0), 'normals_non_face': pts(1.0), 'gt_anchors': pts(0.1)[:, :39]}
    batch['gt_anchors'] = torch.from_numpy((rng.randn(B, 39, 3) * 0.1).astype(np.float32))
    cond = torch.from_numpy((rng.randn(B, 1, 1344) * 0.3).astype(np.float32)).requires_grad_()
    want = {k: float(g['cpu_' + k]) for k in g['cpu_keys']}
    got = L.actual_compute_loss(batch, ours, cond)
    assert set(got) == set(want)
    for k in want:
        assert abs(float(got[k].detach()) - want[k]) <= 1e-5 * max(1.0, abs(want[k])), (k, float(got[k].detach()), want[k])
    # the graph reaches the weights through the spatial gradient (double backward), like the reference's
    total_g = sum(got[k] for k in ('surf_sdf', 'normals', 'grad'))
    gg = torch.autograd.grad(total_g, ours.ensembled_deep_sdf.lin1.weight)[0]
    assert gg.shape == tuple(g['cpu_grad_lin1_shape'])
    gg = gg.reshape(-1).numpy()[g['cpu_grad_lin1_idx']]
    assert float(np.abs(g['cpu_grad_lin1'] - gg).max()) <= 1e-4 * max(1e-6, float(g['cpu_grad_lin1_absmax']))
