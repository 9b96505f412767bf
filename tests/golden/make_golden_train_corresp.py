#!/usr/bin/env python
"""Generate train_corresp.npz: one stage-2 training step of the UNMODIFIED reference (``compute_loss_corresp_forward``,
loss_functions.py:282-322, the weighted total of training_corresp.py:154-176 and one ``backward()``) for both shipped
configurations, so that tests/test_training_cpu.py and tests/test_gpu_training.py compare against the reference without a
reference checkout.

    python oracle/make_ref.py                      # reference modules -> oracle/_ref
    python tests/golden/make_golden_train_corresp.py

torch on the CPU, fp32, training mode.  Configurations: ``nphm`` = DeformationNetwork(compress) 512 x 6 (nphm_def.yaml),
``npm`` = DeepSDF 712 -> 1024 x 8 -> 3 (train_corresp.py:71-77), lambdas of nphm_def.yaml / npm_def.yaml, B = 4, 300
correspondences, 100 samples.  The random numbers the reference draws inside the step (the per-point noise on the compressed
identity code, the raw ``torch.rand`` behind the samples) are recorded and stored, so a replay can inject them.  Weights are
seeded and pinned by per-tensor SHA-256; per weight tensor the gradient's norm and its values at (up to) 4096 seeded positions
are stored, the gradients of the expression codes and of the correspondence points in full."""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
from oracle import ref_loader as R        # noqa: E402
from make_golden_reference import pin_state  # noqa: E402

B, N_CORR, N_SAMP = 4, 300, 100
SEEDS = {'nphm': 20, 'npm': 21}
ID_DIM = {'nphm': 64 + 40 * 32, 'npm': 512}
LAMBDAS = {'nphm': {'corresp': 100.0, 'lat_reg': 5e-5, 'loss_reg_zero': 5e-5},
           'npm': {'corresp': 100.0, 'lat_reg': 5e-5, 'loss_reg_zero': 0.0}}
N_POS = 4096


def positions(numel, i):
    """Seeded positions of weight tensor i (same rule in the tests)."""
    if numel <= N_POS:
        return np.arange(numel)
    return np.sort(np.random.default_rng(1000 + i).choice(numel, N_POS, replace=False))


class Recorder(torch.nn.Module):
    """Passes the decoder calls through and keeps the point tensors they received (the gradient of the correspondence points
    lands on the first one)."""

    def __init__(self, dec):
        super().__init__()
        self.dec = dec
        self.points = []

    def forward(self, xyz, cond, anchors):
        self.points.append(xyz)
        return self.dec(xyz, cond, anchors)


def make_decoder(ns, kind):
    torch.manual_seed(SEEDS[kind])
    if kind == 'nphm':
        return ns.deepSDF.DeformationNetwork(mode='compress', lat_dim_expr=200, lat_dim_id=32, lat_dim_glob_shape=64,
                                             lat_dim_loc_shape=32, n_loc=39, anchors=R.mean_anchors(ns), hidden_dim=512,
                                             nlayers=6, out_dim=3, input_dim=3).train()
    return ns.deepSDF.DeepSDF(lat_dim=712, hidden_dim=1024, geometric_init=False, out_dim=3, input_dim=3).train()


def inputs(kind):
    g = torch.Generator().manual_seed(SEEDS[kind] + 100)
    pts = (torch.rand(B, N_CORR, 3, generator=g) - 0.5) * 1.6
    return {'codes': torch.randn(B, 200, generator=g) * 0.01,
            'codes_shape': torch.randn(B, ID_DIM[kind], generator=g) * 0.05,
            'points_neutral': pts, 'points_posed': pts + 0.02 * torch.randn(B, N_CORR, 3, generator=g),
            'gt_anchors': torch.randn(B, 39, 3, generator=g) * 0.3}


def one(ns, kind, out):
    dec = make_decoder(ns, kind)
    pin_state(out, kind, dec)
    x = inputs(kind)
    codes = torch.nn.Embedding(B, 200)
    codes.weight.data.copy_(x['codes'])
    codes_shape = torch.nn.Embedding(B, ID_DIM[kind])
    codes_shape.weight.data.copy_(x['codes_shape'])
    codes_shape.weight.requires_grad_(False)
    batch = {'idx': torch.arange(B)[:, None], 'subj_ind': torch.arange(B)[:, None], 'points_neutral': x['points_neutral'],
             'points_posed': x['points_posed'], 'gt_anchors': x['gt_anchors']}
    rec = Recorder(dec)
    drawn = {'randn': [], 'rand': []}
    randn, rand = torch.randn, torch.rand

    def rec_randn(*a, **k):
        t = randn(*a, **k)
        drawn['randn'].append(t.clone())
        return t

    def rec_rand(*a, **k):
        t = rand(*a, **k)
        drawn['rand'].append(t.clone())
        return t
    torch.manual_seed(SEEDS[kind] + 200)
    torch.randn, torch.rand = rec_randn, rec_rand
    try:
        losses = ns.loss_functions.compute_loss_corresp_forward(dict(batch), rec, None, codes, codes_shape, 'cpu')
    finally:
        torch.randn, torch.rand = randn, rand
    total = sum(LAMBDAS[kind][k] * v for k, v in losses.items())
    total.backward()
    assert len(drawn['rand']) == 1 and len(drawn['randn']) == (2 if kind == 'nphm' else 0)
    for k, v in x.items():
        out['%s_%s' % (kind, k)] = v.numpy()
    if kind == 'nphm':
        out[kind + '_noise_corresp'] = (drawn['randn'][0]).numpy()        # raw randn; the reference divides by 200
        out[kind + '_noise_samples'] = (drawn['randn'][1]).numpy()
    out[kind + '_rand_samples'] = drawn['rand'][0].numpy()
    out[kind + '_loss_names'] = np.array(list(losses.keys()))
    out[kind + '_loss_values'] = np.array([float(v) for v in losses.values()], np.float64)
    out[kind + '_loss_total'] = np.float64(float(total))
    out[kind + '_grad_codes'] = codes.weight.grad.numpy()
    out[kind + '_grad_points'] = rec.points[0].grad.numpy()
    names, norms = [], []
    for i, (name, p) in enumerate(dec.named_parameters()):
        g = p.grad.detach().reshape(-1).numpy()
        names.append(name)
        norms.append(float(np.linalg.norm(g.astype(np.float64))))
        out['%s_grad_values_%d' % (kind, i)] = g[positions(g.size, i)]
    out[kind + '_param_names'] = np.array(names)
    out[kind + '_grad_norms'] = np.array(norms)


def main():
    ns = R.load()
    assert ns.loss_functions is not None, 'the reference copy lacks loss_functions.py'
    out = {}
    for kind in ('nphm', 'npm'):
        one(ns, kind, out)
    path = os.path.join(HERE, 'train_corresp.npz')
    np.savez_compressed(path, **out)
    print('wrote %s (%d bytes)' % (path, os.path.getsize(path)))


if __name__ == '__main__':
    main()
