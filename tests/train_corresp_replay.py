"""Replay of tests/golden/train_corresp.npz (tests/golden/make_golden_train_corresp.py) on this package: one stage-2 training step,
``compute_loss_corresp_forward`` + weighted total + ``backward()``, with the random numbers the reference drew injected (the
per-point noise through ``deepSDF.condition_noise``, the samples' ``torch.rand``).  Shared by the CPU test (composite path)
and the GPU test (native path)."""
import hashlib
import os
import sys

import numpy as np
import torch

from conftest import load_golden, mean_anchors

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, 'golden'))
import make_golden_train_corresp as G  # noqa: E402  (constants and the position rule; it imports the reference lazily)


def _sha(t):
    a = np.ascontiguousarray(t.detach().cpu().numpy())
    return hashlib.sha256(('%s%s' % (a.dtype, a.shape)).encode() + a.tobytes()).hexdigest()


def make_decoder(kind):
    from nphm_b200.models.deepSDF import DeepSDF, DeformationNetwork
    torch.manual_seed(G.SEEDS[kind])
    if kind == 'nphm':
        return DeformationNetwork(mode='compress', lat_dim_expr=200, lat_dim_id=32, lat_dim_glob_shape=64, lat_dim_loc_shape=32,
                                  n_loc=39, anchors=mean_anchors(), hidden_dim=512, nlayers=6, out_dim=3, input_dim=3).train()
    return DeepSDF(lat_dim=712, hidden_dim=1024, geometric_init=False, out_dim=3, input_dim=3).train()


def replay(kind, device, monkeypatch):
    """-> (golden, losses dict of floats, total, {'params': [grad tensors], 'codes': grad, 'points': grad})"""
    from nphm_b200.models import deepSDF
    from nphm_b200.models.loss_functions import compute_loss_corresp_forward
    g = load_golden('train_corresp.npz')
    dec = make_decoder(kind)
    sd = dec.state_dict()
    assert list(sd.keys()) == list(g[kind + '_keys'])
    assert [_sha(v) for v in sd.values()] == list(g[kind + '_sha256'])      # same initialisation as the reference class
    dec = dec.to(device)
    B = G.B
    codes = torch.nn.Embedding(B, 200).to(device)
    codes_shape = torch.nn.Embedding(B, G.ID_DIM[kind]).to(device)
    with torch.no_grad():
        codes.weight.copy_(torch.from_numpy(g[kind + '_codes']))
        codes_shape.weight.copy_(torch.from_numpy(g[kind + '_codes_shape']))
    codes_shape.weight.requires_grad_(False)
    t = lambda name: torch.from_numpy(g['%s_%s' % (kind, name)]).to(device)
    batch = {'idx': torch.arange(B, device=device)[:, None], 'subj_ind': torch.arange(B, device=device)[:, None],
             'points_neutral': t('points_neutral'), 'points_posed': t('points_posed'), 'gt_anchors': t('gt_anchors')}
    noise = [t('noise_corresp'), t('noise_samples')] if kind == 'nphm' else []
    rand = [t('rand_samples')]

    def fake_noise(shape, dev):
        raw = noise.pop(0)
        assert tuple(shape) == tuple(raw.shape)
        return raw.to(dev) / 200                                             # the reference's randn(...) / 200

    def fake_rand(*shape, **kw):
        raw = rand.pop(0)
        assert tuple(shape) == tuple(raw.shape)
        return raw.to(kw.get('device') or device)
    rec = G.Recorder(dec)
    with monkeypatch.context() as m:
        m.setattr(deepSDF, 'condition_noise', fake_noise)
        m.setattr(torch, 'rand', fake_rand)
        losses = compute_loss_corresp_forward(dict(batch), rec, None, codes, codes_shape, device)
    assert not noise and not rand                                           # every recorded draw was consumed
    total = sum(G.LAMBDAS[kind][k] * v for k, v in losses.items())
    total.backward()
    grads = {'params': [p.grad.detach().cpu() for p in dec.parameters()], 'codes': codes.weight.grad.detach().cpu(),
             'points': rec.points[0].grad.detach().cpu()}
    return g, {k: v.item() for k, v in losses.items()}, total.item(), grads


def compare(kind, g, losses, total, grads):
    """-> dict of relative deviations: losses (relative), gradient samples and full code / point gradients (per tensor,
    relative to max |ref|), gradient norms (relative)."""
    dev = {}
    for name, ref in zip(g[kind + '_loss_names'], g[kind + '_loss_values']):
        dev['loss ' + str(name)] = abs(losses[str(name)] - ref) / abs(ref)
    dev['loss total'] = abs(total - float(g[kind + '_loss_total'])) / abs(float(g[kind + '_loss_total']))
    for i, name in enumerate(g[kind + '_param_names']):
        got = grads['params'][i].reshape(-1).double().numpy()
        ref = g['%s_grad_values_%d' % (kind, i)].astype(np.float64)
        dev['grad %s' % name] = float(np.abs(got[G.positions(got.size, i)] - ref).max() / max(np.abs(ref).max(), 1e-30))
        ref_n = float(g[kind + '_grad_norms'][i])
        dev['norm %s' % name] = abs(float(np.linalg.norm(got)) - ref_n) / max(ref_n, 1e-30)
    for key in ('codes', 'points'):
        ref = g['%s_grad_%s' % (kind, key)].astype(np.float64)
        dev['grad ' + key] = float(np.abs(grads[key].double().numpy() - ref).max() / np.abs(ref).max())
    return dev
