"""Stage-2 training step (the expression / deformation network, reference training_corresp.py:154-176): native vs composite.

One step = ``compute_loss_corresp_forward`` (two decoder forwards: B x 1000 correspondences, B x 100 samples), the weighted
total, ``backward()``, both ``clip_grad_norm_`` calls, AdamW on the decoder and SparseAdam on the expression codes - with
``nphm_b200.set_native_training`` on (layer chain + tcgen05 weight-gradient GEMMs) and off (PyTorch composite).  The two arms
run alternately in one process on identically seeded copies, timed with CUDA events after a synchronise.  The native step
includes re-packing the weights after every optimiser step (``MlpEngine.refresh``, one host synchronise).

    python tools/bench_train_corresp.py [--configs nphm npm] [--steps 200] [--warmup 10] [--out FILE]
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch
import torch.nn as nn

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import nphm_b200  # noqa: E402
from nphm_b200.models.deepSDF import DeepSDF, DeformationNetwork  # noqa: E402
from nphm_b200.models.loss_functions import compute_loss_corresp_forward  # noqa: E402

# scripts/configs/nphm_def.yaml / npm_def.yaml
LAMBDAS = {'nphm': {'corresp': 100.0, 'lat_reg': 5e-5, 'loss_reg_zero': 5e-5},
           'npm': {'corresp': 100.0, 'lat_reg': 5e-5, 'loss_reg_zero': 0.0}}
LR, LR_LAT, GRAD_CLIP = 1e-4, 5e-4, 0.025
WEIGHT_DECAY = {'nphm': 5e-4, 'npm': 1e-5}
ID_DIM = {'nphm': 64 + 40 * 32, 'npm': 512}          # width of the identity code each decoder is conditioned on
EXPR_DIM = 200


def make_setup(kind: str, device, batch_size: int = 32, n_corresp: int = 1000, seed: int = 0):
    """Decoder, codes, optimisers and one fixed batch of the shipped stage-2 shapes (seeded).  Differences from the shipped
    trainer that do not touch the decoder: the batch is synthetic, the anchors are the batch's ``gt_anchors`` (the trainer
    derives them from the identity model's ``mlp_pos`` when it has one), and the expression codes are clipped with
    ``clip_sparse_grad_norm_``."""
    torch.manual_seed(seed)
    if kind == 'nphm':
        dec = DeformationNetwork(mode='compress', lat_dim_expr=EXPR_DIM, lat_dim_id=32, lat_dim_glob_shape=64, lat_dim_loc_shape=32,
                                 n_loc=39, anchors=torch.zeros(1, 39, 3), hidden_dim=512, nlayers=6, out_dim=3, input_dim=3)
    else:                                             # scripts/training/train_corresp.py:71-77
        dec = DeepSDF(lat_dim=512 + EXPR_DIM, hidden_dim=1024, geometric_init=False, out_dim=3, input_dim=3)
    dec = dec.to(device).train()
    codes = nn.Embedding(batch_size, EXPR_DIM, sparse=True).to(device)
    nn.init.normal_(codes.weight, 0.0, 0.01)
    codes_shape = nn.Embedding(batch_size, ID_DIM[kind]).to(device)
    nn.init.normal_(codes_shape.weight, 0.0, 0.05)
    codes_shape.weight.requires_grad_(False)
    pts = (torch.rand(batch_size, n_corresp, 3, device=device) - 0.5) * 1.6
    batch = {'idx': torch.arange(batch_size, device=device)[:, None], 'subj_ind': torch.arange(batch_size, device=device)[:, None],
             'points_neutral': pts, 'points_posed': pts + 0.02 * torch.randn_like(pts),
             'gt_anchors': torch.randn(batch_size, 39, 3, device=device) * 0.3}
    opt = torch.optim.AdamW(dec.parameters(), lr=LR, weight_decay=WEIGHT_DECAY[kind])
    opt_lat = torch.optim.SparseAdam(list(codes.parameters()), lr=LR_LAT)
    return {'kind': kind, 'decoder': dec, 'codes': codes, 'codes_shape': codes_shape, 'batch': batch, 'opt': opt, 'opt_lat': opt_lat,
            'device': device}


def clip_sparse_grad_norm_(params, max_norm: float):
    """``clip_grad_norm_`` for the sparse gradients of the expression codes: this torch's ``clip_grad_norm_`` has no sparse
    norm kernel.  Same rule: scale by max_norm / (total norm + 1e-6) when that is below 1."""
    params = [p for p in params if p.grad is not None]
    if not params:
        return
    grads = [p.grad.coalesce() for p in params]
    total = torch.sqrt(sum(g._values().pow(2).sum() for g in grads))
    coef = torch.clamp(max_norm / (total + 1e-6), max=1.0)
    for g, p in zip(grads, params):
        p.grad = g * coef


def train_step(s, native: bool, step_only_loss: bool = False):
    """One trainer step (training_corresp.py:154-176); returns the loss dict as floats, like the reference."""
    nphm_b200.set_native_training(native)
    s['opt'].zero_grad()
    s['opt_lat'].zero_grad()
    losses = compute_loss_corresp_forward(dict(s['batch']), s['decoder'], None, s['codes'], s['codes_shape'], s['device'])
    total = sum(LAMBDAS[s['kind']][k] * v for k, v in losses.items())
    total.backward()
    if step_only_loss:
        return losses, total
    torch.nn.utils.clip_grad_norm_(s['decoder'].parameters(), max_norm=GRAD_CLIP)
    clip_sparse_grad_norm_(s['codes'].parameters(), max_norm=GRAD_CLIP)
    s['opt'].step()
    s['opt_lat'].step()
    out = {k: v.item() for k, v in losses.items()}
    out['loss'] = total.item()
    return out


def backbone(dec):
    return dec.defDeepSDF if isinstance(dec, DeformationNetwork) else dec


def flops_per_step(s, n_rows: int):
    """Counted from the shapes (not measured): per row, forward 2 sum_l N_l K_l over the point-dependent input columns K_l
    (condition folded into per-query constants; the 32 noise columns ride with xyz), backward the input adjoints
    2 sum_{l>=1} N_l N_{l-1} plus the weight gradients 2 sum_l N_l K_l."""
    net = backbone(s['decoder'])
    lins = [getattr(net, 'lin%d' % i) for i in range(net.num_layers - 1)]
    nd = 32 if isinstance(s['decoder'], DeformationNetwork) else 0
    skip = net.skip_in[0]
    fwd = bwd = 0
    for l, lin in enumerate(lins):
        n = lin.out_features
        k = 3 + nd if l == 0 else (lins[l - 1].out_features + 3 + nd if l == skip else lin.in_features)
        fwd += 2 * n * k
        bwd += 2 * n * k
        if l >= 1:
            bwd += 2 * n * lins[l - 1].out_features
    return {'forward_per_point': fwd, 'forward_backward_per_point': fwd + bwd, 'rows_per_step': n_rows,
            'forward_backward_per_step': (fwd + bwd) * n_rows}


def time_backbone(s, native: bool, iters: int = 50):
    """Backbone forward + backward alone on the B x 1000 correspondence call (weights, condition and points require grad)."""
    net = backbone(s['decoder'])
    dev = s['device']
    B, N = s['batch']['points_neutral'].shape[:2]
    torch.manual_seed(5)
    xyz = s['batch']['points_neutral'].clone().requires_grad_(True)
    cond = (torch.randn(B, net.lat_dim, device=dev) * 0.05).requires_grad_(True)
    noise = torch.randn(B, N, 32, device=dev) / 200 if isinstance(s['decoder'], DeformationNetwork) else None
    up = torch.randn(B, N, net.out_dim_net, device=dev)

    def once():
        if native:
            out = net.forward_native_train(xyz, cond, noise)
        else:
            c = cond[:, None, :].expand(B, N, net.lat_dim)
            if noise is not None:
                c = torch.cat([c[..., :32] + noise, c[..., 32:]], dim=-1)
            out = net._forward_composite(xyz, c)
        torch.autograd.backward(out, up)
    for _ in range(5):
        once()
    torch.cuda.synchronize()
    ts = []
    for _ in range(iters):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        once()
        b.record()
        torch.cuda.synchronize()
        ts.append(a.elapsed_time(b))
    return float(np.median(ts))


def power_limit():
    try:
        return subprocess.run(['nvidia-smi', '--query-gpu=power.limit', '--format=csv,noheader', '-i', str(torch.cuda.current_device())],
                              capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:                            # report, do not guess
        return 'unavailable (%s)' % type(e).__name__


def run(kind: str, steps: int, warmup: int):
    dev = torch.device('cuda:0')
    arms = {'native': make_setup(kind, dev), 'composite': make_setup(kind, dev)}
    times = {'native': [], 'composite': []}
    curves = {'native': [], 'composite': []}
    for i in range(warmup + steps):
        for name in ('native', 'composite'):
            torch.manual_seed(1000 + i)                 # same noise and samples in both arms
            torch.cuda.synchronize()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            out = train_step(arms[name], name == 'native')
            b.record()
            torch.cuda.synchronize()
            if i >= warmup:
                times[name].append(a.elapsed_time(b))
            if i < 10:
                curves[name].append(out['loss'])
    nphm_b200.set_native_training(False)
    B, N = arms['native']['batch']['points_neutral'].shape[:2]
    res = {'config': kind, 'batch_size': B, 'points': [N, 100], 'steps_timed': steps, 'warmup': warmup}
    for name in times:
        t = np.array(times[name])
        res['step_ms_' + name] = {'median': float(np.median(t)), 'p10': float(np.percentile(t, 10)),
                                  'p90': float(np.percentile(t, 90)), 'min': float(t.min()), 'max': float(t.max())}
    res['speedup_median'] = res['step_ms_composite']['median'] / res['step_ms_native']['median']
    res['loss_first10_native'] = curves['native']
    res['loss_first10_composite'] = curves['composite']
    res['backbone_fwd_bwd_ms_native'] = time_backbone(arms['native'], True)
    res['backbone_fwd_bwd_ms_composite'] = time_backbone(arms['composite'], False)
    res['flops_counted'] = flops_per_step(arms['native'], B * (N + 100))
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--configs', nargs='+', default=['nphm', 'npm'], choices=['nphm', 'npm'])
    ap.add_argument('--steps', type=int, default=200)
    ap.add_argument('--warmup', type=int, default=10)
    ap.add_argument('--out', default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('bench_train_corresp: no CUDA device (this measurement needs a B200)')
    result = {'device': torch.cuda.get_device_name(0), 'power_limit': power_limit(),
              'tf32_matmul': bool(torch.backends.cuda.matmul.allow_tf32), 'torch': torch.__version__,
              'results': [run(k, args.steps, args.warmup) for k in args.configs]}
    text = json.dumps(result, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, 'w') as f:
            f.write(text + '\n')


if __name__ == '__main__':
    main()
