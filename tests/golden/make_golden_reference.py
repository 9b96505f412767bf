#!/usr/bin/env python
"""Generate reference_parity.npz and losses.npz: what the UNMODIFIED reference modules return on the inputs of
tests/test_gpu_reference.py, tests/test_gpu_losses.py and tests/test_losses_cpu.py, so that those tests compare
against stored outputs and need no reference checkout.

    python oracle/make_ref.py                      # reference modules -> oracle/_ref (NPHM_REFERENCE_ROOT=<checkout>)
    python tests/golden/make_golden_reference.py

torch on the CPU, fp32 (the reference's own dtype), weights and inputs seeded exactly as the tests make them.
Whole volumes would not fit a fixture, so outputs are sampled: every chunk-boundary index of the chunked
``get_logits`` (where eval mode forces the chunk's last point outside, EnsembledDeepSDF.py:260-261) and the index
before it, plus a seeded uniform sample.  Weights are not stored; a per-tensor SHA-256 pins them instead."""
import hashlib
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
from oracle import ref_loader as R        # noqa: E402

MINI = [-.55, -.5, -.95]
MAXI = [0.55, 0.75, 0.4]


def tensor_sha256(t):
    a = np.ascontiguousarray(t.detach().cpu().numpy())
    return hashlib.sha256(('%s%s' % (a.dtype, a.shape)).encode() + a.tobytes()).hexdigest()


def pin_state(out, prefix, module):
    sd = module.state_dict()
    out[prefix + '_keys'] = np.array(list(sd.keys()))
    out[prefix + '_sha256'] = np.array([tensor_sha256(v) for v in sd.values()])


def chunk_ends(total, nb):
    return np.concatenate([np.arange(nb - 1, total, nb), [total - 1]])


def sample(total, n, seed, exclude=()):
    idx = np.random.default_rng(seed).choice(total, n + len(exclude), replace=False)
    return np.sort(idx[~np.isin(idx, exclude)][:n]).astype(np.int64)


def grid(ns, res):
    g = ns.utils_reconstruction.create_grid_points_from_bounds(MINI, MAXI, res)
    return torch.from_numpy(g).float().reshape(1, -1, 3)                # fitting_pointclouds.py:168-170


def eval_logits_at(ns, dec, lat, pts, ends):
    """``get_logits(dec, lat, pts, nb)`` of an eval-mode decoder without the other points of the volume: the value of
    a point depends only on the point and on whether it ends its chunk.  ``ends`` marks the points that do; they are
    evaluated as the second point of 2-point chunks, the others inside chunks that end in a discarded copy."""
    out = np.empty(pts.shape[1], np.float32)
    e = np.flatnonzero(ends)
    if len(e):
        pairs = pts[:, np.repeat(e, 2)]
        out[e] = ns.reconstruction.get_logits(dec, lat, pairs, nbatch_points=2)[1::2]
    rest = np.flatnonzero(~ends)
    for s in range(0, len(rest), 20000):
        part = rest[s:s + 20000]
        p = pts[:, np.append(part, part[-1])]
        out[part] = ns.reconstruction.get_logits(dec, lat, p, nbatch_points=len(part) + 1)[:-1]
    return out


def parity(ns):
    out = {}
    lat = R.sample_latent(ns, 1)
    pin_state(out, 'ensemble', R.make_ensemble(ns, 0))
    pin_state(out, 'deform', R.make_deformation(ns))

    # configs[0]: 64^3, get_logits in eval and train mode, two chunk sizes
    total = 64 ** 3
    g64 = grid(ns, 64)
    ends = np.union1d(chunk_ends(total, 25000), chunk_ends(total, 20000))
    idx = np.union1d(np.union1d(ends, ends - 1), sample(total, 2048, 0))
    out['c1_idx'] = idx.astype(np.int32)
    dec = R.make_ensemble(ns, 0)
    for train in (False, True):
        dec.train(train)
        for nb in (25000, 20000):
            want = ns.reconstruction.get_logits(dec, lat, g64, nbatch_points=nb)
            assert want.shape == (total,) and want.dtype == np.float32
            out['c1_%s_%d' % ('train' if train else 'eval', nb)] = want[idx]

    # configs[1]: 256^3 eval volume of the benchmark step, chunks of 25 000
    res, nb = 256, 25000
    total = res ** 3
    g256 = grid(ns, res)
    dec.eval()
    last = chunk_ends(total, nb)
    out['c2_last'] = eval_logits_at(ns, dec, lat, g256[:, last], np.ones(len(last), bool))
    out['c2_before_last'] = eval_logits_at(ns, dec, lat, g256[:, last - 1], np.zeros(len(last), bool))
    idx = sample(total, 4096, 1, exclude=last)
    out['c2_idx'] = idx.astype(np.int32)
    out['c2_at_idx'] = eval_logits_at(ns, dec, lat, g256[:, idx], np.zeros(len(idx), bool))
    # drop-in get_logits on explicit points: slabs of 2 chunks + a ragged 7-point chunk
    firsts = [0, 24000, total // 2 - 12345, total - 2216 - nb]
    out['c2_slab_first'] = np.array(firsts)
    for k, f in enumerate(firsts):
        pts = g256[:, f:f + 2 * nb + 7]                          # the last one ends with the grid: 25 000 + 2216 points
        n = pts.shape[1]
        ends = chunk_ends(n, nb)
        rel = np.union1d(np.union1d(ends, ends - 1), np.append(sample(n, 512, 2 + k), 0))
        out['c2_slab%d_idx' % k] = rel.astype(np.int32)
        out['c2_slab%d' % k] = ns.reconstruction.get_logits(dec, lat, pts, nbatch_points=nb)[rel]

    # configs[2]: deformation field on the 64^3 grid, identity field (train mode) at the deformed points
    dfn = R.make_deformation(ns)
    torch.manual_seed(3)
    lat_ex = torch.randn(200) * 0.01
    cond = torch.cat([lat, lat_ex]).reshape(1, 1, -1)
    idx = sample(64 ** 3, 2048, 3)
    with torch.no_grad():
        _, anchors = dec(g64[:, :1], lat.reshape(1, 1, -1), None)
        n = g64.shape[1]
        off = torch.cat([dfn(g64[:, s:s + 50000], cond.repeat(1, min(50000, n - s), 1), anchors)[0]
                         for s in range(0, n, 50000)], dim=1)
        warped = (g64 + off)[:, idx]
        dec.train()
        sdf = dec(warped, lat.reshape(1, 1, -1).repeat(1, len(idx), 1), None)[0]
    out['c3_anchors'] = anchors.numpy()
    out['c3_idx'] = idx.astype(np.int32)
    out['c3_offsets'] = off[0, idx].numpy()
    out['c3_sdf'] = sdf.reshape(-1).numpy()

    # get_logits_backward (reconstruction.py:28-56) with a DeepSDF expression decoder on the 24^3 grid, chunks of 5000
    torch.manual_seed(31)
    ex = ns.deepSDF.DeepSDF(lat_dim=100, hidden_dim=128, nlayers=6, out_dim=3).eval()
    pin_state(out, 'expr', ex)
    dec.eval()
    torch.manual_seed(32)
    lat_ex = torch.randn(1, 1, 100) * 0.1
    g24 = grid(ns, 24)
    total = g24.shape[1]
    want, anc = ns.reconstruction.get_logits_backward(dec, ex, lat.reshape(1, 1, -1), lat_ex, g24, nbatch_points=5000,
                                                      return_anchors=True)
    want0 = ns.reconstruction.get_logits_backward(dec, ex, lat.reshape(1, 1, -1), None, g24, nbatch_points=5000)
    ends = chunk_ends(total, 5000)
    idx = np.union1d(np.union1d(ends, ends - 1), sample(total, 3072, 4))
    out['bw_shape'] = np.array(want.shape)
    out['bw_idx'] = idx.astype(np.int32)
    out['bw_want'] = want[idx]
    out['bw_want0'] = want0[idx]
    out['bw_anchors'] = anc.numpy()
    return out


def cpu_loss_batch():
    """The batch of test_losses_cpu.py."""
    rng = np.random.RandomState(11)
    B, n = 2, 40

    def pts(scale):
        return torch.from_numpy((rng.randn(B, n, 3) * scale).astype(np.float32))
    batch = {'points_face': pts(0.12), 'points_non_face': pts(0.2), 'sup_grad_near': pts(0.15), 'sup_grad_far': pts(0.4),
             'normals_face': pts(1.0), 'normals_non_face': pts(1.0), 'gt_anchors': pts(0.1)[:, :39]}
    batch['gt_anchors'] = torch.from_numpy((rng.randn(B, 39, 3) * 0.1).astype(np.float32))
    cond = torch.from_numpy((rng.randn(B, 1, 1344) * 0.3).astype(np.float32)).requires_grad_()
    return batch, cond


def gpu_loss_batch():
    """The batch of test_gpu_losses.py."""
    rng = np.random.RandomState(5)
    B, n = 3, 700

    def pts(scale):
        return torch.from_numpy((rng.randn(B, n, 3) * scale + np.array([0.0, 0.05, -0.1])).astype(np.float32))

    def unit():
        v = rng.randn(B, n, 3).astype(np.float32)
        return torch.from_numpy(v / np.linalg.norm(v, axis=-1, keepdims=True))
    batch = {'points_face': pts(0.12), 'points_non_face': pts(0.2), 'sup_grad_near': pts(0.15), 'sup_grad_far': pts(0.4),
             'normals_face': unit(), 'normals_non_face': unit(),
             'gt_anchors': torch.from_numpy((rng.randn(B, 39, 3) * 0.1).astype(np.float32))}
    cond = torch.from_numpy((rng.randn(B, 1, 1344) * 0.3).astype(np.float32))
    return batch, cond


def losses(ns):
    out = {}
    ref = R.make_ensemble(ns, 0).train()
    batch, cond = cpu_loss_batch()
    want = ns.loss_functions.actual_compute_loss(batch, ref, cond)
    out['cpu_keys'] = np.array(sorted(want))
    for k in want:
        out['cpu_' + k] = np.float64(want[k].detach())
    total = sum(want[k] for k in ('surf_sdf', 'normals', 'grad'))
    gw = torch.autograd.grad(total, ref.ensembled_deep_sdf.lin1.weight)[0].reshape(-1).numpy()
    idx = np.union1d(np.argsort(-np.abs(gw))[:1024], sample(gw.size, 4096, 5))
    out['cpu_grad_lin1_shape'] = np.array(ref.ensembled_deep_sdf.lin1.weight.shape)
    out['cpu_grad_lin1_absmax'] = np.float64(np.abs(gw).max())
    out['cpu_grad_lin1_idx'] = idx.astype(np.int32)
    out['cpu_grad_lin1'] = gw[idx]
    batch, cond = gpu_loss_batch()
    want = ns.loss_functions.actual_compute_loss(batch, ref, cond)
    out['gpu_keys'] = np.array(sorted(want))
    for k in want:
        out['gpu_' + k] = np.float64(want[k].detach())
    return out


def main():
    torch.set_num_threads(os.cpu_count())
    ns = R.load()
    np.savez_compressed(os.path.join(HERE, 'losses.npz'), **losses(ns))
    np.savez_compressed(os.path.join(HERE, 'reference_parity.npz'), **parity(ns))


if __name__ == '__main__':
    main()
