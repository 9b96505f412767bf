"""Identity-space training / validation losses of the reference, ``NPHM.models.loss_functions``:

  * ``compute_loss``         src/NPHM/models/loss_functions.py:7-17
  * ``actual_compute_loss``  src/NPHM/models/loss_functions.py:20-110   (SURVEY.md 8f-3)
  * ``compute_loss_corresp_forward``  src/NPHM/models/loss_functions.py:282-322  (stage-2 expression training)

Same inputs (a batch dict with ``points_face``, ``points_non_face``, ``sup_grad_far``, ``sup_grad_near``, the normals and
``gt_anchors``), same returned dict (``surf_sdf``, ``normals``, ``space_sdf``, ``grad``, ``lat_reg`` and - for the
ensemble - ``anchors``, ``symm_dist``, ``middle_dist``).  Two ways to get the SDF values and their spatial gradient:

  * **native** (no autograd graph: validation, monitoring, loss curves of a frozen model): one call per batch element and
    point set into ``nphm_ensemble_backward_inputs`` with an upstream gradient of ones - a point's SDF depends on its own
    coordinates only, so that vector-Jacobian product IS the per-point spatial gradient (tcgen05 forward and backward,
    ``csrc/fit.cu``).  Used when autograd is not recording (the reference cannot evaluate these losses at all under
    ``torch.no_grad()``: its ``gradient`` needs a graph) or with ``native=True``; training-mode forward only.
  * **composite** (training): the decoder's autograd path and ``diff_operators.gradient`` with ``create_graph=True`` -
    weight gradients of the normal / eikonal terms need the double backward, which stays in PyTorch.

This module is NOT installed over ``NPHM.models.loss_functions`` by ``install_as_nphm`` (the reference's own file keeps
working on top of the drop-in decoder); import it explicitly.
"""
from __future__ import annotations

import torch

from .EnsembledDeepSDF import FastEnsembleDeepSDFMirrored
from .diff_operators import gradient

_POINT_SETS = ('points_face', 'points_non_face', 'sup_grad_near', 'sup_grad_far')


def compute_loss(batch, decoder, latent_codes, device, native=None):
    """Moves the batch to ``device``, looks the latent codes up by ``batch['idx']`` and evaluates the losses."""
    batch = {k: v for k, v in batch.items() if k != 'path'}
    on_device = {k: v.to(device).float() for k, v in batch.items()}
    glob_cond = latent_codes(batch['idx'].to(device))
    return actual_compute_loss(on_device, decoder, glob_cond, native=native)


def _native_values_and_gradients(decoder, points, glob_cond):
    """points B x N x 3, glob_cond B x 1 x lat_dim -> (sdf B x N x 1, d sdf / d x  B x N x 3), no graph."""
    engine = decoder.engine()
    sdf, grad = [], []
    for b in range(points.shape[0]):
        pts = points[b].contiguous()
        ones = torch.ones(pts.shape[0], device=pts.device, dtype=torch.float32)
        s, _, g = engine.backward_inputs(pts, glob_cond[b].reshape(-1), ones)
        sdf.append(s)
        grad.append(g)
    return torch.stack(sdf)[..., None], torch.stack(grad)


def _composite_values_and_gradients(decoder, points, glob_cond, anchor_preds):
    pts = points.clone().detach().requires_grad_()
    pred, anchors = decoder(pts, glob_cond.repeat(1, pts.shape[1], 1), anchor_preds)
    return pred, gradient(pred, pts), anchors


def _pair_distance(latents):
    """mean over (batch, pairs) of || z_{2i} - z_{2i+1} ||; an odd trailing block is ignored (reference :84-87)."""
    n = latents.shape[1] - latents.shape[1] % 2
    return torch.norm(latents[:, 0:n:2, :] - latents[:, 1:n:2, :], dim=-1).mean()


def actual_compute_loss(batch_cuda, decoder, glob_cond, native=None):
    is_ensemble = isinstance(decoder, FastEnsembleDeepSDFMirrored)
    anchor_preds = batch_cuda['gt_anchors'] if hasattr(decoder, 'anchors') else None
    if native is None:
        native = not torch.is_grad_enabled()
    native = bool(native) and is_ensemble and decoder.training and batch_cuda['points_face'].is_cuda

    pred, grad, anchors = {}, {}, None
    if native:
        with torch.no_grad():
            for name in _POINT_SETS:
                pred[name], grad[name] = _native_values_and_gradients(decoder, batch_cuda[name], glob_cond)
            anchors = decoder.engine().anchors(glob_cond[:, 0, :])
    else:
        with torch.enable_grad():
            for name in _POINT_SETS:
                pred[name], grad[name], a = _composite_values_and_gradients(decoder, batch_cuda[name], glob_cond, anchor_preds)
                if name != 'sup_grad_far':
                    anchors = a                      # the reference keeps the anchors of its third call (sup_grad_near)

    # geometry terms
    sdf_face = pred['points_face'].abs().squeeze()
    sdf_outer = pred['points_non_face'].abs().squeeze()
    normal_face = (grad['points_face'] - batch_cuda['normals_face']).norm(2, dim=-1)
    normal_outer = torch.clamp((grad['points_non_face'] - batch_cuda['normals_non_face']).norm(2, dim=-1), None, 0.75) / 2
    eikonal = torch.cat([(grad[name].norm(dim=-1) - 1).abs()
                         for name in ('points_face', 'points_non_face', 'sup_grad_far', 'sup_grad_near')], dim=-1)
    space_sdf = torch.exp(-1e1 * pred['sup_grad_far'].abs())

    losses = {'surf_sdf': torch.cat([sdf_face, sdf_outer], dim=-1).mean(),
              'normals': torch.cat([normal_face.squeeze(), normal_outer.squeeze()], dim=-1).mean(),
              'space_sdf': space_sdf.mean(),
              'grad': eikonal.mean(),
              'lat_reg': (torch.norm(glob_cond, dim=-1) ** 2).mean()}
    if anchors is None:
        return losses

    symm_dist = middle_dist = None
    if hasattr(decoder, 'lat_dim_glob'):
        z = glob_cond.squeeze(1)
        G, L, n_symm = decoder.lat_dim_glob, decoder.lat_dim_loc, decoder.num_symm_pairs
        symm = z[:, G:G + 2 * n_symm * L].view(z.shape[0], 2 * n_symm, L)
        middle = z[:, G + 2 * n_symm * L:-L].view(z.shape[0], decoder.num_kps - 2 * n_symm, L)
        symm_dist = _pair_distance(symm)
        middle_dist = _pair_distance(middle)
    losses['anchors'] = (anchors - batch_cuda['gt_anchors']).square().mean()
    losses['symm_dist'] = symm_dist
    losses['middle_dist'] = middle_dist
    return losses


def compute_loss_corresp_forward(batch, decoder, decoder_shape, latent_codes, latent_codes_shape, device, epoch=-1,
                                 exp_path=None):
    """Stage-2 training loss of the deformation network (same signature and returned dict as the reference): squared error of
    the posed correspondences, the expression-code magnitude, and the deformation of 100 uniform samples per query in
    [-1.25, 1.25)^3 pushed towards zero.  ``epoch`` and ``exp_path`` are unused, as in the reference.  Both decoder calls
    see a per-query-constant condition, so with :func:`nphm_b200.set_native_training` on they run natively."""
    batch.pop('path', None)
    on_device = {k: v.to(device).float() for k, v in batch.items()}
    cond_shape = latent_codes_shape(batch['subj_ind'].to(device))
    cond_pose = latent_codes(batch['idx'].to(device))
    if decoder_shape is not None and decoder_shape.mlp_pos is not None:
        anchors = decoder_shape.mlp_pos(cond_shape[..., :decoder_shape.lat_dim_glob]).view(cond_pose.shape[0], -1, 3)
        anchors += decoder.anchors.squeeze(0)
    else:
        anchors = on_device['gt_anchors']
    glob_cond = torch.cat([cond_shape, cond_pose], dim=-1)
    points = on_device['points_neutral'].clone().detach().requires_grad_()
    cond = glob_cond.repeat(1, points.shape[1], 1)
    delta, _ = decoder(points, cond, anchors)
    corresp = (points + delta.squeeze() - on_device['points_posed'][:, :, :3]) ** 2
    samples = (torch.rand(cond.shape[0], 100, 3, device=cond.device, dtype=cond.dtype) - 0.5) * 2.5
    delta_samples, _ = decoder(samples, cond[:, :100, :], anchors)
    return {'corresp': corresp.mean(),
            'lat_reg': (torch.norm(cond_pose, dim=-1) ** 2).mean(),
            'loss_reg_zero': (delta_samples ** 2).mean()}
