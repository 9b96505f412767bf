"""Drop-in mirror of the reference module ``NPHM.models.deepSDF``.

Reference interface (file:line):
  * ``DeepSDF``              src/NPHM/models/deepSDF.py:6-89
  * ``sample_point_feature`` src/NPHM/models/deepSDF.py:92-115 (duplicate of the ensemble one)
  * ``DeformationNetwork``   src/NPHM/models/deepSDF.py:118-239

Parameter names (``lin{i}.weight/bias``, ``compressor.0.*``, ``defDeepSDF.lin{i}.*``) and
constructor signatures are those of the reference so checkpoints load with ``strict=True``.
As in :mod:`.EnsembledDeepSDF`, CUDA no-grad calls with a per-query-constant condition run in
the native sm_100a MLP kernel.  With :func:`nphm_b200.set_native_training` on, forwards that autograd
records run natively as well (:class:`_NativeTrain`: first order only); everything else uses a
PyTorch composite that keeps autograd.
"""
from __future__ import annotations

import math
from typing import Optional

import numpy as np
import torch
import torch.nn as nn
from torch.autograd.function import once_differentiable

from .. import _native
from . import _composite
from .EnsembledDeepSDF import sample_point_feature  # same function in the reference (:92-115)

_SQRT2 = math.sqrt(2.0)


def condition_noise(shape, device) -> torch.Tensor:
    """Training-mode noise on the compressed identity code (reference deepSDF.py:220-221).  Both the composite and the
    native path draw it here, with the same call, so that seeded runs of either see the same numbers."""
    return torch.randn(shape, device=device) / 200


class _NativeTrain(torch.autograd.Function):
    """Backbone forward on [xyz | cond_q + (noise, 0)] with native first-order backward (nphm_mlp_forward_train /
    nphm_mlp_backward_train).  Inputs: backbone module, xyz B x N x 3, per-query condition B x lat_dim, noise B x N x k or None,
    then the weights and biases of every layer (saved, so that an in-place change before the backward is caught)."""

    @staticmethod
    def forward(ctx, backbone, xyz, cond, noise, *params):
        eng = backbone.engine()
        out, ws = eng.forward_train(xyz, cond, noise)
        ctx.eng, ctx.ws, ctx.noise = eng, ws, noise
        ctx.save_for_backward(xyz, cond, *params)
        return out

    @staticmethod
    def backward(ctx, grad_out):
        if torch.is_grad_enabled():
            raise RuntimeError('the native training backward is first order only (create_graph=True asks for more): switch it '
                               'off with nphm_b200.set_native_training(False) for losses that differentiate twice')
        return _native_train_backward(ctx, grad_out)


@once_differentiable
def _native_train_backward(ctx, grad_out):
    if ctx.ws is None:
        raise RuntimeError('a native training forward can be differentiated once: its workspace is released by the first '
                           'backward (retain_graph=True is not supported with nphm_b200.set_native_training(True))')
    xyz, cond, *params = ctx.saved_tensors             # raises if a weight was modified in place since the forward
    need = ctx.needs_input_grad
    gw, gb, g_cond, g_xyz = ctx.eng.backward_train(xyz, cond, ctx.noise, ctx.ws, grad_out, want_w=need[4::2],
                                                   want_b=need[5::2], want_cond=need[2], want_xyz=need[1])
    ctx.ws = None                                      # the workspace (activations of the whole batch) goes with the first backward
    grads = [g for pair in zip(gw, gb) for g in pair]
    return (None, g_xyz, g_cond, None, *grads)


class DeepSDF(nn.Module):
    """Plain DeepSDF MLP: ``[xyz(+posenc) | latent] -> hidden x nlayers -> out_dim`` with the input
    re-injected (and the sum scaled by 1/sqrt(2)) at layer ``nlayers // 2``."""

    def __init__(
            self,
            lat_dim,
            hidden_dim,
            nlayers=8,
            geometric_init=True,
            radius_init=1,
            beta=100,
            out_dim=1,
            num_freq_bands=None,
            input_dim=3,
    ):
        super().__init__()
        d_spatial = input_dim if num_freq_bands is None else input_dim * (2 * num_freq_bands + 1)
        d_in = lat_dim + d_spatial
        self.lat_dim = lat_dim
        self.input_dim = input_dim
        self.out_dim_net = out_dim
        widths = [d_in] + [hidden_dim] * nlayers + [out_dim]
        self.num_layers = len(widths)
        self.skip_in = [nlayers // 2]
        self.num_freq_bands = num_freq_bands
        if num_freq_bands is not None:
            self.freq_bands = 2 ** torch.arange(num_freq_bands)

        for layer in range(self.num_layers - 1):
            fan_out = widths[layer + 1] - (d_in if layer + 1 in self.skip_in else 0)
            lin = nn.Linear(widths[layer], fan_out)
            if geometric_init and layer == self.num_layers - 2:
                # sphere-like initialisation of the output layer (reference :47-53)
                nn.init.normal_(lin.weight, mean=np.sqrt(np.pi) / np.sqrt(widths[layer]), std=0.00001)
                nn.init.constant_(lin.bias, -radius_init)
            setattr(self, 'lin' + str(layer), lin)

        self.beta = beta
        self.activation = nn.Softplus(beta=beta) if beta > 0 else nn.ReLU()
        self._engine = None

    def engine(self) -> "_native.MlpEngine":
        if self._engine is None:
            self._engine = _native.MlpEngine(self)
        self._engine.refresh(self)
        return self._engine

    def _fused_ok(self, xyz, lat_rep) -> bool:
        if not xyz.is_cuda or self.num_freq_bands is not None or self.beta != 100:
            return False
        n_lin = self.num_layers - 1
        hidden = _native.hidden_width(self, n_lin)
        if self.out_dim_net > 8 or not _native.stack_supported(n_lin - 1, hidden, self.lat_dim):
            return False             # depths the native stack builder rejects: PyTorch composite path
        if torch.is_grad_enabled() and (xyz.requires_grad or lat_rep.requires_grad
                                        or any(p.requires_grad for p in self.parameters())):
            return False
        return xyz.dtype == torch.float32 and xyz.dim() == 3

    def _native_train_ok(self, xyz, lat_rep) -> bool:
        """A training forward (autograd recording, something requires grad) the native path takes; the condition must still
        be constant per query (checked by the caller)."""
        if not _native.native_training() or not torch.is_grad_enabled():
            return False
        if not (xyz.requires_grad or lat_rep.requires_grad or any(p.requires_grad for p in self.parameters())):
            return False
        if not (xyz.is_cuda and lat_rep.is_cuda and xyz.dtype == torch.float32 and lat_rep.dtype == torch.float32
                and xyz.dim() == 3 and xyz.shape[-1] == 3 and xyz.shape[1] > 0 and lat_rep.dim() == 3
                and lat_rep.shape[0] == xyz.shape[0]):
            return False
        if self.num_freq_bands is not None or self.beta != 100 or self.out_dim_net > 8:
            return False
        n_lin = self.num_layers - 1
        if not _native.stack_supported(n_lin - 1, _native.hidden_width(self, n_lin), self.lat_dim):
            return False
        return 1 <= self.skip_in[0] < n_lin - 1           # chain_ready's skip constraint (csrc/mlp_chain.cu)

    def forward_native_train(self, xyz, cond, noise=None):
        """xyz B x N x 3, cond B x lat_dim (per query), noise B x N x k or None -> B x N x out_dim, native backward."""
        params = []
        for i in range(self.num_layers - 1):
            lin = getattr(self, 'lin%d' % i)
            params += [lin.weight, lin.bias]
        return _NativeTrain.apply(self, xyz, cond, noise, *params)

    def forward(self, xyz, lat_rep, anchors=None):
        if self._native_train_ok(xyz, lat_rep):
            cond = _native.constant_latent_rows(lat_rep)
            if cond is not None:
                return self.forward_native_train(xyz, cond), None
        if self._fused_ok(xyz, lat_rep):
            cond = _native.constant_latent_rows(lat_rep)
            if cond is not None:
                return self.engine().query(xyz, cond), None
        return self._forward_composite(xyz, lat_rep), None

    def _forward_composite(self, xyz, lat_rep):
        if self.num_freq_bands is not None:
            feats = [xyz]
            for freq in self.freq_bands:
                feats += [torch.sin(xyz * freq), torch.cos(xyz * freq)]
            xyz = torch.cat(feats, dim=-1)
        if lat_rep.shape[-2] == 1 and xyz.shape[-2] != 1:
            lat_rep = lat_rep.expand(*xyz.shape[:-1], lat_rep.shape[-1])
        layers = [getattr(self, 'lin%d' % i) for i in range(self.num_layers - 1)]
        return _composite.skip_mlp(torch.cat([xyz, lat_rep], dim=-1), layers, self.skip_in, self.activation)


def _input_jacobian(backbone: DeepSDF, xyz, cond):
    """Forward-mode derivative of the backbone output w.r.t. ``xyz`` (the condition does not depend on the point):
    returns ``(out  ... x out_dim,  J  ... x out_dim x 3)``.  Same function as three reverse-mode passes through
    :meth:`DeepSDF._forward_composite` (what the reference's ``jac`` does, diff_operators.py:26-54) at a third of the
    launches: the three tangents ride through the layers as one batched matmul,
    ``T_{l+1} = sigmoid(beta z_l) * (T_l W_l^T)``."""
    if cond.shape[-2] == 1 and xyz.shape[-2] != 1:
        cond = cond.expand(*xyz.shape[:-1], cond.shape[-1])
    inp = torch.cat([xyz, cond], dim=-1)
    h, T = inp, None
    last = backbone.num_layers - 2
    for layer in range(last + 1):
        lin = getattr(backbone, 'lin' + str(layer))
        W = lin.weight
        if layer in backbone.skip_in:
            wh = h.shape[-1]
            h = torch.cat([h, inp], dim=-1) / _SQRT2
            dz = (torch.matmul(T, W[:, :wh].t()) + W[:, wh:wh + 3].t()) / _SQRT2
        elif T is None:
            dz = W[:, :3].t().expand(*xyz.shape[:-1], 3, W.shape[0])
        else:
            dz = torch.matmul(T, W.t())
        z = lin(h)
        if layer < last:
            h = backbone.activation(z)
            T = torch.sigmoid(backbone.beta * z).unsqueeze(-2) * dz
        else:
            return z, dz.transpose(-1, -2)


class DeformationNetwork(nn.Module):
    """Forward deformation field F_ex(x; z_ex, z_id): canonical point -> offset.

    ``mode='compress'`` (the shipped configuration, ``scripts/configs/nphm_def.yaml``) conditions a
    :class:`DeepSDF` backbone on ``[Linear([z_id | anchors]) (32) | z_ex]``; the other four modes of the
    reference are kept for API completeness (composite path only)."""

    def __init__(
            self,
            mode,
            lat_dim_expr,
            lat_dim_id,
            lat_dim_glob_shape,
            lat_dim_loc_shape,
            n_loc,
            anchors,
            hidden_dim,
            nlayers=8,
            out_dim=1,
            input_dim=3,
    ):
        super().__init__()
        self.mode = mode
        self.lat_dim_glob_shape = lat_dim_glob_shape
        self.lat_dim_loc_shape = lat_dim_loc_shape
        self.lat_dim_expr = lat_dim_expr
        self.input_dim = input_dim
        self.num_kps = n_loc
        self.out_dim = out_dim + 1

        if mode == 'glob_only':
            self.lat_dim = lat_dim_glob_shape + lat_dim_expr
        elif mode == 'expr_only':
            self.lat_dim = lat_dim_expr
        elif mode == 'interpolate':
            self.lat_dim = lat_dim_glob_shape + lat_dim_expr + lat_dim_loc_shape
        elif mode == 'compress':
            self.lat_dim = lat_dim_expr + lat_dim_id
            self.compressor = nn.Sequential(
                nn.Linear((lat_dim_loc_shape + 3) * n_loc + lat_dim_loc_shape + lat_dim_glob_shape, 32))
        elif mode == 'GNN':
            self.lat_dim = lat_dim_expr * 2
            self.pos_enc = nn.Sequential(nn.Linear(3, lat_dim_loc_shape), nn.ReLU(),
                                         nn.Linear(lat_dim_loc_shape, lat_dim_loc_shape))
            self.local_combiner = nn.Sequential(nn.Linear(lat_dim_loc_shape, lat_dim_loc_shape), nn.ReLU(),
                                                nn.Linear(lat_dim_loc_shape, lat_dim_loc_shape))
            self.global_combiner = nn.Sequential(
                nn.Linear(lat_dim_glob_shape + n_loc * lat_dim_loc_shape, 512), nn.ReLU(),
                nn.Linear(512, lat_dim_expr))
        else:
            raise ValueError('Unknown mode!')

        self.defDeepSDF = DeepSDF(lat_dim=self.lat_dim,
                                  hidden_dim=hidden_dim,
                                  nlayers=nlayers,
                                  geometric_init=False,
                                  out_dim=out_dim,
                                  input_dim=input_dim).float()
        self.anchors = anchors

    # ------------------------------------------------------------------
    def _condition(self, xyz, lat_rep, anchors, per_point: bool, with_noise: bool = True):
        """Condition vector of the backbone.  ``per_point=False`` returns ``B x 1 x C`` when the
        mode allows a per-query constant (used by the fused path; ``with_noise=False``: also in training
        mode, the native training path adds the noise itself)."""
        B, N, _ = xyz.shape
        E = self.lat_dim_expr
        if self.mode == 'glob_only':
            return torch.cat([lat_rep[..., :self.lat_dim_glob_shape], lat_rep[..., -E:]], dim=-1)
        if self.mode == 'expr_only':
            return lat_rep[..., -E:]
        if self.mode == 'interpolate':
            loc = lat_rep[:, 0, self.lat_dim_glob_shape:-E - self.lat_dim_loc_shape] \
                .reshape(B, self.num_kps, self.lat_dim_loc_shape)
            a0 = anchors[:, 0] if anchors.dim() == 4 else anchors
            interp = sample_point_feature(xyz[..., :3], a0[..., :3], loc.unsqueeze(1), background=False)
            lat_n = lat_rep.expand(B, N, lat_rep.shape[-1])
            return torch.cat([lat_n[..., :self.lat_dim_glob_shape], interp, lat_n[..., -E:]], dim=-1)
        if self.mode == 'compress':
            # uses the identity code and anchors of point 0 only (reference :218-219)
            a0 = anchors[:, 0] if anchors.dim() == 4 else anchors                 # B x K x 3
            first = torch.cat([lat_rep[:, 0, :-E], a0.reshape(B, -1)], dim=-1)     # B x 1461
            compressed = self.compressor(first).unsqueeze(1)                      # B x 1 x 32
            if per_point or (self.training and with_noise):
                compressed = compressed.expand(B, N, compressed.shape[-1])
                if self.training and with_noise:
                    compressed = compressed + condition_noise(compressed.shape, compressed.device)
                return torch.cat([compressed, lat_rep[..., -E:].expand(B, N, E)], dim=-1)
            return torch.cat([compressed, lat_rep[:, :1, -E:]], dim=-1)           # B x 1 x 232
        if self.mode == 'GNN':
            a0 = anchors[:, 0] if anchors.dim() == 4 else anchors
            offs = self.pos_enc(a0)
            g = self.lat_dim_glob_shape
            loc = lat_rep[:, 0, g:g + self.num_kps * self.lat_dim_loc_shape] \
                .reshape(B, self.num_kps, self.lat_dim_loc_shape)
            combined = self.global_combiner(
                torch.cat([lat_rep[:, 0, :g], self.local_combiner(offs + loc).reshape(B, -1)], dim=-1))
            return torch.cat([combined.unsqueeze(1).expand(B, N, combined.shape[-1]),
                              lat_rep[..., -E:].expand(B, N, E)], dim=-1)
        raise ValueError('Unknown mode')

    def offset_jacobian(self, xyz, lat_rep, anchors):
        """``d offsets / d xyz`` (B x N x 3 x 3) by forward-mode differentiation, or ``None`` when the fast path does not
        apply (condition depends on the point, positional encoding, ReLU backbone, training-mode noise)."""
        backbone = self.defDeepSDF
        if (self.training or self.mode not in ('compress', 'expr_only', 'glob_only') or backbone.num_freq_bands is not None
                or backbone.beta <= 0 or 0 in backbone.skip_in or xyz.dim() != 3):
            return None
        cond = self._condition(xyz, lat_rep, anchors, per_point=lat_rep.shape[1] != 1)
        _, J = _input_jacobian(backbone, xyz, cond)
        return J[..., :3, :]

    def forward(self,
                xyz: torch.Tensor,
                lat_rep: torch.Tensor,
                anchors: Optional[torch.Tensor]) -> (torch.Tensor, torch.Tensor):
        """xyz: B x N x 3; lat_rep: B x N|1 x (lat_id + lat_expr) = ``[z_id | z_ex]``;
        anchors: B x N x K x 3 or B x K x 3.  Returns ``(offsets B x N x 3, last channel B x N x 1)``."""
        if xyz.dim() < 3:
            xyz = xyz.unsqueeze(0)
        backbone = self.defDeepSDF
        if self.mode in ('compress', 'expr_only', 'glob_only') and backbone._native_train_ok(xyz, lat_rep):
            lat = _native.constant_latent_rows(lat_rep)
            if lat is not None:
                # condition built in torch (compressor, anchors upstream keep autograd); the noise rides with xyz
                B, N, _ = xyz.shape
                cond = self._condition(xyz, lat.unsqueeze(1), anchors, per_point=False, with_noise=False)[:, 0]
                noise = (condition_noise((B, N, self.compressor[0].out_features), xyz.device)
                         if self.training and self.mode == 'compress' else None)
                pred = backbone.forward_native_train(xyz, cond, noise)
                return pred[..., :3], pred[..., -1:]
        fused = (backbone._fused_ok(xyz, lat_rep) and not self.training
                 and self.mode in ('compress', 'expr_only', 'glob_only')
                 and not (anchors is not None and torch.is_grad_enabled() and anchors.requires_grad))
        if fused:
            lat = _native.constant_latent_rows(lat_rep)
            if lat is not None:
                cond = self._condition(xyz, lat.unsqueeze(1), anchors, per_point=False)   # B x 1 x C
                pred = backbone.engine().query(xyz, cond[:, 0])
                return pred[..., :3], pred[..., -1:]
        cond = self._condition(xyz, lat_rep, anchors, per_point=True)
        pred = backbone._forward_composite(xyz, cond)
        return pred[..., :3], pred[..., -1:]
