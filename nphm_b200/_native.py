"""ctypes binding of ``libnphm_b200.so`` (C ABI declared in ``include/nphm_b200.h``).

PyTorch is used here only for device memory, streams and the caching allocator; the arithmetic of
the hot path happens inside the library.  There is NO fallback: if the library is missing or a call
fails, an exception is raised.
"""
from __future__ import annotations

import ctypes
import os
from ctypes import (POINTER, Structure, byref, c_char_p, c_double, c_float, c_int, c_longlong,
                    c_void_p)
from typing import Optional

import numpy as np
import torch

IMPL_AUTO, IMPL_SIMT, IMPL_TC, IMPL_TC_PRUNED = 0, 1, 2, 3
_IMPL_BY_NAME = {'auto': IMPL_AUTO, 'simt': IMPL_SIMT, 'tc': IMPL_TC, 'tc_pruned': IMPL_TC_PRUNED}

# NPHM_B200_LIB: developer override used for A/B runs of kernel variants (tools/ab_bench.sh); default = the in-tree build
_LIB_PATH = os.environ.get('NPHM_B200_LIB') or os.path.join(os.path.dirname(os.path.abspath(__file__)), 'libnphm_b200.so')
_lib = None

# every symbol include/nphm_b200.h declares (tests check that the library exports all of them)
EXPORTED_SYMBOLS = (
    'nphm_last_error', 'nphm_abi_version', 'nphm_device_info',
    'nphm_ensemble_create', 'nphm_ensemble_destroy', 'nphm_ensemble_set_prune_threshold', 'nphm_ensemble_load_weights',
    'nphm_ensemble_query', 'nphm_ensemble_query_grid', 'nphm_ensemble_get_logits_host',
    'nphm_mlp_create', 'nphm_mlp_destroy', 'nphm_mlp_load_weights', 'nphm_mlp_query',
    'nphm_mlp_query_layers', 'nphm_mlp_jacobian', 'nphm_mlp_backward_inputs', 'nphm_mlp_inverse_jacobian', 'nphm_adam_step',
    'nphm_mc_workspace_bytes', 'nphm_mc_count', 'nphm_mc_emit', 'nphm_marching_cubes_host',
    'nphm_fit_workspace_bytes', 'nphm_fit_identity_step', 'nphm_fit_surface_grad', 'nphm_fit_apply_gradient',
    'nphm_ensemble_backward_inputs', 'nphm_ensemble_anchors',
    'nphm_broyden_workspace_bytes', 'nphm_mlp_broyden_search', 'nphm_nearest_neighbors',
    'nphm_mlp_train_workspace_bytes', 'nphm_mlp_forward_train', 'nphm_mlp_backward_train',
)


class NativeError(RuntimeError):
    pass


# Native first-order training (DeepSDF / DeformationNetwork forwards recorded by autograd run on the layer chain and its
# weight-gradient GEMMs).  Opt-in: at forward time it cannot be seen whether a double backward will follow, and the identity
# losses (stage 1) differentiate the spatial gradient through the same forward.
_native_training = os.environ.get('NPHM_NATIVE_TRAINING', '0') == '1'


def set_native_training(enabled: bool = True) -> None:
    """Switch native first-order training on or off (initial value: environment variable ``NPHM_NATIVE_TRAINING=1``)."""
    global _native_training
    _native_training = bool(enabled)


def native_training() -> bool:
    return _native_training


# kernels of this library launched per call (ncu launch lists under profiles/); bench.py counts its launches with these
MC_LAUNCHES = 3                      # classify rows, scan rows, emit rows


def launches_per_grid_query(impl='auto') -> int:
    """grid axes, anchors, folded constants, [tensor-core records], ensemble kernel."""
    return 4 + (1 if impl in ('auto', 'tc', 'tc_pruned') else 0)


class EnsembleConfig(Structure):
    _fields_ = [('n_loc', c_int), ('n_symm_pairs', c_int), ('lat_dim_glob', c_int), ('lat_dim_loc', c_int),
                ('hidden_dim', c_int), ('n_layers', c_int), ('pos_mlp_dim', c_int)]


class MlpConfig(Structure):
    _fields_ = [('lat_dim', c_int), ('hidden_dim', c_int), ('n_layers', c_int), ('out_dim', c_int)]


class McParams(Structure):
    _fields_ = [('nx', c_int), ('ny', c_int), ('nz', c_int), ('x_global0', c_int), ('ghost_lo', c_int),
                ('negate', c_int), ('iso', c_double)]


class FitParams(Structure):
    _fields_ = [('lambda_surface', c_float), ('lambda_reg_global', c_float), ('lambda_reg_loc', c_float),
                ('lambda_reg_unobserved', c_float), ('lambda_symm_dist', c_float), ('clamp', c_float),
                ('lr', c_float), ('step', c_int)]


def stack_supported(n_hidden_layers: int, hidden: int, cond_dim: int) -> bool:
    """Configurations ``build_stack`` (csrc/api.cu) accepts; anything else takes the composite PyTorch path."""
    return 2 <= n_hidden_layers <= 10 and hidden > cond_dim + 3


def hidden_width(module, n_lin: int) -> int:
    """Hidden width of a DeepSDF-style stack: the input width of its LAST linear layer (``lin0`` is narrowed to
    ``hidden - d_in`` when the skip connection sits at layer 1, i.e. for 2 or 3 hidden layers)."""
    return getattr(module, 'lin%d' % (n_lin - 1)).in_features


def impl_code(impl) -> int:
    if isinstance(impl, str):
        return _IMPL_BY_NAME[impl]
    return int(impl)


def default_impl() -> int:
    """Kernel selection for the drop-in modules; override with NPHM_B200_IMPL=auto|simt|tc."""
    return _IMPL_BY_NAME[os.environ.get('NPHM_B200_IMPL', 'auto')]


def lib() -> ctypes.CDLL:
    """Load the native library (once).  Raises if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(_LIB_PATH):
        raise NativeError('%s is missing: build it with `python -c "import __graft_entry__ as g; g.build()"` '
                          '(or `make -C nphm_b200/csrc`). The fused CUDA path has no fallback.' % _LIB_PATH)
    L = ctypes.CDLL(_LIB_PATH)
    L.nphm_last_error.restype = c_char_p
    L.nphm_abi_version.restype = c_int
    L.nphm_device_info.argtypes = [POINTER(c_int)] * 3
    L.nphm_ensemble_create.argtypes = [POINTER(EnsembleConfig), POINTER(c_void_p)]
    L.nphm_ensemble_destroy.argtypes = [c_void_p]
    L.nphm_ensemble_destroy.restype = None
    L.nphm_ensemble_set_prune_threshold.argtypes = [c_void_p, c_float]
    L.nphm_ensemble_load_weights.argtypes = [c_void_p, POINTER(c_void_p), POINTER(c_void_p), POINTER(c_void_p),
                                             POINTER(c_void_p), c_void_p, c_void_p]
    L.nphm_ensemble_query.argtypes = [c_void_p, c_void_p, c_void_p, c_int, c_longlong, c_longlong, c_void_p,
                                      c_void_p, c_int, c_void_p]
    L.nphm_ensemble_query_grid.argtypes = [c_void_p, c_void_p, POINTER(c_double), POINTER(c_double), c_int,
                                           c_longlong, c_longlong, c_longlong, c_void_p, c_void_p, c_int, c_void_p]
    L.nphm_ensemble_get_logits_host.argtypes = [c_void_p, c_void_p, POINTER(c_double), POINTER(c_double), c_int,
                                                c_longlong, c_void_p, c_int]
    L.nphm_mlp_create.argtypes = [POINTER(MlpConfig), POINTER(c_void_p)]
    L.nphm_mlp_destroy.argtypes = [c_void_p]
    L.nphm_mlp_destroy.restype = None
    L.nphm_mlp_load_weights.argtypes = [c_void_p, POINTER(c_void_p), POINTER(c_void_p), c_void_p]
    L.nphm_mlp_query.argtypes = [c_void_p, c_void_p, c_void_p, c_int, c_longlong, c_void_p, c_int, c_void_p]
    L.nphm_mlp_query_layers.argtypes = [c_void_p, c_void_p, c_void_p, c_int, c_longlong, c_void_p, c_void_p]
    L.nphm_mlp_jacobian.argtypes = [c_void_p, c_void_p, c_void_p, c_int, c_longlong, c_void_p, c_void_p, c_void_p]
    L.nphm_mlp_backward_inputs.argtypes = [c_void_p, c_void_p, c_void_p, c_int, c_longlong, c_void_p, c_void_p, c_void_p, c_void_p]
    L.nphm_mc_workspace_bytes.argtypes = [POINTER(McParams)]
    L.nphm_mc_workspace_bytes.restype = c_longlong
    L.nphm_mc_count.argtypes = [c_void_p, POINTER(McParams), c_void_p, POINTER(c_longlong), POINTER(c_longlong),
                                c_void_p]
    L.nphm_mc_emit.argtypes = [c_void_p, POINTER(McParams), c_void_p, c_longlong, c_void_p, c_void_p, c_void_p]
    L.nphm_marching_cubes_host.argtypes = [c_void_p, c_int, c_int, c_int, c_double, c_int, c_void_p, c_void_p,
                                           POINTER(c_longlong), POINTER(c_longlong)]
    L.nphm_fit_workspace_bytes.argtypes = [c_void_p, c_longlong]
    L.nphm_fit_workspace_bytes.restype = c_longlong
    L.nphm_fit_identity_step.argtypes = [c_void_p, c_void_p, c_longlong, c_void_p, c_void_p, c_void_p,
                                         POINTER(FitParams), c_int, c_void_p, c_void_p, c_void_p, c_void_p]
    L.nphm_fit_surface_grad.argtypes = [c_void_p, c_void_p, c_longlong, c_void_p, c_void_p, c_float, c_void_p, c_void_p,
                                        c_void_p, c_void_p, c_void_p]
    L.nphm_ensemble_anchors.argtypes = [c_void_p, c_void_p, c_int, c_void_p, c_void_p]
    L.nphm_ensemble_backward_inputs.argtypes = [c_void_p, c_void_p, c_longlong, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                                c_void_p, c_void_p]
    L.nphm_fit_apply_gradient.argtypes = [c_void_p, c_void_p, c_void_p, c_void_p, POINTER(FitParams), c_void_p, c_void_p,
                                          c_void_p, c_int, c_void_p, c_void_p, c_void_p]
    L.nphm_adam_step.argtypes = [c_void_p, c_void_p, c_void_p, c_void_p, c_longlong, c_float, c_int, c_void_p]
    L.nphm_mlp_inverse_jacobian.argtypes = [c_void_p, c_void_p, c_void_p, c_int, c_longlong, c_void_p, c_void_p, c_void_p]
    L.nphm_broyden_workspace_bytes.argtypes = [c_longlong]
    L.nphm_broyden_workspace_bytes.restype = c_longlong
    L.nphm_mlp_broyden_search.argtypes = [c_void_p, c_void_p, c_int, c_longlong, c_void_p, c_void_p, c_void_p, c_int,
                                          c_float, c_float, c_float, c_void_p, c_void_p, POINTER(c_int), c_void_p,
                                          c_void_p]
    L.nphm_nearest_neighbors.argtypes = [c_void_p, c_longlong, c_void_p, c_longlong, c_void_p, c_void_p, c_void_p]
    L.nphm_mlp_train_workspace_bytes.argtypes = [c_void_p, c_int, c_longlong, c_int]
    L.nphm_mlp_train_workspace_bytes.restype = c_longlong
    L.nphm_mlp_forward_train.argtypes = [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_longlong, c_void_p, c_void_p,
                                         c_void_p]
    L.nphm_mlp_backward_train.argtypes = [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_longlong, c_void_p,
                                          POINTER(c_void_p), POINTER(c_void_p), c_void_p, c_void_p, c_void_p, c_void_p]
    for name in EXPORTED_SYMBOLS:                      # fail at load time, not at first use, if a symbol is missing
        getattr(L, name)
    _lib = L
    return L


def check(rc: int, what: str = ''):
    if rc != 0:
        msg = lib().nphm_last_error()
        raise NativeError('%s failed (%d): %s' % (what or 'libnphm_b200 call', rc,
                                                   msg.decode() if msg else 'unknown error'))


def _stream_ptr(device) -> int:
    return torch.cuda.current_stream(device).cuda_stream


def _ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


def _ptr_array(tensors):
    arr = (c_void_p * len(tensors))()
    for i, t in enumerate(tensors):
        arr[i] = t.data_ptr()
    return arr


def constant_latent_rows(lat_rep: torch.Tensor) -> Optional[torch.Tensor]:
    """``B x N x D`` (or ``B x 1 x D``) latent -> ``B x D`` if it is the same for all points of a batch
    entry, else ``None``.  Broadcast views (stride 0) are recognised without reading the data; a
    materialised ``repeat`` costs one comparison pass."""
    if lat_rep.dim() == 2:
        return lat_rep.contiguous()
    if lat_rep.shape[1] == 1 or lat_rep.stride(1) == 0:
        return lat_rep[:, 0].contiguous()
    first = lat_rep[:, :1]
    if bool((lat_rep == first).all()):
        return first[:, 0].contiguous()
    return None


def _f32c(t: torch.Tensor) -> torch.Tensor:
    return t.detach().to(dtype=torch.float32).contiguous()


class _Versioned:
    """Tracks parameter identity/version so that packed weights are rebuilt after in-place updates,
    ``load_state_dict`` or ``.to(device)``."""

    def _signature(self, params):
        return tuple((p.data_ptr(), p._version, str(p.device)) for p in params)


class EnsembleEngine(_Versioned):
    """Native handle for one ``FastEnsembleDeepSDFMirrored`` (packed weights live on its device)."""

    def __init__(self, module):
        self._h = c_void_p()
        e = module.ensembled_deep_sdf
        n_lin = e.num_layers - 1
        cfg = EnsembleConfig(module.num_kps, module.num_symm_pairs, module.lat_dim_glob, module.lat_dim_loc,
                             hidden_width(e, n_lin), n_lin - 1, module.pos_mlp_dim)
        check(lib().nphm_ensemble_create(byref(cfg), byref(self._h)), 'nphm_ensemble_create')
        self.n_lin = n_lin
        self.n_loc = module.num_kps
        self.lat_dim = module.lat_dim
        self._sig = None
        self.device = None

    def __del__(self):
        try:
            if self._h and _lib is not None:
                _lib.nphm_ensemble_destroy(self._h)
        except Exception:
            pass

    @property
    def handle(self):
        return self._h

    def set_prune_threshold(self, tau: float):
        """tau of the opt-in pruned kernel (impl='tc_pruned')."""
        check(lib().nphm_ensemble_set_prune_threshold(self._h, float(tau)), 'nphm_ensemble_set_prune_threshold')

    def _params(self, module):
        e = module.ensembled_deep_sdf
        ps = []
        for i in range(self.n_lin):
            lin = getattr(e, 'lin%d' % i)
            ps += [lin.weight, lin.bias]
        for i in (0, 2, 4):
            ps += [module.mlp_pos[i].weight, module.mlp_pos[i].bias]
        return ps

    def refresh(self, module):
        ps = self._params(module)
        anc = module.anchors            # plain attribute (EnsembledDeepSDF.py:192): may be re-assigned after first use
        sig = self._signature(ps) + ((anc.data_ptr(), anc._version, str(anc.device)) if anc is not None else (None,))
        if sig == self._sig:
            return
        dev = ps[0].device
        if dev.type != 'cuda':
            raise NativeError('the fused ensemble needs the module on a CUDA device (got %s)' % dev)
        with torch.cuda.device(dev):
            tens = [_f32c(p) for p in ps]
            lw = tens[0:2 * self.n_lin:2]
            lb = tens[1:2 * self.n_lin:2]
            pw = tens[2 * self.n_lin::2]
            pb = tens[2 * self.n_lin + 1::2]
            mean = _f32c(module.mean_anchors(dev)).reshape(-1)
            check(lib().nphm_ensemble_load_weights(self._h, _ptr_array(lw), _ptr_array(lb), _ptr_array(pw),
                                                   _ptr_array(pb), mean.data_ptr(), _stream_ptr(dev)),
                  'nphm_ensemble_load_weights')
            # the library copies on the current stream; keep the temporaries alive until it is done
            torch.cuda.current_stream(dev).synchronize()
        self._sig = sig
        self.device = dev

    # ---------------------------------------------------------------- queries
    def query(self, xyz: torch.Tensor, latents: torch.Tensor, eval_quirk: bool, quirk_period: Optional[int] = None,
              impl: Optional[int] = None):
        """xyz B x N x 3, latents B x lat_dim -> (sdf B x N x 1, anchors B x n_loc x 3)."""
        B, N, _ = xyz.shape
        dev = xyz.device
        xyz = _f32c(xyz)
        latents = _f32c(latents).to(dev)
        sdf = torch.empty(B, N, 1, device=dev, dtype=torch.float32)
        anchors = torch.empty(B, self.n_loc, 3, device=dev, dtype=torch.float32)
        period = 0 if not eval_quirk else (N if quirk_period is None else int(quirk_period))
        with torch.cuda.device(dev):
            check(lib().nphm_ensemble_query(self._h, xyz.data_ptr(), latents.data_ptr(), B, N, period,
                                            sdf.data_ptr(), anchors.data_ptr(),
                                            default_impl() if impl is None else impl_code(impl), _stream_ptr(dev)),
                  'nphm_ensemble_query')
        return sdf, anchors

    def anchors(self, latents: torch.Tensor) -> torch.Tensor:
        """latents B x lat_dim -> anchors B x n_loc x 3 (the anchor head only, ``nphm_ensemble_anchors``)."""
        lat = _f32c(latents).reshape(-1, self.lat_dim)
        dev = lat.device
        out = torch.empty(lat.shape[0], self.n_loc, 3, device=dev, dtype=torch.float32)
        with torch.cuda.device(dev):
            check(lib().nphm_ensemble_anchors(self._h, lat.data_ptr(), lat.shape[0], out.data_ptr(), _stream_ptr(dev)),
                  'nphm_ensemble_anchors')
        return out

    def backward_inputs(self, xyz: torch.Tensor, latent: torch.Tensor, grad_sdf: torch.Tensor):
        """Vector-Jacobian product of the training-mode forward (``nphm_ensemble_backward_inputs``): xyz (N,3), latent
        (lat_dim,), grad_sdf (N,) -> (sdf (N,), d/d latent (lat_dim,), d/d xyz (N,3)) - what autograd gives for
        ``decoder(xyz, latent)[0].backward(grad_sdf)``, without building a graph."""
        dev = xyz.device
        pts = _f32c(xyz).reshape(-1, 3)
        lat = _f32c(latent).reshape(-1).to(dev)
        g = _f32c(grad_sdf).reshape(-1)
        n = pts.shape[0]
        sdf = torch.empty(n, device=dev, dtype=torch.float32)
        g_lat = torch.empty(self.lat_dim, device=dev, dtype=torch.float32)
        g_pts = torch.empty(n, 3, device=dev, dtype=torch.float32)
        with torch.cuda.device(dev):
            check(lib().nphm_ensemble_backward_inputs(self._h, pts.data_ptr(), n, lat.data_ptr(), g.data_ptr(), sdf.data_ptr(),
                                                      g_lat.data_ptr(), g_pts.data_ptr(), None, _stream_ptr(dev)),
                  'nphm_ensemble_backward_inputs')
        return sdf, g_lat, g_pts

    def query_grid(self, latent: torch.Tensor, mini, maxi, res: int, first: int, count: int, quirk_period: int,
                   impl: Optional[int] = None, out: Optional[torch.Tensor] = None):
        """One latent over grid points [first, first+count) of the res^3 grid -> (sdf (count,), anchors)."""
        dev = latent.device
        latent = _f32c(latent).reshape(-1)
        if out is None:
            out = torch.empty(count, device=dev, dtype=torch.float32)
        anchors = torch.empty(self.n_loc, 3, device=dev, dtype=torch.float32)
        gmin = (c_double * 3)(*[float(v) for v in mini])
        gmax = (c_double * 3)(*[float(v) for v in maxi])
        with torch.cuda.device(dev):
            check(lib().nphm_ensemble_query_grid(self._h, latent.data_ptr(), gmin, gmax, int(res), int(first),
                                                 int(count), int(quirk_period), out.data_ptr(), anchors.data_ptr(),
                                                 default_impl() if impl is None else impl_code(impl),
                                                 _stream_ptr(dev)),
                  'nphm_ensemble_query_grid')
        return out, anchors


def _mlp_impl(impl) -> int:
    code = default_impl() if impl is None else impl_code(impl)
    return IMPL_AUTO if code == IMPL_TC_PRUNED else code


class MlpEngine(_Versioned):
    """Native handle for one ``DeepSDF`` stack (also the backbone of ``DeformationNetwork``)."""

    def __init__(self, module):
        self._h = c_void_p()
        self.n_lin = module.num_layers - 1
        hidden = hidden_width(module, self.n_lin)
        cfg = MlpConfig(module.lat_dim, hidden, self.n_lin - 1, module.out_dim_net)
        check(lib().nphm_mlp_create(byref(cfg), byref(self._h)), 'nphm_mlp_create')
        self.out_dim = module.out_dim_net
        # which kernel family AUTO picks (mirrors tc_mlp_supported in csrc/tc_mlp.cu): the fully fused tcgen05 kernel takes the
        # forward-deformation backbone only; every other shape runs layer by layer on the generic tcgen05 linear layer
        # (csrc/tc_linear.cu, any width - e.g. the NPM baseline 515 -> 1024 x 8); the fp32 FFMA kernel is kept for impl='simt'
        self.fused_shape = (hidden == 512 and self.n_lin == 7 and module.lat_dim == 232 and module.out_dim_net == 3)
        self.simt_ok = hidden <= 880
        self.shapes = [tuple(getattr(module, 'lin%d' % i).weight.shape) for i in range(self.n_lin)]
        self._sig = None

    def __del__(self):
        try:
            if self._h and _lib is not None:
                _lib.nphm_mlp_destroy(self._h)
        except Exception:
            pass

    def refresh(self, module):
        ps = []
        for i in range(self.n_lin):
            lin = getattr(module, 'lin%d' % i)
            ps += [lin.weight, lin.bias]
        sig = self._signature(ps)
        if sig == self._sig:
            return
        dev = ps[0].device
        if dev.type != 'cuda':
            raise NativeError('the fused MLP needs the module on a CUDA device (got %s)' % dev)
        with torch.cuda.device(dev):
            tens = [_f32c(p) for p in ps]
            check(lib().nphm_mlp_load_weights(self._h, _ptr_array(tens[0::2]), _ptr_array(tens[1::2]),
                                              _stream_ptr(dev)), 'nphm_mlp_load_weights')
            torch.cuda.current_stream(dev).synchronize()
        self._sig = sig

    def query(self, xyz: torch.Tensor, cond: torch.Tensor, impl: Optional[int] = None) -> torch.Tensor:
        """xyz B x N x 3, cond B x lat_dim -> B x N x out_dim."""
        code = _mlp_impl(impl)
        if (code == IMPL_AUTO and not self.fused_shape) or (code == IMPL_SIMT and not self.simt_ok):
            return self.query_layers(xyz, cond)
        B, N, _ = xyz.shape
        dev = xyz.device
        xyz = _f32c(xyz)
        cond = _f32c(cond).to(dev)
        out = torch.empty(B, N, self.out_dim, device=dev, dtype=torch.float32)
        with torch.cuda.device(dev):
            check(lib().nphm_mlp_query(self._h, xyz.data_ptr(), cond.data_ptr(), B, N, out.data_ptr(), code, _stream_ptr(dev)),
                  'nphm_mlp_query')
        return out

    def query_layers(self, xyz: torch.Tensor, cond: torch.Tensor) -> torch.Tensor:
        """Forward, layer by layer on the generic tcgen05 linear layer (any width): xyz B x N x 3, cond B x lat_dim."""
        B, N, _ = xyz.shape
        dev = xyz.device
        xyz = _f32c(xyz)
        cond = _f32c(cond).to(dev)
        out = torch.empty(B, N, self.out_dim, device=dev, dtype=torch.float32)
        with torch.cuda.device(dev):
            check(lib().nphm_mlp_query_layers(self._h, xyz.data_ptr(), cond.data_ptr(), B, N, out.data_ptr(), _stream_ptr(dev)),
                  'nphm_mlp_query_layers')
        return out

    def jacobian(self, xyz: torch.Tensor, cond: torch.Tensor):
        """(out B x N x out_dim, J B x N x out_dim x 3 = d out / d xyz) in one forward-mode pass (nphm_mlp_jacobian)."""
        B, N, _ = xyz.shape
        dev = xyz.device
        xyz = _f32c(xyz)
        cond = _f32c(cond).to(dev)
        out = torch.empty(B, N, self.out_dim, device=dev, dtype=torch.float32)
        J = torch.empty(B, N, self.out_dim, 3, device=dev, dtype=torch.float32)
        with torch.cuda.device(dev):
            check(lib().nphm_mlp_jacobian(self._h, xyz.data_ptr(), cond.data_ptr(), B, N, out.data_ptr(), J.data_ptr(),
                                          _stream_ptr(dev)), 'nphm_mlp_jacobian')
        return out, J

    def inverse_jacobian(self, xyz: torch.Tensor, cond: torch.Tensor):
        """(out B x N x 3, (I + d out / d xyz)^-1  B x N x 3 x 3) - the reference's ``jac(...).inverse()`` in one native call."""
        B, N, _ = xyz.shape
        dev = xyz.device
        xyz = _f32c(xyz)
        cond = _f32c(cond).to(dev)
        out = torch.empty(B, N, 3, device=dev, dtype=torch.float32)
        J = torch.empty(B, N, 3, 3, device=dev, dtype=torch.float32)
        with torch.cuda.device(dev):
            check(lib().nphm_mlp_inverse_jacobian(self._h, xyz.data_ptr(), cond.data_ptr(), B, N, out.data_ptr(), J.data_ptr(),
                                                  _stream_ptr(dev)), 'nphm_mlp_inverse_jacobian')
        return out, J

    def backward_inputs(self, xyz: torch.Tensor, cond: torch.Tensor, grad_out: torch.Tensor, want_xyz: bool = False,
                        reuse_value_pass: bool = False):
        """Adjoint pass (nphm_mlp_backward_inputs): grad_out B x N x out_dim -> (d/d cond  B x lat_dim, d/d xyz B x N x 3 | None).
        ``reuse_value_pass``: the preceding ``jacobian`` / ``inverse_jacobian`` call was at the same (xyz, cond)."""
        B, N, _ = xyz.shape
        dev = xyz.device
        xyz = _f32c(xyz)
        cond = _f32c(cond).to(dev)
        g = _f32c(grad_out)
        g_cond = torch.empty(B, cond.shape[-1], device=dev, dtype=torch.float32)
        g_xyz = torch.empty(B, N, 3, device=dev, dtype=torch.float32) if want_xyz else None
        with torch.cuda.device(dev):
            check(lib().nphm_mlp_backward_inputs(self._h, None if reuse_value_pass else xyz.data_ptr(), cond.data_ptr(), B, N,
                                                 g.data_ptr(), g_cond.data_ptr(), _ptr(g_xyz), _stream_ptr(dev)),
                  'nphm_mlp_backward_inputs')
        return g_cond, g_xyz

    def forward_train(self, xyz: torch.Tensor, cond: torch.Tensor, noise: Optional[torch.Tensor] = None):
        """Training forward (nphm_mlp_forward_train): xyz B x N x 3, cond B x lat_dim, noise B x N x noise_dim (added to the
        first noise_dim condition columns) or None -> (out B x N x out_dim, workspace).  The workspace (a uint8 tensor allocated
        on the current stream) holds the activations ``backward_train`` reads."""
        B, N, _ = xyz.shape
        dev = xyz.device
        xyz = _f32c(xyz)
        cond = _f32c(cond).to(dev)
        nd = 0 if noise is None else int(noise.shape[-1])
        noise = None if noise is None else _f32c(noise)
        out = torch.empty(B, N, self.out_dim, device=dev, dtype=torch.float32)
        with torch.cuda.device(dev):
            n_bytes = int(lib().nphm_mlp_train_workspace_bytes(self._h, B, N, nd))
            if n_bytes < 0:
                check(-1, 'nphm_mlp_train_workspace_bytes')
            ws = torch.empty(n_bytes, device=dev, dtype=torch.uint8)
            check(lib().nphm_mlp_forward_train(self._h, xyz.data_ptr(), cond.data_ptr(), _ptr(noise), nd, B, N, out.data_ptr(),
                                               ws.data_ptr(), _stream_ptr(dev)), 'nphm_mlp_forward_train')
        return out, ws

    def backward_train(self, xyz: torch.Tensor, cond: torch.Tensor, noise: Optional[torch.Tensor], workspace: torch.Tensor,
                       grad_out: torch.Tensor, want_w=True, want_b=True, want_cond: bool = True, want_xyz: bool = True):
        """Gradients of ``sum(out * grad_out)`` for the ``forward_train`` call that filled ``workspace`` (nphm_mlp_backward_train).
        ``want_w`` / ``want_b``: bool, or one bool per layer.  Returns (grad_w list, grad_b list, d/d cond B x lat_dim,
        d/d xyz B x N x 3); entries not asked for are None."""
        B, N, _ = xyz.shape
        dev = xyz.device
        xyz = _f32c(xyz)
        cond = _f32c(cond).to(dev)
        nd = 0 if noise is None else int(noise.shape[-1])
        noise = None if noise is None else _f32c(noise)
        g = _f32c(grad_out)
        per_layer = lambda want: [bool(want)] * self.n_lin if isinstance(want, bool) else [bool(w) for w in want]
        ww, wb = per_layer(want_w), per_layer(want_b)
        gw = [torch.empty(self.shapes[l], device=dev, dtype=torch.float32) if ww[l] else None for l in range(self.n_lin)]
        gb = [torch.empty(self.shapes[l][0], device=dev, dtype=torch.float32) if wb[l] else None for l in range(self.n_lin)]
        g_cond = torch.empty(B, cond.shape[-1], device=dev, dtype=torch.float32) if want_cond else None
        g_xyz = torch.empty(B, N, 3, device=dev, dtype=torch.float32) if want_xyz else None

        def ptrs(ts):
            if not any(t is not None for t in ts):
                return None
            arr = (c_void_p * len(ts))()
            for i, t in enumerate(ts):
                arr[i] = None if t is None else t.data_ptr()
            return arr
        with torch.cuda.device(dev):
            check(lib().nphm_mlp_backward_train(self._h, xyz.data_ptr(), cond.data_ptr(), _ptr(noise), nd, B, N, g.data_ptr(),
                                                ptrs(gw), ptrs(gb), _ptr(g_cond), _ptr(g_xyz), workspace.data_ptr(),
                                                _stream_ptr(dev)), 'nphm_mlp_backward_train')
        return gw, gb, g_cond, g_xyz

    def broyden_search(self, obs: torch.Tensor, cond: torch.Tensor, x_init: torch.Tensor, J_inv_init: torch.Tensor,
                       max_steps: int = 15, cvg_thresh: float = 1e-6, dvg_thresh: float = 0.2, eps: float = 1e-6,
                       early_exit: bool = True):
        """Roots of ``x + F(x; cond) - obs`` by the reference's Broyden iteration, entirely on the device.
        obs, x_init: B x N x 3, cond: B x lat_dim, J_inv_init: B x N x 3 x 3.
        Returns ``(x B x N x 3, diff B x N, valid B x N bool, steps taken)``."""
        B, N, _ = obs.shape
        dev = obs.device
        obs = _f32c(obs)
        cond = _f32c(cond).to(dev)
        x = _f32c(x_init).clone()
        jinv = _f32c(J_inv_init.reshape(B, N, 9))
        diff = torch.empty(B, N, device=dev, dtype=torch.float32)
        valid = torch.empty(B, N, device=dev, dtype=torch.uint8)
        steps = c_int(0)
        with torch.cuda.device(dev):
            ws = torch.empty(max(int(lib().nphm_broyden_workspace_bytes(B * N)), 256), device=dev, dtype=torch.uint8)
            check(lib().nphm_mlp_broyden_search(self._h, cond.data_ptr(), B, N, obs.data_ptr(), x.data_ptr(),
                                                jinv.data_ptr(), int(max_steps), float(cvg_thresh), float(dvg_thresh),
                                                float(eps), diff.data_ptr(), valid.data_ptr(),
                                                byref(steps) if early_exit else None,       # None: no host sync, all steps run
                                                ws.data_ptr(), _stream_ptr(dev)), 'nphm_mlp_broyden_search')
        return x, diff, valid.bool(), steps.value


# ------------------------------------------------------------------------------------------ marching cubes
def marching_cubes_device(volume: torch.Tensor, iso: float = 0.0, negate: bool = False, x_global0: int = 0,
                          ghost_lo: bool = False, vert_id_base: Optional[int] = None):
    """GPU marching cubes on a CUDA float32 volume (nx, ny, nz).  Returns (verts (V,3) float64 CUDA in global
    index units, tris (T,3) int64 CUDA).  With ``vert_id_base=None`` ids start at 0; a sharded caller passes the
    number of vertices of all earlier slabs, see ``nphm_b200.distributed``."""
    assert volume.is_cuda and volume.dtype == torch.float32 and volume.dim() == 3
    vol = volume.contiguous()
    dev = vol.device
    p = McParams(vol.shape[0], vol.shape[1], vol.shape[2], int(x_global0), int(bool(ghost_lo)), int(bool(negate)),
                 float(iso))
    L = lib()
    ws_bytes = L.nphm_mc_workspace_bytes(byref(p))
    if ws_bytes < 0:
        check(-1, 'nphm_mc_workspace_bytes')
    ws = torch.empty(max(int(ws_bytes), 256), device=dev, dtype=torch.uint8)
    nv, nt = c_longlong(0), c_longlong(0)
    with torch.cuda.device(dev):
        check(L.nphm_mc_count(vol.data_ptr(), byref(p), ws.data_ptr(), byref(nv), byref(nt), _stream_ptr(dev)),
              'nphm_mc_count')
        verts = torch.empty(nv.value, 3, device=dev, dtype=torch.float64)
        tris = torch.empty(nt.value, 3, device=dev, dtype=torch.int64)
        if nv.value or nt.value:
            check(L.nphm_mc_emit(vol.data_ptr(), byref(p), ws.data_ptr(), int(vert_id_base or 0),
                                 verts.data_ptr(), tris.data_ptr(), _stream_ptr(dev)), 'nphm_mc_emit')
    return verts, tris


def marching_cubes_count(volume: torch.Tensor, iso=0.0, negate=False, x_global0=0, ghost_lo=False):
    """Pass 1 only: (n_verts, n_tris, params, workspace) for a slab; used by the sharded extraction."""
    vol = volume.contiguous()
    dev = vol.device
    p = McParams(vol.shape[0], vol.shape[1], vol.shape[2], int(x_global0), int(bool(ghost_lo)), int(bool(negate)),
                 float(iso))
    L = lib()
    ws = torch.empty(max(int(L.nphm_mc_workspace_bytes(byref(p))), 256), device=dev, dtype=torch.uint8)
    nv, nt = c_longlong(0), c_longlong(0)
    with torch.cuda.device(dev):
        check(L.nphm_mc_count(vol.data_ptr(), byref(p), ws.data_ptr(), byref(nv), byref(nt), _stream_ptr(dev)),
              'nphm_mc_count')
    return nv.value, nt.value, p, ws


def marching_cubes_emit(volume: torch.Tensor, p: McParams, ws: torch.Tensor, n_verts: int, n_tris: int,
                        vert_id_base: int):
    vol = volume.contiguous()
    dev = vol.device
    verts = torch.empty(n_verts, 3, device=dev, dtype=torch.float64)
    tris = torch.empty(n_tris, 3, device=dev, dtype=torch.int64)
    if n_verts or n_tris:
        with torch.cuda.device(dev):
            check(lib().nphm_mc_emit(vol.data_ptr(), byref(p), ws.data_ptr(), int(vert_id_base), verts.data_ptr(),
                                     tris.data_ptr(), _stream_ptr(dev)), 'nphm_mc_emit')
    return verts, tris


def marching_cubes_host(volume: np.ndarray, iso: float = 0.0, negate: bool = False):
    """== ``mcubes.marching_cubes`` on a host array through the host-buffer C entry point."""
    vol = np.ascontiguousarray(volume, dtype=np.float32)
    nx, ny, nz = vol.shape
    nv, nt = c_longlong(0), c_longlong(0)
    L = lib()
    check(L.nphm_marching_cubes_host(vol.ctypes.data, nx, ny, nz, float(iso), int(negate), None, None,
                                     byref(nv), byref(nt)), 'nphm_marching_cubes_host')
    verts = np.empty((nv.value, 3), np.float64)
    tris = np.empty((nt.value, 3), np.int64)
    if nv.value or nt.value:
        check(L.nphm_marching_cubes_host(vol.ctypes.data, nx, ny, nz, float(iso), int(negate), verts.ctypes.data,
                                         tris.ctypes.data, byref(nv), byref(nt)), 'nphm_marching_cubes_host')
    return verts, tris.view(np.uint64)


# ------------------------------------------------------------------------------------------ evaluation metrics
def nearest_neighbors(src: torch.Tensor, tgt: torch.Tensor):
    """(dist (n_src,) float64, idx (n_src,) int64) of the nearest ``tgt`` point of every ``src`` point (CUDA float32 clouds)."""
    assert src.is_cuda and tgt.is_cuda and src.shape[-1] == 3 and tgt.shape[-1] == 3
    dev = src.device
    s, t = _f32c(src).reshape(-1, 3), _f32c(tgt).reshape(-1, 3)
    dist = torch.empty(s.shape[0], device=dev, dtype=torch.float64)
    idx = torch.empty(s.shape[0], device=dev, dtype=torch.int64)
    with torch.cuda.device(dev):
        check(lib().nphm_nearest_neighbors(s.data_ptr(), s.shape[0], t.data_ptr(), t.shape[0], dist.data_ptr(), idx.data_ptr(),
                                           _stream_ptr(dev)), 'nphm_nearest_neighbors')
    return dist, idx
