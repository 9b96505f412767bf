"""Native first-order training (nphm_mlp_forward_train / nphm_mlp_backward_train, csrc/tc_wgrad.cu) on the GPU.

The weight, condition and point gradients are compared with float64 autograd of the composite module; the full-size stage-2
step (tools/bench_train_corresp.py) with the native path on is compared with the composite step on the same GPU."""
import copy
import importlib.util
import os

import pytest
import torch
import torch.nn.functional as F

from conftest import make_deformation

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
_NETS = {}


def _net(kind, device):
    if kind not in _NETS:
        from nphm_b200.models.deepSDF import DeepSDF
        if kind == 'deform':
            _NETS[kind] = (make_deformation(device).defDeepSDF, 232)
        elif kind == 'npm':
            torch.manual_seed(12)
            _NETS[kind] = (DeepSDF(lat_dim=512, hidden_dim=1024, nlayers=8, geometric_init=True).to(device), 512)
        else:
            torch.manual_seed(12)
            _NETS[kind] = (DeepSDF(lat_dim=40, hidden_dim=96, nlayers=5, geometric_init=False, out_dim=3).to(device), 40)
    return _NETS[kind]


def _inputs(net, lat_dim, B, N, nd, device, seed=3):
    g = torch.Generator(device='cpu').manual_seed(seed)
    xyz = ((torch.rand(B, N, 3, generator=g) - 0.5) * 0.8).to(device)
    cond = (torch.randn(B, lat_dim, generator=g) * 0.05).to(device)
    noise = (torch.randn(B, N, nd, generator=g) / 200).to(device) if nd else None
    up = torch.randn(B, N, net.out_dim_net, generator=g).to(device)
    return xyz, cond, noise, up


def _clone(net):
    """Deep copy without the native handle (each copy gets its own engine)."""
    eng, net._engine = net._engine, None
    try:
        return copy.deepcopy(net)
    finally:
        net._engine = eng


def _reference(net, xyz, cond, noise, up):
    """float64 autograd of the composite: (out, [dW_l, db_l ...], d cond, d xyz)."""
    n64 = _clone(net).double()
    x = xyz.double().requires_grad_(True)
    c = cond.double().requires_grad_(True)
    B, N, _ = xyz.shape
    cp = c[:, None, :].expand(B, N, c.shape[-1])
    if noise is not None:
        cp = cp + F.pad(noise.double(), (0, c.shape[-1] - noise.shape[-1]))
    out = n64._forward_composite(x, cp)
    params = []
    for i in range(n64.num_layers - 1):
        lin = getattr(n64, 'lin%d' % i)
        params += [lin.weight, lin.bias]
    grads = torch.autograd.grad((out * up.double()).sum(), params + [c, x])
    return out, list(grads[:-2]), grads[-2], grads[-1]


def _rel(got, ref):
    return float((got.double() - ref).abs().max() / ref.abs().max().clamp_min(1e-30))


@pytest.mark.parametrize('N', [1, 127, 129, 1000])
@pytest.mark.parametrize('B', [1, 3])
@pytest.mark.parametrize('nd', [0, 32])
@pytest.mark.parametrize('kind', ['deform', 'npm', 'small'])
def test_backward_train_matches_float64_autograd(cuda_device, kind, nd, B, N):
    """Value, weight / bias / condition / point gradients of one training forward + backward against float64 autograd:
    values <= 1e-5 absolute, gradients <= 2e-4 x max |ref| per tensor (5e-4 for the 8 x 1024 NPM stack, as the chain adjoint
    test).  N = 1, 127, 129, 1000 put the last 128-row tile's pad rows at every position the reduction sees."""
    net, lat_dim = _net(kind, cuda_device)
    xyz, cond, noise, up = _inputs(net, lat_dim, B, N, nd, cuda_device)
    eng = net.engine()
    out, ws = eng.forward_train(xyz, cond, noise)
    gw, gb, g_cond, g_xyz = eng.backward_train(xyz, cond, noise, ws, up)
    ref_out, ref_p, ref_c, ref_x = _reference(net, xyz, cond, noise, up)
    verr = float((out.double() - ref_out).abs().max())
    tol = 5e-4 if kind == 'npm' else 2e-4
    errs = {'cond': _rel(g_cond, ref_c), 'xyz': _rel(g_xyz, ref_x)}
    for l in range(len(gw)):
        errs['W%d' % l] = _rel(gw[l], ref_p[2 * l])
        errs['b%d' % l] = _rel(gb[l], ref_p[2 * l + 1])
    worst = max(errs, key=errs.get)
    print('%s nd=%d B=%d N=%d: value err %.3g, worst gradient %s %.3g' % (kind, nd, B, N, verr, worst, errs[worst]))
    assert verr < 1e-5
    assert errs[worst] < tol, errs


def test_backward_train_null_outputs_and_determinism(cuda_device):
    """Every combination of NULL outputs gives what the full call gives; two identical calls give bitwise-identical weight
    (and bias) gradients."""
    net, lat_dim = _net('small', cuda_device)
    xyz, cond, noise, up = _inputs(net, lat_dim, 3, 333, 32, cuda_device, seed=9)
    eng = net.engine()
    _, ws = eng.forward_train(xyz, cond, noise)
    full = eng.backward_train(xyz, cond, noise, ws, up)
    again = eng.backward_train(xyz, cond, noise, ws, up)
    for a, b in zip(full[0] + full[1], again[0] + again[1]):
        assert torch.equal(a, b)
    # per-layer NULL entries, including the layers whose condition columns come from the per-query sums (0 and skip)
    n_lin, skip = len(full[0]), net.skip_in[0]
    for drop in (0, skip, n_lin - 1):
        keep = [l != drop for l in range(n_lin)]
        gw, gb, _, _ = eng.backward_train(xyz, cond, noise, ws, up, want_w=keep, want_b=keep, want_cond=False, want_xyz=False)
        for l in range(n_lin):
            assert (gw[l] is None and gb[l] is None) if l == drop else (torch.equal(gw[l], full[0][l]) and torch.equal(gb[l], full[1][l]))
    for mask in range(16):
        ww, wb, wc, wx = (bool(mask & 1), bool(mask & 2), bool(mask & 4), bool(mask & 8))
        gw, gb, gc, gx = eng.backward_train(xyz, cond, noise, ws, up, want_w=ww, want_b=wb, want_cond=wc, want_xyz=wx)
        for want, got, ref in ((ww, gw, full[0]), (wb, gb, full[1])):
            for g, r in zip(got, ref):
                assert (g is None) != want
                if want:
                    assert torch.equal(g, r)
        for want, g, r in ((wc, gc, full[2]), (wx, gx, full[3])):
            assert (g is None) != want
            if want:
                assert float((g - r).abs().max()) <= 1e-6 * float(r.abs().max())


def test_backward_train_refusals(cuda_device):
    """A workspace of another shape, another noise width or older weights is refused; so are a double backward, a second
    backward through a retained graph and an in-place weight change between forward and backward."""
    import nphm_b200
    from nphm_b200._native import NativeError
    net, lat_dim = _net('small', cuda_device)
    net = _clone(net)
    eng = net.engine()
    xyz, cond, noise, up = _inputs(net, lat_dim, 2, 100, 32, cuda_device)
    _, ws = eng.forward_train(xyz, cond, noise)
    x2, c2, n2, u2 = _inputs(net, lat_dim, 2, 50, 32, cuda_device)
    with pytest.raises(NativeError, match='another|not'):
        eng.backward_train(x2, c2, n2, ws, u2)
    with pytest.raises(NativeError):
        eng.backward_train(xyz, cond, noise[..., :16].contiguous(), ws, up)
    with torch.no_grad():
        net.lin0.weight.mul_(1.0)
    eng = net.engine()                                  # reloads: the workspace now holds a forward of older weights
    with pytest.raises(NativeError, match='older weights'):
        eng.backward_train(xyz, cond, noise, ws, up)

    nphm_b200.set_native_training(True)
    try:
        xa = xyz.clone().requires_grad_(True)
        lat = cond[:, None, :].expand(2, 100, lat_dim)
        out, _ = net(xa, lat)
        with pytest.raises(RuntimeError, match='set_native_training'):
            torch.autograd.grad(out.sum(), xa, create_graph=True)
        out, _ = net(xa, lat)
        out.sum().backward(retain_graph=True)
        with pytest.raises(RuntimeError, match='differentiated once'):
            out.sum().backward()
        out, _ = net(xa, lat)
        with torch.no_grad():
            net.lin1.weight.add_(0.0)
        with pytest.raises(RuntimeError, match='modified by an inplace operation'):
            out.sum().backward()
    finally:
        nphm_b200.set_native_training(False)


def test_switch_off_never_calls_the_library(cuda_device, monkeypatch):
    """With the switch off, a training-mode forward under autograd stays on the composite."""
    import nphm_b200
    from nphm_b200 import _native
    dfn = make_deformation(cuda_device).train()
    nphm_b200.set_native_training(False)

    def fail():
        raise AssertionError('library called with native training off')
    monkeypatch.setattr(_native, 'lib', fail)
    xyz = (torch.rand(2, 50, 3, device=cuda_device) - 0.5).requires_grad_(True)
    lat = torch.randn(2, 1, 1544, device=cuda_device).expand(2, 50, 1544) * 0.05
    anchors = torch.randn(2, 39, 3, device=cuda_device) * 0.3
    delta, _ = dfn(xyz, lat, anchors)
    delta.sum().backward()
    assert xyz.grad is not None


class _CountNative:
    """Counts the native training calls (MlpEngine.forward_train / backward_train), so a test can tell the native path ran."""

    def __init__(self, monkeypatch):
        from nphm_b200 import _native
        self.calls = {'forward_train': 0, 'backward_train': 0}
        for name in self.calls:
            orig = getattr(_native.MlpEngine, name)

            def wrapped(*a, _orig=orig, _name=name, **k):
                self.calls[_name] += 1
                return _orig(*a, **k)
            monkeypatch.setattr(_native.MlpEngine, name, wrapped)

    def take(self):
        c, self.calls = dict(self.calls), {k: 0 for k in self.calls}
        return c


@pytest.mark.parametrize('kind', ['nphm', 'npm'])
def test_native_training_step_matches_reference_golden(cuda_device, kind, monkeypatch):
    """One stage-2 step with the native path on (the reference's noise and samples injected) against the unmodified reference
    (tests/golden/train_corresp.npz, B = 4, 300 + 100 points): losses <= 1e-5 relative, gradients <= 2e-4 x max |ref| per
    tensor on the stored positions and for the code / point gradients, norms <= 1e-4 relative."""
    import nphm_b200
    from train_corresp_replay import compare, replay
    count = _CountNative(monkeypatch)
    nphm_b200.set_native_training(True)
    try:
        dev = compare(kind, *replay(kind, cuda_device, monkeypatch))
    finally:
        nphm_b200.set_native_training(False)
    assert count.take() == {'forward_train': 2, 'backward_train': 2}      # correspondences and samples, both native
    for group, tol in (('loss', 1e-5), ('grad', 2e-4), ('norm', 1e-4)):
        sub = {k: v for k, v in dev.items() if k.startswith(group)}
        worst = max(sub, key=sub.get)
        print('%s native vs reference golden: worst %s %.3g' % (kind, worst, sub[worst]))
        assert sub[worst] <= tol, sub


def _bench_module():
    spec = importlib.util.spec_from_file_location('bench_train_corresp', os.path.join(ROOT, 'tools', 'bench_train_corresp.py'))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


@pytest.mark.parametrize('kind', ['nphm', 'npm'])
def test_full_size_step_native_matches_composite(cuda_device, kind, monkeypatch):
    """B = 32, 1000 + 100 points, the shipped lambdas: gradients of the first step within 2e-4 x max |composite| per tensor,
    loss curves within 1e-3 relative over 10 optimiser steps (weights change and are re-packed every step)."""
    bench = _bench_module()
    request_off = __import__('nphm_b200').set_native_training
    count = _CountNative(monkeypatch)
    arms = {'native': bench.make_setup(kind, cuda_device), 'composite': bench.make_setup(kind, cuda_device)}
    grads = {}
    for name, s in arms.items():
        torch.manual_seed(77)
        bench.train_step(s, name == 'native', step_only_loss=True)
        assert count.take() == ({'forward_train': 2, 'backward_train': 2} if name == 'native' else
                                {'forward_train': 0, 'backward_train': 0})
        grads[name] = [p.grad.detach().clone() for p in s['decoder'].parameters()] + [s['codes'].weight.grad.to_dense().clone()]
    worst = max(_rel(a, b.double()) for a, b in zip(grads['native'], grads['composite']))
    print('%s full-size step: worst per-tensor gradient deviation %.3g' % (kind, worst))
    assert worst < 2e-4
    arms = {'native': bench.make_setup(kind, cuda_device), 'composite': bench.make_setup(kind, cuda_device)}
    curves = {'native': [], 'composite': []}
    for i in range(10):
        for name, s in arms.items():
            torch.manual_seed(500 + i)
            curves[name].append(bench.train_step(s, name == 'native')['loss'])
    request_off(False)
    dev = max(abs(a - b) / abs(b) for a, b in zip(curves['native'], curves['composite']))
    print('%s loss curves: max relative deviation %.3g over 10 steps' % (kind, dev))
    assert dev < 1e-3
