"""Native-training switch and the training-mode composite path (no GPU needed)."""
import os
import subprocess
import sys

import pytest
import torch

from conftest import make_deformation

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _switch_in_fresh_process(env_value):
    env = dict(os.environ)
    env.pop('NPHM_NATIVE_TRAINING', None)
    if env_value is not None:
        env['NPHM_NATIVE_TRAINING'] = env_value
    code = 'import nphm_b200; print(nphm_b200.native_training())'
    out = subprocess.run([sys.executable, '-B', '-c', code], cwd=ROOT, env=env, capture_output=True, text=True, check=True)
    return out.stdout.strip()


def test_native_training_defaults_off_and_reads_the_environment():
    assert _switch_in_fresh_process(None) == 'False'
    assert _switch_in_fresh_process('0') == 'False'
    assert _switch_in_fresh_process('1') == 'True'


def test_set_native_training_toggles():
    import nphm_b200
    before = nphm_b200.native_training()
    try:
        nphm_b200.set_native_training(True)
        assert nphm_b200.native_training()
        nphm_b200.set_native_training(False)
        assert not nphm_b200.native_training()
    finally:
        nphm_b200.set_native_training(before)


def test_training_noise_is_drawn_through_the_helper(monkeypatch):
    """The training-mode composite adds exactly what ``condition_noise`` returns to the compressed code (per point)."""
    from nphm_b200.models import deepSDF
    dfn = make_deformation().train()
    torch.manual_seed(4)
    B, N = 2, 7
    xyz = torch.rand(B, N, 3) - 0.5
    lat = (torch.randn(B, 1, 1544) * 0.05).expand(B, N, 1544)
    anchors = torch.randn(B, 39, 3) * 0.3
    fixed = torch.randn(B, N, 32) / 200
    calls = []

    def noise(shape, device):
        calls.append(tuple(shape))
        return fixed
    monkeypatch.setattr(deepSDF, 'condition_noise', noise)
    got, _ = dfn(xyz, lat, anchors)
    assert calls == [(B, N, 32)]
    with torch.no_grad():
        first = torch.cat([lat[:, 0, :-200], anchors.reshape(B, -1)], dim=-1)
        cond = torch.cat([dfn.compressor(first)[:, None, :] + fixed, lat[..., -200:]], dim=-1)
        ref = dfn.defDeepSDF._forward_composite(xyz, cond)[..., :3]
    assert torch.allclose(got, ref, atol=1e-7, rtol=0)


@pytest.mark.parametrize('kind', ['nphm', 'npm'])
def test_composite_training_step_matches_reference_golden(kind, monkeypatch):
    """One stage-2 step of the training-mode composite (the reference's noise and samples injected) against the unmodified
    reference (tests/golden/train_corresp.npz): losses, gradient samples, norms and the code / point gradients <= 1e-5."""
    import nphm_b200
    from train_corresp_replay import compare, replay
    nphm_b200.set_native_training(False)
    dev = compare(kind, *replay(kind, torch.device('cpu'), monkeypatch))
    worst = max(dev, key=dev.get)
    print('%s composite vs reference golden: worst %s %.3g' % (kind, worst, dev[worst]))
    assert dev[worst] <= 1e-5, dev
