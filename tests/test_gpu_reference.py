"""GPU parity against the UNMODIFIED REFERENCE MODULES, on BASELINE.json's own configurations.  What the reference returns
is stored in golden/reference_parity.npz (tests/golden/make_golden_reference.py: its own modules, torch fp32, on seeded
weights and inputs that the mirrors here reproduce bit for bit); volumes are sampled at every chunk-boundary index, the
index before it, and a seeded uniform set of points:

  * configs[0]: the 64^3 grid, eval and train mode, through ``get_logits``
  * configs[1]: the 256^3 grid - the volume of the benchmark step (all 672 chunk-boundary indices 24 999, 49 999, ...,
    16 777 215, and the far field where exp() underflows) from the in-kernel-grid path the bench times (``query_grid``),
    plus the drop-in ``get_logits`` path on explicit points
  * configs[2]: deformation network on a 64^3 grid, ``get_logits_backward`` with a DeepSDF-type expression decoder

The CUDA kernels are called through the C ABI.  Tolerance: 1e-5 abs (north_star)."""
import hashlib

import numpy as np
import pytest
import torch

from conftest import MAXI, MINI, load_golden, make_deformation, make_ensemble, sample_latent

pytestmark = pytest.mark.gpu
TOL = 1e-5


@pytest.fixture(scope='module')
def ref():
    return load_golden('reference_parity.npz')


def tensor_sha256(t):
    a = np.ascontiguousarray(t.detach().cpu().numpy())
    return hashlib.sha256(('%s%s' % (a.dtype, a.shape)).encode() + a.tobytes()).hexdigest()


def assert_state_is_the_reference(ref, prefix, module):
    sd = module.state_dict()
    assert list(sd.keys()) == list(ref[prefix + '_keys'])
    assert [tensor_sha256(v) for v in sd.values()] == list(ref[prefix + '_sha256'])


def chunk_ends(total, nb):
    return np.concatenate([np.arange(nb - 1, total, nb), [total - 1]])


def _grid(res, dev):
    from nphm_b200.utils.reconstruction import create_grid_points_from_bounds
    g = create_grid_points_from_bounds(MINI, MAXI, res)
    return torch.from_numpy(g).to(dev, dtype=torch.float).reshape(1, -1, 3)          # fitting_pointclouds.py:168-170


def test_mirror_initialises_like_the_reference(cuda_device, ref):
    assert_state_is_the_reference(ref, 'ensemble', make_ensemble(0))
    assert_state_is_the_reference(ref, 'deform', make_deformation())


@pytest.mark.parametrize('train', [False, True])
def test_config1_64cube_full_vs_reference(cuda_device, ref, train):
    """BASELINE.json configs[0]: single-head SDF query on the 64^3 grid, nbatch_points 25 000 (-sample) and 20 000 (fitting)."""
    from nphm_b200.models.reconstruction import get_logits
    dec = make_ensemble(0, device=cuda_device)
    dec.train(train)
    lat = sample_latent(1).to(cuda_device)
    grid = _grid(64, cuda_device)
    idx = ref['c1_idx']
    for nb in (25000, 20000):
        want = ref['c1_%s_%d' % ('train' if train else 'eval', nb)]
        got = get_logits(dec, lat, grid, nbatch_points=nb)
        assert got.shape == (64 ** 3,) and got.dtype == want.dtype
        err = float(np.abs(got[idx] - want).max())
        print('64^3 train=%s nbatch=%d: max abs err %.3g over %d points' % (train, nb, err, len(idx)))
        assert err < TOL


def test_config2_256cube_full_volume_vs_reference(cuda_device, ref):
    """BASELINE.json configs[1]: the 16.7 M-point volume of the benchmark step against the reference."""
    from nphm_b200.models.reconstruction import get_logits
    res, nb = 256, 25000
    total = res ** 3
    dec = make_ensemble(0, device=cuda_device).eval()
    lat = sample_latent(1).to(cuda_device)
    # (a) the path bench.py times: grid generated in the kernel
    vol, _ = dec.engine().query_grid(lat, MINI, MAXI, res, 0, total, quirk_period=nb)
    got = vol.cpu().numpy()
    idx, want = ref['c2_idx'], ref['c2_at_idx']
    diff = np.abs(got[idx] - want)
    worst = int(diff.argmax())
    print('256^3 in-kernel grid: max abs err %.3g at flat index %d (sdf %.4g)' % (diff.max(), idx[worst], want[worst]))
    assert diff.max() < TOL
    # every chunk-boundary index carries the eval-mode quirk value in both
    last = chunk_ends(total, nb)
    assert np.abs(got[last] - ref['c2_last']).max() < TOL
    assert np.abs(got[last - 1] - ref['c2_before_last']).max() < TOL
    assert np.abs(ref['c2_last'] - ref['c2_before_last']).max() > 1e-4     # the quirk is visible in the reference's own output
    # far field (sum of anchor weights underflows, SDF ~ 0.002 * global member)
    far = np.abs(want) < 1e-2
    assert far.sum() > 1000 and diff[far].max() < TOL
    # (b) the drop-in get_logits on explicit points, sampled slabs incl. the ragged last chunk
    grid = _grid(res, cuda_device)
    for k, first in enumerate(ref['c2_slab_first']):
        pts = grid[:, first:first + 2 * nb + 7]          # (a 1-point last chunk crashes the reference itself: squeeze -> 0-dim)
        g2 = get_logits(dec, lat, pts, nbatch_points=nb)
        assert np.abs(g2[ref['c2_slab%d_idx' % k]] - ref['c2_slab%d' % k]).max() < TOL
    # a window of the grid path equals the same window of the full volume (first/count addressing)
    part, _ = dec.engine().query_grid(lat, MINI, MAXI, res, 1234567, 300001, quirk_period=nb)
    assert torch.equal(part, vol[1234567:1234567 + 300001])


def test_config3_deformation_and_joint_vs_reference(cuda_device, ref):
    """BASELINE.json configs[2] at 64^3: forward-deformation field and the identity field at the deformed points."""
    dfn = make_deformation(cuda_device)
    dec = make_ensemble(0, device=cuda_device).eval()
    lat_id = sample_latent(1).to(cuda_device)
    torch.manual_seed(3)
    lat_ex = (torch.randn(200) * 0.01).to(cuda_device)
    cond = torch.cat([lat_id, lat_ex]).reshape(1, 1, -1)
    grid = _grid(64, cuda_device)
    idx = torch.from_numpy(ref['c3_idx'].astype(np.int64)).to(cuda_device)
    want_off = torch.from_numpy(ref['c3_offsets']).to(cuda_device)
    with torch.no_grad():
        anchors = torch.from_numpy(ref['c3_anchors']).to(cuda_device)
        n = grid.shape[1]
        got_off, _ = dfn(grid, cond.repeat(1, n, 1), anchors)
        err = float((got_off[0, idx] - want_off).abs().max())
        print('deformation 64^3: max abs err %.3g (|offset| max %.3g)' % (err, float(want_off.abs().max())))
        assert err < TOL
        warped = (grid[0, idx] + want_off)[None]
        dec.train()                                          # no chunk quirk: compare the plain field
        m = warped.shape[1]
        got_sdf, _ = dec(warped, lat_id.reshape(1, 1, -1).expand(1, m, -1), None)
        assert float((got_sdf.reshape(-1).cpu() - torch.from_numpy(ref['c3_sdf'])).abs().max()) < TOL


def test_get_logits_backward_vs_reference(cuda_device, ref):
    """models/reconstruction.py:28-56 with a DeepSDF-type expression decoder (the only kind it works with upstream)."""
    from nphm_b200.models.deepSDF import DeepSDF
    from nphm_b200.models.reconstruction import get_logits_backward
    torch.manual_seed(31)
    ex = DeepSDF(lat_dim=100, hidden_dim=128, nlayers=6, out_dim=3).to(cuda_device).eval()
    assert_state_is_the_reference(ref, 'expr', ex)
    dec = make_ensemble(0, device=cuda_device).eval()
    lat_id = sample_latent(1).to(cuda_device)
    torch.manual_seed(32)
    lat_ex = (torch.randn(1, 1, 100) * 0.1).to(cuda_device)
    grid = _grid(24, cuda_device)
    idx = ref['bw_idx']
    got, anc_g = get_logits_backward(dec, ex, lat_id.reshape(1, 1, -1), lat_ex, grid, nbatch_points=5000,
                                     return_anchors=True)
    assert got.shape == tuple(ref['bw_shape']) and np.abs(got[idx] - ref['bw_want']).max() < TOL
    assert float(np.abs(anc_g.cpu().numpy() - ref['bw_anchors']).max()) < 1e-6
    # encoding_expr=None: plain get_logits
    got0 = get_logits_backward(dec, ex, lat_id.reshape(1, 1, -1), None, grid, nbatch_points=5000)
    assert np.abs(got0[idx] - ref['bw_want0']).max() < TOL
