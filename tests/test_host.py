"""CPU suite, part 2: host-side logic of the drop-in modules (composite path), API surface, and that the C-ABI
library loads and exports every symbol include/nphm_b200.h declares (no compute calls without a GPU)."""
import ctypes
import hashlib
import os
import re

import numpy as np
import pytest
import torch

from conftest import ROOT, load_golden, make_deformation, make_ensemble, make_npm, mean_anchors


def sd_hash(sd):
    h = hashlib.sha256()
    for k in sorted(sd.keys()):
        h.update(k.encode())
        h.update(np.ascontiguousarray(sd[k].detach().cpu().numpy()).tobytes())
    return h.hexdigest()


def test_initialisation_is_bit_identical_to_reference():
    g, d = load_golden('ensemble.npz'), load_golden('deform.npz')
    assert sd_hash(make_ensemble(0).state_dict()) == str(g['sha256_a'])
    assert sd_hash(make_ensemble(5, 2.0).state_dict()) == str(g['sha256_b'])
    assert sd_hash(make_deformation().state_dict()) == str(d['sha256_def'])
    assert sd_hash(make_npm().state_dict()) == str(d['sha256_npm'])


def test_state_dict_contract():
    sd = make_ensemble(0).state_dict()
    assert sd['ensembled_deep_sdf.lin0.weight'].shape == (24, 200, 99)
    assert sd['ensembled_deep_sdf.lin1.weight'].shape == (24, 101, 200)
    assert sd['ensembled_deep_sdf.lin2.weight'].shape == (24, 200, 200)
    assert sd['ensembled_deep_sdf.lin4.bias'].shape == (24, 1)
    assert sd['mlp_pos.4.weight'].shape == (117, 256)
    assert not any(k.startswith('anchors') or '_set_of_member' in k for k in sd)
    dsd = make_deformation().state_dict()
    assert dsd['compressor.0.weight'].shape == (32, 1461)
    assert dsd['defDeepSDF.lin0.weight'].shape == (512, 235)
    assert dsd['defDeepSDF.lin2.weight'].shape == (277, 512)
    assert dsd['defDeepSDF.lin6.weight'].shape == (3, 512)
    dec = make_ensemble(0)
    assert (dec.lat_dim, dec.lat_dim_glob, dec.lat_dim_loc, dec.num_kps, dec.num_symm_pairs) == (1344, 64, 32, 39, 16)


def test_composite_forward_matches_reference_outputs():
    g = load_golden('ensemble.npz')
    for tag, seed, scale in (('a', 0, 1.0), ('b', 5, 2.0)):
        dec = make_ensemble(seed, scale)
        x = torch.from_numpy(g['points_' + tag]).unsqueeze(0)
        lat = torch.from_numpy(g['latent_' + tag]).reshape(1, 1, -1)
        with torch.no_grad():
            dec.eval()
            s_eval, anc = dec(x, lat, None)
            dec.train()
            s_train, _ = dec(x, lat.repeat(1, x.shape[1], 1), None)     # materialised per-point latent
        assert s_eval.shape == (1, x.shape[1], 1) and anc.shape == (1, 39, 3)
        assert np.abs(s_eval.numpy().reshape(-1) - g['sdf_eval_' + tag]).max() < 1e-5
        assert np.abs(s_train.numpy().reshape(-1) - g['sdf_train_' + tag]).max() < 1e-5
        assert np.abs(anc.numpy()[0] - g['anchors_' + tag]).max() < 1e-6


def test_composite_deformation_and_get_logits():
    from nphm_b200.models.reconstruction import get_logits
    from nphm_b200.utils.reconstruction import create_grid_points_from_bounds
    d = load_golden('deform.npz')
    dfn = make_deformation()
    pts = torch.from_numpy(d['points']).unsqueeze(0)
    cond = torch.cat([torch.from_numpy(d['latent_id']), torch.from_numpy(d['z_ex'])]).reshape(1, 1, -1)
    with torch.no_grad():
        off, last = dfn(pts, cond.repeat(1, pts.shape[1], 1), torch.from_numpy(d['anchors']).unsqueeze(0))
        npm_out, none = make_npm()(pts, torch.from_numpy(d['z_npm']).reshape(1, 1, -1).repeat(1, pts.shape[1], 1))
    assert none is None
    assert np.abs(off.numpy()[0] - d['offsets']).max() < 1e-5 and np.abs(last.numpy().reshape(-1) - d['last']).max() < 1e-5
    assert np.abs(npm_out.numpy().reshape(-1) - d['npm_out']).max() < 1e-5
    g = load_golden('ensemble.npz')
    dec = make_ensemble(0).eval()
    grid = torch.from_numpy(create_grid_points_from_bounds([-.55, -.5, -.95], [0.55, 0.75, 0.4], 20)).float().unsqueeze(0)
    logits = get_logits(dec, torch.from_numpy(g['latent_a']), grid, nbatch_points=3000)
    assert logits.shape == (8000,) and logits.dtype == np.float32
    assert np.abs(logits - g['logits20_a']).max() < 1e-5


def test_autograd_flows_through_composite_path():
    dec = make_ensemble(0).train()
    x = torch.randn(1, 16, 3) * 0.2
    x.requires_grad_(True)
    z = torch.zeros(1, 1, 1344, requires_grad=True)
    s, anc = dec(x, z, None)
    (gx,) = torch.autograd.grad(s.sum(), x, create_graph=True)
    (gx.pow(2).sum() + anc.sum()).backward()                      # double backward (eikonal-style)
    assert z.grad is not None and torch.isfinite(z.grad).all() and z.grad.abs().sum() > 0


def test_install_as_nphm_aliases():
    import nphm_b200
    import sys
    saved = {k: v for k, v in sys.modules.items() if k == 'NPHM' or k.startswith('NPHM.')}
    try:
        nphm_b200.install_as_nphm(force=True)
        from NPHM.models.EnsembledDeepSDF import FastEnsembleDeepSDFMirrored as A
        from NPHM.models.deepSDF import DeepSDF, DeformationNetwork      # noqa: F401
        from NPHM.models.reconstruction import deform_mesh, get_logits, get_logits_backward      # noqa: F401
        from NPHM.utils.reconstruction import create_grid_points_from_bounds, mesh_from_logits    # noqa: F401
        from nphm_b200.models.EnsembledDeepSDF import FastEnsembleDeepSDFMirrored as B
        assert A is B
    finally:
        for k in [k for k in sys.modules if k == 'NPHM' or k.startswith('NPHM.')]:
            del sys.modules[k]
        sys.modules.update(saved)


def test_install_as_nphm_keeps_the_rest_of_the_reference_importable(tmp_path):
    """After install_as_nphm() every NPHM.* name the reference's scripts import must still resolve: the seven hot-path
    modules here, everything else (env_paths, data.*, evaluation.*, models.training / loss_functions / training_corresp,
    utils.mesh_operations) in the reference checkout on sys.path.  A stand-in checkout with the same module names and
    the same inter-module imports as /root/reference/src/NPHM is used (the real one needs trimesh, wandb, ...)."""
    import nphm_b200
    import sys
    pkg = tmp_path / 'NPHM'
    for d in ('', 'data', 'evaluation', 'models', 'utils'):
        (pkg / d).mkdir(exist_ok=True)
    (pkg / '__init__.py').write_text('')
    (pkg / 'data' / '__init__.py').write_text('')
    (pkg / 'env_paths.py').write_text('ASSETS = "/nowhere/"\n')
    (pkg / 'data' / 'manager.py').write_text('from NPHM import env_paths\nclass DataManager:\n    root = env_paths.ASSETS\n')
    (pkg / 'data' / 'face_dataset.py').write_text('from NPHM.data.manager import DataManager\nclass ScannerData:\n    m = DataManager\n')
    (pkg / 'evaluation' / 'metrics.py').write_text('def eval_pointcloud():\n    return 1\n')
    (pkg / 'utils' / 'mesh_operations.py').write_text('def cut_trimesh_vertex_mask():\n    return 2\n')
    # the reference's own (slow) versions of the shadowed modules must NOT win
    (pkg / 'models' / 'deepSDF.py').write_text('raise ImportError("reference deepSDF imported instead of the mirror")\n')
    (pkg / 'models' / 'reconstruction.py').write_text('raise ImportError("reference reconstruction imported")\n')
    (pkg / 'models' / 'loss_functions.py').write_text(
        'from NPHM.models.diff_operators import gradient\nfrom NPHM.models.iterative_root_finding import search, jac, nabla\n'
        'def compute_loss():\n    return gradient\ndef compute_loss_corresp_forward():\n    return search\n')
    (pkg / 'models' / 'training.py').write_text(
        'from NPHM.models.loss_functions import compute_loss\nfrom NPHM.models.reconstruction import get_logits\n'
        'from NPHM.utils.reconstruction import create_grid_points_from_bounds, mesh_from_logits\n'
        'from NPHM import env_paths\nclass TrainerAutoDecoder:\n    fn = staticmethod(get_logits)\n')
    (pkg / 'models' / 'training_corresp.py').write_text(
        'from NPHM.models.loss_functions import compute_loss_corresp_forward\nfrom NPHM.models.reconstruction import get_logits, deform_mesh\n'
        'class TrainerAutoDecoder:\n    fn = staticmethod(deform_mesh)\n')
    saved = {k: v for k, v in sys.modules.items() if k == 'NPHM' or k.startswith('NPHM.')}
    for k in saved:
        del sys.modules[k]
    sys.path.insert(0, str(tmp_path))
    try:
        for mode in ('fresh', 'reference imported first'):
            for k in [k for k in sys.modules if k == 'NPHM' or k.startswith('NPHM.')]:
                del sys.modules[k]
            if mode != 'fresh':
                from NPHM import env_paths as _e          # noqa: F401  (what INTEGRATION.md's one-liner does first)
                with pytest.raises(RuntimeError):
                    nphm_b200.install_as_nphm()
                nphm_b200.install_as_nphm(force=True)
            else:
                nphm_b200.install_as_nphm()
            # scripts/fitting/fitting_pointclouds.py:1-7, scripts/training/train*.py:9-11, scripts/evaluation/eval.py
            from NPHM import env_paths
            import NPHM.env_paths as env_paths2
            from NPHM.data.manager import DataManager
            from NPHM.data.face_dataset import ScannerData
            from NPHM.evaluation.metrics import eval_pointcloud
            from NPHM.utils.mesh_operations import cut_trimesh_vertex_mask
            from NPHM.models.training import TrainerAutoDecoder
            from NPHM.models import training_corresp as training
            from NPHM.models.loss_functions import compute_loss, compute_loss_corresp_forward
            from NPHM.models.deepSDF import DeepSDF, DeformationNetwork
            from NPHM.models.EnsembledDeepSDF import FastEnsembleDeepSDFMirrored
            from NPHM.models.fitting import inference_identity_space, inference_iterative_root_finding_joint
            from NPHM.models.reconstruction import deform_mesh, get_logits, get_logits_backward
            from NPHM.utils.reconstruction import create_grid_points_from_bounds, mesh_from_logits
            from NPHM.models.iterative_root_finding import search, jac, nabla
            from NPHM.models.diff_operators import gradient
            import nphm_b200.models.reconstruction as mine
            import nphm_b200.models.deepSDF as mine_sdf
            assert env_paths is env_paths2 and env_paths.ASSETS == '/nowhere/' and DataManager.root == '/nowhere/'
            assert ScannerData.m is DataManager and eval_pointcloud() == 1 and cut_trimesh_vertex_mask() == 2
            assert get_logits is mine.get_logits and DeepSDF is mine_sdf.DeepSDF
            assert TrainerAutoDecoder.fn is mine.get_logits and training.TrainerAutoDecoder.fn is mine.deform_mesh
            assert compute_loss() is gradient and compute_loss_corresp_forward() is search
    finally:
        sys.path.remove(str(tmp_path))
        for k in [k for k in sys.modules if k == 'NPHM' or k.startswith('NPHM.')]:
            del sys.modules[k]
        sys.modules.update(saved)


def test_library_exports_every_declared_symbol():
    from nphm_b200 import _native
    header = open(os.path.join(ROOT, 'include', 'nphm_b200.h')).read()
    declared = set(re.findall(r'\b(nphm_[a-z_0-9]+)\s*\(', header))
    assert declared == set(_native.EXPORTED_SYMBOLS), declared ^ set(_native.EXPORTED_SYMBOLS)
    so = os.path.join(ROOT, 'nphm_b200', 'libnphm_b200.so')
    if not os.path.exists(so):
        pytest.fail('libnphm_b200.so not built: run __graft_entry__.build()')
    lib = ctypes.CDLL(so)
    for name in declared:
        assert hasattr(lib, name), name
    lib.nphm_abi_version.restype = ctypes.c_int
    assert lib.nphm_abi_version() == 1


def test_fused_path_refuses_to_run_without_library(monkeypatch):
    """The product path must fail loudly when the CUDA extension is missing."""
    from nphm_b200 import _native
    monkeypatch.setattr(_native, '_lib', None)
    monkeypatch.setattr(_native, '_LIB_PATH', '/nonexistent/libnphm_b200.so')
    with pytest.raises(_native.NativeError):
        _native.lib()


def test_mc_tables_identical_in_oracle_and_product():
    a = open(os.path.join(ROOT, 'oracle', 'mc_tables_oracle.h')).read().split('\n', 4)[4]
    b = open(os.path.join(ROOT, 'nphm_b200', 'csrc', 'mc_tables.h')).read().split('\n', 4)[4]
    assert a == b
    import subprocess, sys
    assert subprocess.run([sys.executable, os.path.join(ROOT, 'tools', 'gen_mc_tables.py')]).returncode == 0


def test_bench_reference_arm_contract(tmp_path):
    """`bench.py --impl reference`: rank 0 prints one JSON line with the contract's keys, other ranks exit 0 silently."""
    import json, os, subprocess, sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    cmd = [sys.executable, os.path.join(root, 'bench.py'), '--impl', 'reference', '--steps', '1', '--warmup', '0', '--res', '32',
           '--cpu-sample-chunks', '1']
    env = dict(os.environ, RANK='1', WORLD_SIZE='2', LOCAL_RANK='1')
    r = subprocess.run(cmd, env=env, capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and r.stdout.strip() == ''
    from oracle import ref_loader
    if not ref_loader.available():
        pytest.skip('rank 0 times the reference modules themselves: build oracle/_ref with oracle/make_ref.py')
    env = dict(os.environ, RANK='0', WORLD_SIZE='1', LOCAL_RANK='0')
    r = subprocess.run(cmd, env=env, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line['impl'] == 'reference' and line['metric'] == 'sdf_query_points_per_s' and line['unit'] == 'points/s'
    assert line['higher_is_better'] is True and line['value'] > 0 and line['e2e']['value'] == line['value']
    assert line['e2e']['h2d_bytes_per_step'] == 0 and line['e2e']['d2h_bytes_per_step'] == 0
    assert line['cpu_baseline']['kind'] == 'reference' and line['cpu_baseline']['cores'] >= 1
    assert 'workload' in line['config']
