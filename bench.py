#!/usr/bin/env python
"""Benchmark of the NPHM hot path on B200 (contract: see the task statement / DESIGN.md section "Measurement").

N = 1 (BASELINE.json configs[1]): a step = SDF of the 40-member ensemble on the 256^3 grid + marching cubes of one head.
  value   SDF query points/s, inputs (latent, weights) resident in HBM, grid generated in-kernel
  e2e     the same through the reference-facing drop-in API with HOST buffers: pinned latent -> H2D,
          get_logits(...) -> numpy volume (D2H), mesh_from_logits(numpy) -> mesh (H2D volume, D2H mesh)
  stock_gpu   the UNMODIFIED reference modules (.cuda(), its own get_logits, 672 chunks) on the same B200, full volume;
          the volume it returns is also compared with ours (parity on all 16.7 M points)
  cpu_baseline  the UNMODIFIED reference modules on the host cores, bounded sample (+ C marching cubes on the step's volume)
N > 1 (BASELINE.json configs[4]): a step = ONE head on the 512^3 grid, x-slabs sharded over the N ranks
  (nphm_b200.distributed.extract_mesh_sharded): per-rank SDF + marching-cubes count, all_gather of the counts, emit with
  global ids, batched NVLink gather of the mesh on rank 0.  STRONG scaling of one mesh extraction; every rank then handles
  res^3/N points, i.e. the per-GPU work of the N = 1 run at N = 8.  The independent-replica number (one 256^3 head
  per rank, no collective) is reported as a secondary key.

    python bench.py --gpus 1 --steps 5 --warmup 3
    python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N --steps K --warmup W
    python bench.py --impl reference        # CPU arm: the reference's own modules (oracle/_ref) on the host cores
    python bench.py --gpus 1 --steps 5 --warmup 3 --dump-outputs DIR       # + the last timed step's outputs as DIR/*.npy
"""
import argparse
import atexit
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

sys.dont_write_bytecode = True    # the tree may be read-only: no __pycache__ next to the imported modules
ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tests'))

MINI = [-.55, -.5, -.95]
MAXI = [0.55, 0.75, 0.4]
FLOP_PER_POINT = 9.616e6          # dense reference formulation, SURVEY.md 8(d)
CHUNK = 25000                     # nbatch_points of scripts/fitting -sample (fitting_pointclouds.py:208)
L2_NOTE = 'flushed between iterations (256 MB write)'
DUMP_BYTES = 63 * 10 ** 6        # array data of --dump-outputs: 64 MB in all with room for the .npy headers
DUMP_SEED = 0


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=5)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='auto', choices=['auto', 'simt', 'tc', 'reference'])
    ap.add_argument('--res', type=int, default=0, help='grid resolution (default 256 at N=1, 512 at N>1)')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-stock-gpu', action='store_true')
    ap.add_argument('--cpu-sample-chunks', type=int, default=2)
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help='after the timed steps, write what the last one computed as DIR/<name>.npy (float32/float64, '
                         'at most 64 MB in all; larger outputs as a sample of rows drawn with a fixed seed)')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs and args.impl == 'reference':
        ap.error('--dump-outputs writes what this project computes; the reference arm does not run it')
    return args


def dump_outputs(dirname, arrays):
    """Writes each array (numpy or torch, rows along the first axis) as ``dirname/<name>.npy``: floating point as is,
    integers as float64 (exact below 2^53).  The smallest arrays are written first, each whole if it fits an equal share
    of what is left of DUMP_BYTES; a larger one is replaced by the rows at ``DUMP_SEED``-seeded random positions (sorted),
    the same positions in every run with the same row count, so two builds can be compared output for output."""
    os.makedirs(dirname, exist_ok=True)
    host = {}
    for name, a in arrays.items():
        a = a.detach().cpu().numpy() if hasattr(a, 'detach') else np.asarray(a)
        host[name] = a if a.dtype in (np.float32, np.float64) else a.astype(np.float64)
    left = DUMP_BYTES
    for i, name in enumerate(sorted(host, key=lambda k: host[k].nbytes)):
        a = host[name]
        share = left // (len(host) - i)
        if a.nbytes > share:
            row_bytes = max(1, a.nbytes // max(1, a.shape[0]))
            rows = np.random.default_rng(DUMP_SEED).choice(a.shape[0], share // row_bytes, replace=False)
            a = a[np.sort(rows)]
        np.save(os.path.join(dirname, name + '.npy'), a)
        left -= a.nbytes


def workload_name(res, world):
    """One name for both arms of the benchmark."""
    if world > 1:
        return ('single-head %d^3 grid mesh extraction (40-member ensemble SDF, seeded random weights + marching cubes), '
                'x-slabs sharded over the GPUs, mesh gathered on rank 0' % res)
    return ('single-head %d^3 grid SDF (40-member ensemble, seeded random weights) + marching cubes, random latent' % res)


def bench_config(res, world):
    return {'workload': workload_name(res, world), 'res': res, 'nbatch_points': CHUNK, 'l2': L2_NOTE}


def default_res(args):
    return args.res or (256 if args.gpus <= 1 else 512)


# ------------------------------------------------------------------------------------------------ reference legs
def reference_setup(device='cpu'):
    """The UNMODIFIED reference modules (oracle/_ref) with the SURVEY 8(d) synthetic model + latent."""
    import torch
    from oracle import ref_loader as R
    ns = R.load()
    dec = R.make_ensemble(ns, 0, device=device).eval()
    lat = R.sample_latent(ns, 1).to(device)
    return ns, dec, lat, torch


def grid_chunk(res, chunk_id):
    """Points [chunk_id*CHUNK, +CHUNK) of the res^3 grid, computed like utils/reconstruction.py:5-20 -> float32 (n,3)."""
    total = res ** 3
    first = chunk_id * CHUNK
    idx = np.arange(first, min(first + CHUNK, total))
    axes = [np.linspace(MINI[a], MAXI[a], res) for a in range(3)]
    return np.stack([axes[0][idx // (res * res)], axes[1][(idx // res) % res], axes[2][idx % res]], axis=1).astype(np.float32)


class CpuReference:
    """Times the reference's own ``get_logits`` (models/reconstruction.py:6-25) on whole chunks of the grid, all host
    threads (torch intra-op pool)."""

    def __init__(self):
        self.ns, self.dec, self.lat, torch = reference_setup('cpu')
        self.torch = torch
        self.threads = os.cpu_count() or 1
        torch.set_num_threads(self.threads)

    def time_chunks(self, res, chunk_ids):
        torch = self.torch
        pts = torch.from_numpy(np.concatenate([grid_chunk(res, c) for c in chunk_ids], axis=0)).unsqueeze(0)
        t0 = time.perf_counter()
        out = self.ns.reconstruction.get_logits(self.dec, self.lat, pts, nbatch_points=CHUNK)
        return time.perf_counter() - t0, pts.shape[1], out


def spread_chunks(res, n, offset=0):
    """n chunk ids spread evenly over the grid (near and far field, chunk-boundary classes all occur)."""
    n_chunks = (res ** 3 + CHUNK - 1) // CHUNK - 1            # full chunks only
    return [int((offset + (i + 0.5) * n_chunks / n)) % n_chunks for i in range(n)]


def c_marching_cubes_seconds(volume_neg_applied):
    """Single-threaded C restatement of PyMCubes (oracle/mc_oracle.c; mcubes itself is not in this image) on a volume."""
    from oracle import nphm_oracle as O
    t0 = time.perf_counter()
    v, t = O.marching_cubes(volume_neg_applied, 0.0)
    return time.perf_counter() - t0, len(v), len(t)


def stock_gpu_run(res, dev, quick_chunks=0):
    """The reference as its users run it: unmodified modules .cuda(), its own get_logits over the (1, res^3, 3) CUDA grid
    in chunks of 25 000 with a D2H per chunk.  Returns (dict, volume numpy)."""
    ns, dec, lat, torch = reference_setup(dev)
    grid = torch.from_numpy(ns.utils_reconstruction.create_grid_points_from_bounds(MINI, MAXI, res)).to(dev, dtype=torch.float)
    grid = grid.reshape(1, -1, 3)                               # fitting_pointclouds.py:168-170
    if quick_chunks:
        grid = grid[:, :quick_chunks * CHUNK]
    ns.reconstruction.get_logits(dec, lat, grid[:, :3 * CHUNK], nbatch_points=CHUNK)       # warm-up (cuBLAS, allocator)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    vol = ns.reconstruction.get_logits(dec, lat, grid, nbatch_points=CHUNK)
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    n = grid.shape[1]
    del grid
    torch.cuda.empty_cache()
    return {'value': n / dt, 'unit': 'points/s', 'seconds': dt, 'points': int(n),
            'what': 'unmodified reference modules (oracle/_ref) .cuda(): get_logits, nbatch_points=25000, fp32 '
                    '(torch default: TF32 off), wall clock incl. its per-chunk D2H'}, vol


def run_reference_arm(args):
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    world = args.gpus
    res = default_res(args)
    total = res ** 3
    ref = CpuReference()
    per_step = max(1, args.cpu_sample_chunks // 2)
    n_warm, n_steps = max(args.warmup, 1), args.steps
    ids = spread_chunks(res, (n_warm + n_steps) * per_step)
    times, pts_per_step = [], 0
    for i in range(n_warm + n_steps):
        dt, pts_per_step, _ = ref.time_chunks(res, ids[i * per_step:(i + 1) * per_step])
        if i >= n_warm:
            times.append(dt)
    med = float(np.median(times))
    sdf_rate = pts_per_step / med
    # marching cubes: the C restatement on the step's own volume when a GPU can produce it with the reference itself
    mc = {'t_mc_s': None}
    stock = None
    try:
        import torch
        if torch.cuda.is_available() and res <= 256:
            stock, vol = stock_gpu_run(res, torch.device('cuda', 0))
            t_mc, nv, nt = c_marching_cubes_seconds(-vol.reshape(res, res, res))
            mc = {'t_mc_s': t_mc, 'vertices': nv, 'triangles': nt, 'volume': 'the step\'s own SDF volume (reference on the GPU)'}
    except Exception as exc:          # noqa: BLE001 - the GPU leg is a bonus for this arm
        mc['error'] = repr(exc)
    if mc['t_mc_s'] is None:
        from conftest import sphere_volume
        t_mc, nv, nt = c_marching_cubes_seconds(sphere_volume(min(res, 256), radius=0.37))
        t_mc *= (res / min(res, 256)) ** 3
        mc = {'t_mc_s': t_mc, 'vertices': nv, 'triangles': nt, 'volume': 'sphere SDF (no GPU for the reference volume)'}
    est_step = total / sdf_rate + mc['t_mc_s']
    value = total / est_step
    cores = ref.threads
    sample = ('%d timed steps (median) of %d chunk(s) x %d grid points spread over the %d^3 grid through the UNMODIFIED '
              'reference get_logits (oracle/_ref, torch CPU fp32, %d threads), %d discarded warm-up step(s); + single-threaded '
              'C restatement of PyMCubes on %s; value = points of the full grid / (points/sdf_rate + t_mc)'
              % (n_steps, per_step, CHUNK, res, cores, n_warm, mc['volume']))
    line = {
        'impl': 'reference', 'metric': 'sdf_query_points_per_s', 'value': value, 'unit': 'points/s',
        'n_gpus': world, 'steps': args.steps, 'warmup': args.warmup,
        'ms_per_step': 1e3 * med, 'higher_is_better': True, 'scaling': 'strong' if world > 1 else 'weak',
        'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
        'config': bench_config(res, world),
        'cpu_baseline': {'value': value, 'unit': 'points/s', 'cores': cores, 'kind': 'reference', 'sample': sample,
                         'detail': {'points_per_step': int(pts_per_step), 'step_s_median': med,
                                    'step_s_min': float(min(times)), 'step_s_max': float(max(times)),
                                    'sdf_points_per_s': sdf_rate, 'est_full_step_s': est_step, **mc}},
        'e2e': {'value': value, 'unit': 'points/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
        'note': 'ms_per_step is the measured wall time of one bounded sample step, not of the full grid',
    }
    if stock is not None:
        line['stock_gpu'] = stock
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------ clocks
class ClockSampler:
    Q = ('index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,'
         'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,'
         'clocks_event_reasons.sw_power_cap')

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.proc = None
        self.lines = []
        self.first = 0

    def start(self):
        if os.environ.get('NPHM_BENCH_NO_SAMPLER'):
            return
        try:
            self.proc = subprocess.Popen(['nvidia-smi', '-i', str(self.gpu), '--query-gpu=' + self.Q,
                                          '--format=csv,noheader,nounits', '-lms', os.environ.get('NPHM_BENCH_SAMPLE_MS', '200')],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            atexit.register(self.proc.kill)      # no sampler left running when the benchmark fails before stop()
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def mark(self):
        """Start of the timed region: earlier samples (taken while nvidia-smi initialised, during warm-up) are dropped."""
        self.first = len(self.lines)

    def stop(self):
        if self.proc is None:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons, power = [], [], set(), []
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        for ln in self.lines[self.first:]:
            f = [x.strip() for x in ln.split(',')]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2])); power.append(float(f[3]))
            except ValueError:
                continue
            for name, val in zip(names, f[5:9]):
                if val.lower().startswith('active'):
                    reasons.add(name)
        if not sm:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['no samples']}
        return {'sm_mhz': float(np.median(sm)), 'sm_max_mhz': float(max(mx)), 'reasons': sorted(reasons),
                'power_w_max': max(power), 'samples': len(sm)}


def load_peaks():
    try:
        return json.load(open(os.path.join(ROOT, 'MEASURED_PEAKS.json')))
    except Exception:
        return {}


def roofline_block(res_key, flops, sdf_ms, note_extra=''):
    peaks = load_peaks()
    peak_tf = peaks.get('bf16_tflops_sustained', None)
    peak_src = 'measured (MEASURED_PEAKS.json bf16_tflops_sustained)'
    if peak_tf is None:
        peak_tf, peak_src = 1590.0, 'fallback (B200_PROFILING.md)'
    achieved_tf = flops / (sdf_ms * 1e-3) / 1e12
    traffic, traffic_src = None, 'no ncu capture recorded for this resolution'
    try:
        with open(os.path.join(ROOT, 'profiles', 'traffic.json')) as f:
            rec = json.load(f).get(str(res_key))
        if rec:
            traffic = rec['dram_bytes_read'] + rec['dram_bytes_write']
            traffic_src = 'bytes, ' + rec['source'] + ' (profiles/traffic.json)'
    except (OSError, ValueError, KeyError):
        pass
    return {'bound': 'tensor', 'achieved': achieved_tf, 'peak': peak_tf, 'unit': 'TFLOP/s',
            'frac': achieved_tf / peak_tf, 'traffic': traffic,
            'note': 'dominant kernel = fused ensemble SDF query; algorithmic 9.616 MFLOP/point (dense reference '
                    'formulation) / CUDA-event time of the query' + note_extra + '; peak: ' + peak_src +
                    '; traffic: ' + traffic_src}


# ------------------------------------------------------------------------------------------------ GPU arm, N = 1
def run_single(args, torch, dev):
    from conftest import make_ensemble, sample_latent
    from nphm_b200 import _native
    from nphm_b200.models.reconstruction import get_logits
    from nphm_b200.utils.reconstruction import create_grid_points_from_bounds, mesh_from_logits

    res = default_res(args)
    total = res ** 3
    dec = make_ensemble(0, device=dev).eval()
    eng = dec.engine()
    lat = sample_latent(1).to(dev)
    volume = torch.empty(total, device=dev, dtype=torch.float32)
    flush = torch.empty(64 * 1024 * 1024, device=dev, dtype=torch.float32)      # 256 MB > 126 MB L2
    launches = {'n': 0}
    per_step_launches = _native.launches_per_grid_query(args.impl) + _native.MC_LAUNCHES

    def step_device():
        """grid SDF (in-kernel grid) + marching cubes, everything resident on the device."""
        eng.query_grid(lat, MINI, MAXI, res, 0, total, quirk_period=CHUNK, out=volume)
        v, t = _native.marching_cubes_device(volume.view(res, res, res), 0.0, negate=True)
        launches['n'] += per_step_launches
        return v, t

    sampler = ClockSampler(dev.index)
    n_warm = max(args.warmup, 3)
    for i in range(n_warm):
        if i == n_warm - 1:
            sampler.start()             # nvidia-smi takes driver locks while it initialises: let that happen in warm-up
        step_device()
        flush.zero_()
    import gc
    gc.collect()
    gc.disable()                        # no collector pauses inside the timed regions (host sits between MC passes)
    torch.cuda.synchronize()
    sampler.mark()
    launches['n'] = 0
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    kev = [[torch.cuda.Event(enable_timing=True) for _ in range(4)] for _ in range(args.steps)]
    ev[0].record()
    n_tris = 0
    for i in range(args.steps):
        kev[i][0].record()
        eng.query_grid(lat, MINI, MAXI, res, 0, total, quirk_period=CHUNK, out=volume)
        kev[i][1].record()
        v, t = _native.marching_cubes_device(volume.view(res, res, res), 0.0, negate=True)
        kev[i][2].record()
        launches['n'] += per_step_launches
        n_tris = t.shape[0]
        if i == args.steps - 1:
            last_mesh = (v, t)          # for --dump-outputs (the last step: no allocation follows in the loop)
        del v, t                        # the mesh buffers go back to torch's caching allocator (no cudaMalloc in the loop)
        flush.zero_()                   # L2 flush between timed iterations (inside the timed region)
        kev[i][3].record()
    ev[1].record()
    torch.cuda.synchronize()
    clocks = sampler.stop()
    ms_total = ev[0].elapsed_time(ev[1])
    sdf_ms = float(np.mean([k[0].elapsed_time(k[1]) for k in kev]))   # prep kernels + the ensemble kernel
    mc_ms = float(np.mean([k[1].elapsed_time(k[2]) for k in kev]))    # marching cubes kernels + count readback
    flush_ms = float(np.mean([k[2].elapsed_time(k[3]) for k in kev]))
    ms_per_step = ms_total / args.steps
    value = total / (ms_per_step * 1e-3)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {'sdf': volume, 'vertices': last_mesh[0], 'triangles': last_mesh[1]})
    del last_mesh

    # ---- opt-in pruned kernel (reported separately; NOT the dense reference computation) ---------------------
    pruned = None
    if args.impl in ('auto', 'tc'):
        tau = 1e-8
        eng.set_prune_threshold(tau)
        ref_vol = volume.clone()
        pv = torch.empty_like(volume)
        for _ in range(2):
            eng.query_grid(lat, MINI, MAXI, res, 0, total, quirk_period=CHUNK, out=pv, impl='tc_pruned')
        torch.cuda.synchronize()
        p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        p0.record()
        for _ in range(args.steps):
            eng.query_grid(lat, MINI, MAXI, res, 0, total, quirk_period=CHUNK, out=pv, impl='tc_pruned')
        p1.record()
        torch.cuda.synchronize()
        pms = p0.elapsed_time(p1) / args.steps
        pruned = {'tau': tau, 'sdf_ms': pms, 'value': total / (pms * 1e-3), 'unit': 'points/s',
                  'max_abs_diff_vs_dense': float((pv - ref_vol).abs().max().item()),
                  'note': 'NPHM_IMPL_TC_PRUNED: members with normalised blend weight < tau on a whole 8x4x4 tile are skipped'}
        del pv, ref_vol

    # ---- end to end through the drop-in API with host buffers ---------------------------------------------
    grid_points = torch.from_numpy(create_grid_points_from_bounds(MINI, MAXI, res)).to(dev, dtype=torch.float)
    grid_points = grid_points.reshape(1, -1, 3)                 # uploaded once, like fitting_pointclouds.py:166-170
    lat_host = lat.cpu().pin_memory()
    h2d = d2h = 0

    def step_e2e():
        nonlocal h2d, d2h
        z = lat_host.to(dev, non_blocking=True)                                  # H2D: latent
        logits = get_logits(dec, z, grid_points, nbatch_points=CHUNK)            # D2H: volume (numpy)
        mesh = mesh_from_logits(logits, MINI, MAXI, res)                         # H2D volume, GPU MC, D2H mesh
        h2d = lat_host.numel() * 4 + logits.nbytes
        d2h = logits.nbytes + np.asarray(mesh.vertices).nbytes + np.asarray(mesh.faces).nbytes
        return mesh

    for _ in range(2):
        step_e2e()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    e2e_steps = max(2, min(args.steps, 5))
    for _ in range(e2e_steps):
        step_e2e()
    torch.cuda.synchronize()
    e2e_value = total / ((time.perf_counter() - t0) / e2e_steps)
    gc.enable()
    del grid_points

    line = {
        'metric': 'sdf_query_points_per_s', 'value': value, 'unit': 'points/s', 'n_gpus': 1,
        'steps': args.steps, 'warmup': n_warm, 'ms_per_step': ms_per_step,
        'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
        'config': bench_config(res, 1), 'impl_kernel': args.impl, 'triangles': int(n_tris),
        'meshes_per_s': 1.0 / (ms_per_step * 1e-3),
        'sdf_ms': sdf_ms, 'mc_ms': mc_ms, 'l2_flush_ms': flush_ms,
        'gpu_launches': launches['n'],
        'clocks': clocks,
        'e2e': {'value': e2e_value, 'unit': 'points/s', 'h2d_bytes_per_step': int(h2d), 'd2h_bytes_per_step': int(d2h),
                'api': 'get_logits + mesh_from_logits (drop-in, numpy in/out)'},
        'roofline': roofline_block(res, FLOP_PER_POINT * total, sdf_ms),
    }
    if pruned is not None:
        line['pruned_opt_in'] = pruned

    # ---- the reference itself: stock GPU path on this B200 (+ parity on the whole volume), CPU sample -----------
    ours = volume.cpu().numpy()
    if not args.no_stock_gpu:
        try:
            stock, ref_vol = stock_gpu_run(res, dev)
            diff = np.abs(ours - ref_vol)
            stock['speedup_value'] = value / stock['value']
            stock['speedup_e2e'] = e2e_value / stock['value']
            stock['parity_max_abs_diff'] = float(diff.max())
            stock['parity_points'] = int(diff.size)
            stock['parity_tolerance'] = 1e-5
            line['stock_gpu'] = stock
        except Exception as exc:      # noqa: BLE001
            line['stock_gpu'] = {'unavailable': repr(exc)}
    if not args.no_cpu_baseline:
        try:
            ref = CpuReference()
            ids = spread_chunks(res, args.cpu_sample_chunks + 1, offset=3)
            ref.time_chunks(res, ids[:1])                                   # discarded warm-up chunk
            dts = []
            for c in ids[1:]:
                dt, npts, out = ref.time_chunks(res, [c])
                dts.append(dt)
                # bonus: the CPU reference's chunk against our volume (same indices)
                line.setdefault('cpu_parity_max_abs_diff', 0.0)
                line['cpu_parity_max_abs_diff'] = max(line['cpu_parity_max_abs_diff'],
                                                      float(np.abs(out - ours[c * CHUNK:c * CHUNK + npts]).max()))
            rate = CHUNK / float(np.median(dts))
            t_mc, nv, nt = c_marching_cubes_seconds(-ours.reshape(res, res, res))
            est = total / rate + t_mc
            line['cpu_baseline'] = {
                'value': total / est, 'unit': 'points/s', 'cores': ref.threads, 'kind': 'reference',
                'sample': '%d chunks x %d grid points through the UNMODIFIED reference get_logits (oracle/_ref, torch CPU fp32, '
                          '%d threads; median, one warm-up chunk discarded) + single-threaded C restatement of PyMCubes on this '
                          'step\'s volume (%.2f s); extrapolated to %d^3' % (len(dts), CHUNK, ref.threads, t_mc, res),
                'detail': {'chunk_s': dts, 'sdf_points_per_s': rate, 't_mc_s': t_mc, 'est_full_step_s': est}}
        except Exception as exc:      # noqa: BLE001
            line['cpu_baseline'] = {'unavailable': repr(exc)}
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------ GPU arm, N > 1
def run_sharded(args, torch, dist, dev, world, rank):
    from conftest import make_ensemble, sample_latent
    from nphm_b200 import _native
    from nphm_b200.distributed import ensemble_slab_fn, extract_mesh_sharded, plan_slabs, slab_planes

    res = default_res(args)
    total = res ** 3
    dec = make_ensemble(0, device=dev).eval()
    eng = dec.engine()
    lat = sample_latent(1).to(dev)                             # the same head on every rank
    fn = ensemble_slab_fn(dec, lat, MINI, MAXI, res, CHUNK)
    flush = torch.empty(64 * 1024 * 1024, device=dev, dtype=torch.float32)
    per_step_launches = _native.launches_per_grid_query(args.impl) + _native.MC_LAUNCHES

    def barrier():
        dist.barrier()
        torch.cuda.synchronize()

    sampler = ClockSampler(dev.index)
    n_warm = max(args.warmup, 3)
    for i in range(n_warm):
        if i == n_warm - 1:
            sampler.start()
        extract_mesh_sharded(fn, res, 0.0, True)
        flush.zero_()
    import gc
    gc.collect()
    gc.disable()
    barrier()
    sampler.mark()
    phases = {}
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    ev[0].record()
    for _ in range(args.steps):
        verts, tris = extract_mesh_sharded(fn, res, 0.0, True, timings=phases)
        flush.zero_()
    ev[1].record()
    barrier()
    clocks = sampler.stop()
    keys = ['sdf_ms', 'mc_count_ms', 'count_exchange_ms', 'mc_emit_ms', 'gather_ms']
    t = torch.tensor([ev[0].elapsed_time(ev[1])] + [phases.get(k, 0.0) for k in keys] + [float(phases.get('gather_bytes', 0))],
                     device=dev, dtype=torch.float64)
    tmax = t.clone()
    dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
    tsum = t.clone()
    dist.all_reduce(tsum, op=dist.ReduceOp.SUM)
    ms_per_step = tmax[0].item() / args.steps
    phase_max = {k: tmax[1 + i].item() / args.steps for i, k in enumerate(keys)}
    gather_bytes = int(tsum[-1].item())
    value = total / (ms_per_step * 1e-3)
    if args.dump_outputs and rank == 0:                        # the mesh is gathered on rank 0 only
        dump_outputs(args.dump_outputs, {'vertices': verts, 'triangles': tris})

    # ---- e2e: public API with host buffers (pinned latent H2D every step, the mesh D2H on rank 0) ------------------
    lat_host = lat.cpu().pin_memory()
    h2d = d2h = 0

    def step_e2e():
        nonlocal h2d, d2h
        z = lat_host.to(dev, non_blocking=True)
        f = ensemble_slab_fn(dec, z, MINI, MAXI, res, CHUNK)
        v, tr = extract_mesh_sharded(f, res, 0.0, True)
        h2d = lat_host.numel() * 4
        if v is not None:
            vh, th = v.cpu().numpy(), tr.cpu().numpy()
            d2h = vh.nbytes + th.nbytes
    step_e2e()
    barrier()
    t0 = time.perf_counter()
    e2e_steps = max(2, min(args.steps, 5))
    for _ in range(e2e_steps):
        step_e2e()
    barrier()
    e2e_s = torch.tensor([(time.perf_counter() - t0) / e2e_steps], device=dev, dtype=torch.float64)
    dist.all_reduce(e2e_s, op=dist.ReduceOp.MAX)
    e2e_value = total / e2e_s.item()

    # ---- secondary: independent replicas (one 256^3 head per rank, no collective) ------------------------------
    r_res = 256
    r_total = r_total_pts = r_res ** 3
    r_vol = torch.empty(r_total, device=dev, dtype=torch.float32)
    r_lat = sample_latent(1 + rank).to(dev)
    for _ in range(2):
        eng.query_grid(r_lat, MINI, MAXI, r_res, 0, r_total, quirk_period=CHUNK, out=r_vol)
    barrier()
    r0, r1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    r0.record()
    r_steps = max(2, min(args.steps, 5))
    for _ in range(r_steps):
        eng.query_grid(r_lat, MINI, MAXI, r_res, 0, r_total, quirk_period=CHUNK, out=r_vol)
        v, tr = _native.marching_cubes_device(r_vol.view(r_res, r_res, r_res), 0.0, negate=True)
        del v, tr
        flush.zero_()
    r1.record()
    barrier()
    r_ms = torch.tensor([r0.elapsed_time(r1) / r_steps], device=dev, dtype=torch.float64)
    dist.all_reduce(r_ms, op=dist.ReduceOp.MAX)
    del r_vol
    gc.enable()

    # ---- identical to the single-GPU extraction? (rank 0 recomputes the whole mesh alone, outside the timed region) --
    identical = None
    if rank == 0:
        try:
            vol, _ = eng.query_grid(lat, MINI, MAXI, res, 0, total, CHUNK)
            v1, t1 = _native.marching_cubes_device(vol.view(res, res, res), 0.0, negate=True)
            identical = bool(torch.equal(v1, verts) and torch.equal(t1, tris))
            del vol, v1, t1
        except Exception as exc:      # noqa: BLE001
            identical = 'check failed: %r' % (exc,)
    if rank == 0:
        planes = [slab_planes(*c)[1] for c in plan_slabs(res, world)]
        sdf_points_max = max(planes) * res * res
        limiting = max(phase_max, key=phase_max.get)
        line = {
            'metric': 'sdf_query_points_per_s', 'value': value, 'unit': 'points/s', 'n_gpus': world,
            'steps': args.steps, 'warmup': n_warm, 'ms_per_step': ms_per_step,
            'higher_is_better': True, 'scaling': 'strong', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
            'config': bench_config(res, world), 'impl_kernel': args.impl,
            'triangles': int(tris.shape[0]), 'vertices': int(verts.shape[0]),
            'meshes_per_s': 1.0 / (ms_per_step * 1e-3),
            'phases_ms_max_over_ranks': phase_max, 'limiting_phase': limiting,
            'sdf_ms': phase_max['sdf_ms'], 'gather_ms': phase_max['gather_ms'],
            'count_exchange_ms': phase_max['count_exchange_ms'],
            'nvlink_gather_bytes_per_step': gather_bytes,
            'identical_to_single_gpu': identical,
            'gpu_launches': per_step_launches * args.steps,
            'collectives_per_step': 'all_gather (2 int64 per rank) + one batched isend/irecv group (mesh buffers -> rank 0)',
            'clocks': clocks,
            'e2e': {'value': e2e_value, 'unit': 'points/s', 'h2d_bytes_per_step': int(h2d), 'd2h_bytes_per_step': int(d2h),
                    'api': 'extract_mesh_sharded (latent from pinned host memory, mesh to numpy on rank 0)'},
            'roofline': roofline_block(res, FLOP_PER_POINT * sdf_points_max, phase_max['sdf_ms'],
                                       note_extra=' of the slowest rank (%d planes incl. ghost/closing planes)' % max(planes)),
            'replicas': {'value': world * r_total_pts / (r_ms.item() * 1e-3), 'unit': 'points/s', 'ms_per_step': r_ms.item(),
                         'what': 'independent replicas: one 256^3 head (SDF + marching cubes) per rank, no collective (weak scaling)'},
        }
        print(json.dumps(line))


def main():
    args = parse()
    if args.impl == 'reference':
        run_reference_arm(args)
        return
    import torch
    import torch.distributed as dist

    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    os.environ['NPHM_B200_IMPL'] = args.impl
    if world > 1:
        dist.init_process_group('nccl', device_id=dev)
        try:
            run_sharded(args, torch, dist, dev, world, rank)
        finally:
            dist.destroy_process_group()
    else:
        run_single(args, torch, dev)


if __name__ == '__main__':
    main()
