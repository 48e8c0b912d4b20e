#!/usr/bin/env python
"""bench.py -- NanoWrap CG shrinkwrap hot path on B200 (contract: see DESIGN.md "Measurement").

    python bench.py --gpus N --steps K --warmup W [--impl reference] [--workload c3|c2|c1] [--dump-outputs DIR]

A *step* is one CG iteration of ``ShrinkwrapMeshConjGrad.search`` over the rank's whole point shard
(nearest-face rebuild included, as the reference rebuilds it every iteration; host remesh excluded,
SURVEY 8d).  Default workload = BASELINE.json configs[2], the one the north-star target is quoted on:
two-lobed necked shape, 10 M localisations per GPU, 501 762-vertex mesh (weak scaling: points per GPU
fixed, mesh replicated).  Iterations run in blocks of 5 (remesh_frequency) like the reference's driver;
each block starts from a fresh topology upload, so the nearest-face search starts cold once per block.

Prints ONE JSON line on rank 0.
"""
from __future__ import annotations

import argparse
import ctypes
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True     # the benchmark writes nothing into the tree it runs from (which may be read-only)

WORKLOADS = {
    # name: (points per GPU, geodesic frequency n -> 10 n^2 + 2 vertices, curvature_weight, block length)
    'c1': dict(points=10_000, geo=8, curvature_weight=20.0, block=10, desc='config0: ~10k localisations, 642-vertex mesh'),
    'c2': dict(points=1_000_000, geo=71, curvature_weight=10.0, block=5, desc='config1: 1M localisations, 50 412-vertex mesh'),
    'c3': dict(points=10_000_000, geo=224, curvature_weight=10.0, block=5, desc='config2: 10M localisations, 501 762-vertex two-lobed mesh'),
    'c4': dict(points=12_500_000, geo=316, curvature_weight=10.0, block=5, desc='config3: 100M localisations over 8 GPUs (12.5M per GPU), 998 562-vertex replicated mesh'),
    'c4s': dict(points=100_000_000, geo=316, curvature_weight=10.0, block=5, strong=True,
                desc='config3 as BASELINE states it: 100M localisations IN TOTAL sharded over the ranks (strong scaling), 998 562-vertex replicated mesh'),
    'c5': dict(points=2_000_000, geo=632, curvature_weight=50.0, block=5, desc='config4: curvature stress, 3 994 242-vertex mesh, sparse 2M-localisation cloud'),
}
CPU_SAMPLE = 'c2'         # bounded CPU sample of the cpu_baseline leg: same shape, same 20 localisations per vertex, 1/10 of c3
STAGES = ['refit', 'shift', 'sweep1', 'allreduce_acc', 'mesh_prior', 'sweep2', 'allreduce_scalars', 'solve_update', 'seed_leaders',
          'topology_build', 'adjoint']


def build_workload(name, seed, points=None, rank=0, world=1):
    """(mesh, points, sigma, cfg) of a BASELINE config; `points` overrides the number of localisations (parity tests draw a
    subset-sized cloud over the full-size mesh)."""
    from ch_shrinkwrap_b200 import minimesh, synth
    from ch_shrinkwrap_b200.membrane_mesh import MembraneMesh
    cfg = dict(WORKLOADS[name])
    cfg['rank'], cfg['world'] = rank, world
    if points is not None:
        cfg['points'] = int(points)
    shape = synth.two_lobed()
    v, f = minimesh.geodesic_sphere(cfg['geo'])
    v, f = minimesh.spatially_sorted(v, f)       # arbitrary generator order -> spatially coherent vertex / face order
    r = synth.radial_surface(shape, v, n_bisect=32)
    if cfg.get('strong'):
        # strong scaling: the SAME global cloud whatever the number of ranks -- 8 seeded chunks, rank r of N holds chunks
        # [8 r / N, 8 (r + 1) / N).  Every chunk covers the whole surface, so every rank sees the same mix of queries.
        rank, world = cfg.get('rank', 0), cfg.get('world', 1)
        assert 8 % world == 0, 'strong-scaling workload needs 1, 2, 4 or 8 ranks'
        per = cfg['points'] // 8
        parts = [synth.mesh_surface_cloud(v * r[:, None], f, per, seed=seed + 1000 * c) for c in range(8 * rank // world, 8 * (rank + 1) // world)]
        pts = np.concatenate([p for p, _ in parts]); sig = np.concatenate([q for _, q in parts])
        del parts
    else:
        pts, sig = synth.mesh_surface_cloud(v * r[:, None], f, cfg['points'], seed=seed)
    mesh = MembraneMesh(v * (1.2 * r)[:, None], f, kc=1.0, step_size=cfg['curvature_weight'],
                        remesh_frequency=cfg['block'], delaunay_remesh_frequency=0)
    return mesh, pts, sig, cfg


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = 'index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,' \
        'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap'

    def __init__(self, gpu_index):
        self.idx = gpu_index
        self.proc = None
        self.path = None

    def start(self):
        try:
            fd, self.path = tempfile.mkstemp(suffix='.csv')
            os.close(fd)
            self.proc = subprocess.Popen(['nvidia-smi', '-i', str(self.idx), '--query-gpu=' + self.Q, '--format=csv,noheader,nounits',
                                          '-lms', '100'], stdout=open(self.path, 'w'), stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        out = {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': [], 'samples': 0}
        if self.proc is None:
            return out
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        try:
            rows = [l.strip().split(', ') for l in open(self.path) if l.strip()]
            os.unlink(self.path)
            sm = [float(r[1]) for r in rows if len(r) >= 9]
            names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
            reasons = set()
            for r in rows:
                if len(r) >= 9:
                    for k, nme in enumerate(names):
                        if r[5 + k].strip().lower().startswith('active'):
                            reasons.add(nme)
            if sm:
                out.update(sm_mhz=float(np.median(sm)), sm_max_mhz=float(rows[0][2]), reasons=sorted(reasons), samples=len(sm))
        except Exception:
            pass
        return out


def run_blocks(mesh, pts, s_inv, lam, n_iters, block, handle_profile=True):
    """n_iters CG iterations in blocks: new solver object + topology upload per block (what
    MembraneMesh.opt_conjugate_gradient does, _membrane_mesh.pyx:1510-1517).  Returns
    (device ms inside nw_search summed over blocks, wall seconds of constructor+search, last solver object, blocks run)."""
    from ch_shrinkwrap_b200.mesh_conj_grad import ShrinkwrapMeshConjGrad
    dev_ms, wall, done, blocks = 0.0, 0.0, 0, 0
    sm = ctypes.c_double(0.0)
    cg = None
    while done < n_iters:
        n_it = min(block, n_iters - done)
        t0 = time.perf_counter()
        cg = ShrinkwrapMeshConjGrad(mesh, pts, device=getattr(mesh, '_nw_device', 0), comm=getattr(mesh, '_nw_comm', None))
        mesh.cg = cg
        cg.search(pts, lams=[lam], num_iters=n_it, sigma_inv=s_inv)
        wall += time.perf_counter() - t0
        cg._h.call('nw_get_profile', None, None, ctypes.byref(sm))
        dev_ms += sm.value
        done += cg.loopcount          # the stop rule may end a block early: count the iterations that ran
        blocks += 1
    return dev_ms, wall, cg, blocks


def cpu_reference_run(workload, steps, warmup, seed):
    """The reference's own CPU path on `workload`: the UNMODIFIED ``ShrinkwrapMeshConjGrad.search``
    (mesh_conj_grad.py:150-292: scipy cKDTree(workers=-1), numpy, the C scatter) imported through oracle/refharness.py from
    the build product oracle/_ref/ (kind "reference"); only if that is missing, the oracle's numpy/scipy restatement
    (kind "port").  One solver object, `warmup` untimed iterations, then `steps` timed ones.
    Returns dict(value, seconds, P, M, cores, kind, sample)."""
    from oracle import refharness
    mesh, pts, sig, cfg = build_workload(workload, seed)
    s_inv = (1.0 / sig.ravel()).astype(np.float32)
    lam = cfg['curvature_weight'] * 1.0 / 2.0
    if refharness.available():
        kind, how = 'reference', 'unmodified reference (%s)' % refharness.kind()
        oc = refharness.reference_solver(mesh, pts)
    else:
        from oracle import build as obuild
        from oracle import nanowrap_oracle as orc
        obuild.build_oracle_c()
        kind, how = 'port', 'oracle port (reference not staged under oracle/_ref/)'
        oc = orc.OracleConjGrad(mesh, pts)
        mesh.cg = oc
    if warmup > 0:
        oc.search(pts, lams=[lam], num_iters=warmup, sigma_inv=s_inv)
    t0 = time.perf_counter()
    oc.search(pts, lams=[lam], num_iters=steps, sigma_inv=s_inv)
    dt = time.perf_counter() - t0
    P = len(pts)
    return dict(value=P * steps / dt, seconds=dt, P=P, M=len(mesh._vertices), cores=os.cpu_count(), kind=kind,
                sample='%s: %d CG iterations after %d warm-up, %s' % (cfg['desc'], steps, warmup, how), mesh=mesh)


def cpu_curvature_run(mesh):
    """The reference's c_curvature_grad (membrane_mesh_utils.c:915-1250, compiled from the reference's own source into
    oracle/_ref/libref_curvature.so) on the whole mesh: vertices/s on one host core (the reference loop is serial)."""
    from oracle import refharness
    mesh.update_geometry()
    try:
        t0 = time.perf_counter()
        refharness.reference_curvature(mesh, kc=1.0, seed=1)
        dt = time.perf_counter() - t0
        kind = 'reference'
    except Exception:
        from oracle import build as obuild
        from oracle import nanowrap_oracle as orc
        obuild.build_oracle_c()
        t0 = time.perf_counter()
        orc.curvature_grad(mesh)
        dt = time.perf_counter() - t0
        kind = 'port'
    M = len(mesh._vertices)
    return {'value': M / dt, 'unit': 'vertices/s', 'seconds': dt, 'vertices': M, 'cores': 1, 'kind': kind}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=5)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--workload', default='c3', choices=sorted(WORKLOADS))
    ap.add_argument('--seed', type=int, default=1234)
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--random-shards', action='store_true', help='strong scaling: keep the random 1/N shards (no spatial-block exchange)')
    ap.add_argument('--cpu-steps', type=int, default=5, help='timed iterations of the cpu_baseline sample (our arm)')
    ap.add_argument('--ref-steps', type=int, default=0, help='reference arm: timed full-size iterations (default min(steps, 2))')
    ap.add_argument('--ref-warmup', type=int, default=-1, help='reference arm: untimed full-size iterations (default 0)')
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help='after the timed steps, write what the last timed search() call returned (vertices, float32 (M, 3)) '
                         'and its test statistic / residual norm histories (tests, ress, float64) as DIR/<name>.npy')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs and args.impl != 'ours':
        ap.error('--dump-outputs writes the outputs of --impl ours')
    rank = int(os.environ.get('RANK', '0'))
    local_rank = int(os.environ.get('LOCAL_RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    unit = 'localisation*iterations/s'
    metric = 'localisation_iterations_per_s'

    # ------------------------------------------------------------------ reference arm (CPU, rank 0 only)
    if args.impl == 'reference':
        if rank != 0:
            return
        # The SAME workload as our arm (default c3: 10 M localisations, 501 762 vertices).  One reference iteration at this
        # size takes minutes of host time, so the arm times a bounded number of full-size steps (default: the FIRST 2 iterations of the fit,
        # no warm-up -- our arm's window is the first K iterations from the same start mesh; --ref-steps / --ref-warmup) whatever --steps / --warmup ask for, and says so in the line.
        K = args.ref_steps if args.ref_steps > 0 else min(args.steps, 2)
        W = args.ref_warmup if args.ref_warmup >= 0 else 0
        r = cpu_reference_run(args.workload, K, W, args.seed)
        cfg = WORKLOADS[args.workload]
        curv = cpu_curvature_run(r['mesh'])
        line = {
            'impl': 'reference', 'metric': metric, 'value': r['value'], 'unit': unit, 'n_gpus': args.gpus, 'steps': K,
            'warmup': W, 'ms_per_step': 1e3 * r['seconds'] / K, 'higher_is_better': True, 'scaling': 'weak',
            'vs_baseline': None, 'dtype': 'f32 (fp64 nearest-face compare and Gram sums)', 'data': 'synthetic',
            'config': {'workload': cfg['desc'] + ' per GPU', 'points_timed': r['P'], 'vertices_timed': r['M'],
                       'same_config_as_gpu_arm': True, 'requested_steps': args.steps, 'requested_warmup': args.warmup,
                       'timed': 'full-size steps of the same workload; bounded to %d timed + %d warm-up iterations' % (K, W)},
            'cg_iters_per_s': K / r['seconds'],
            'cpu_baseline': {'value': r['value'], 'unit': unit, 'cores': r['cores'], 'kind': r['kind'], 'sample': r['sample'],
                             'curvature': curv},
            'e2e': {'value': r['value'], 'unit': unit, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
            'gpu_launches': 0,
        }
        print(json.dumps(line))
        return

    # ------------------------------------------------------------------ our arm
    from ch_shrinkwrap_b200 import _lib
    _lib.load()
    dist = None
    comm = None
    if world > 1:
        import torch
        import torch.distributed as dist
        torch.cuda.set_device(local_rank)
        dist.init_process_group('nccl', device_id=torch.device('cuda', local_rank))
        uid = ctypes.create_string_buffer(128)
        if rank == 0:
            rc = _lib.load().nw_comm_unique_id(uid)
            assert rc == 0, 'nw_comm_unique_id failed'
        t = torch.frombuffer(bytearray(uid.raw), dtype=torch.uint8).cuda()
        dist.broadcast(t, 0)
        comm = (rank, world, bytes(t.cpu().numpy().tobytes()))

    def barrier():
        if dist is not None:
            dist.barrier()

    def allmax(x):
        if dist is None:
            return x
        import torch
        t = torch.tensor([x], dtype=torch.float64, device='cuda')
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    strong = bool(WORKLOADS[args.workload].get('strong'))
    mesh, pts, sig, cfg = build_workload(args.workload, args.seed if strong else args.seed + 1000 * rank, rank=rank, world=world)
    if strong and world > 1 and not args.random_shards:
        # strong scaling: every rank generated a random 1/N of the cloud; hand every point to the rank that owns its spatial
        # block (interleaved cubes, ch_shrinkwrap_b200/sharding.py) so that each rank's points are dense where it has any --
        # a one-off ingest step, outside every timed region
        import torch
        from ch_shrinkwrap_b200 import sharding
        lo_t = torch.tensor(pts.min(0), device='cuda'); hi_t = torch.tensor(pts.max(0), device='cuda')
        dist.all_reduce(lo_t, op=dist.ReduceOp.MIN); dist.all_reduce(hi_t, op=dist.ReduceOp.MAX)
        ids, c = sharding.block_ids(pts, lo_t.cpu().numpy(), hi_t.cpu().numpy(), len(pts) * world)
        hist = torch.from_numpy(np.bincount(ids, minlength=c ** 3)).cuda()
        dist.all_reduce(hist)                                            # global points per cube
        table, load = sharding.balanced_owner_table(hist.cpu().numpy(), world)
        pts, sig = sharding.exchange_to_owners([pts, sig], table[ids], dist, torch.device('cuda', local_rank))
        torch.cuda.empty_cache()
    mesh._nw_device = local_rank
    mesh._nw_comm = comm
    s_inv = (1.0 / sig.ravel()).astype(np.float32)
    lam = cfg['curvature_weight'] * 1.0 / 2.0            # lam = curvature_weight * kc / 2 (_membrane_mesh.pyx:1486)
    P, M, F = len(pts), len(mesh._vertices), len(mesh.faces)
    block = cfg['block']
    W = max(args.warmup, 3)
    K = args.steps
    start_pos = mesh._vertices['position'].copy()

    # CUDA context + module load happen once per process, before any timing
    from ch_shrinkwrap_b200.mesh_conj_grad import _session_for
    _session_for(mesh, local_rank, comm)

    # ---- e2e: public API with HOST buffers: first block pays the point upload + Hilbert sort, every block the
    #      topology H2D and the position D2H.  Timed by wall clock around constructor + search().
    # warm-up (lazy module loading, first-touch allocations), then forget the uploaded points so that the timed run
    # pays the host->device copy and the Hilbert sort again
    run_blocks(mesh, pts, s_inv, lam, W, block)
    mesh._vertices['position'][:] = start_pos
    mesh.update_geometry()
    mesh._nw_session.points_key = None
    barrier()
    t0 = time.perf_counter()
    _, e2e_wall, cg, n_blocks = run_blocks(mesh, pts, s_inv, lam, K, block)
    e2e_s = allmax(time.perf_counter() - t0)
    h = cg._h
    topo_bytes = M * 12 * 2 + F * 12 + M * 80 + M
    e2e = {'value': P * world * K / e2e_s, 'unit': unit,
           'h2d_bytes_per_step': int((P * 24 + n_blocks * (topo_bytes + M * 12)) / K),
           'd2h_bytes_per_step': int(n_blocks * M * 12 / K),
           'note': 'ShrinkwrapMeshConjGrad(...).search() per block of %d iterations, host numpy in/out; includes the one-off upload '
                   'and Hilbert sort of the points (pageable host memory), per-block topology upload and position read-back' % block}

    # ---- device-resident: points already in HBM; warm-up then K timed iterations (CUDA events inside nw_search)
    mesh._vertices['position'][:] = start_pos
    mesh.update_geometry()
    run_blocks(mesh, pts, s_inv, lam, W, block)
    mesh._vertices['position'][:] = start_pos
    mesh.update_geometry()
    h.call('nw_reset_seeds')              # the timed run starts cold like a fit does: no faces / foot points left over from the warm-up
    h.call('nw_set_profile', 1)
    launches0 = h.lib.nw_launch_count(h.h)
    clocks = ClockSampler(local_rank)
    barrier()
    h.call('nw_sync')
    clocks.start()
    try:
        dev_ms, _, cg, _ = run_blocks(mesh, pts, s_inv, lam, K, block)
        h.call('nw_sync')
        barrier()
    finally:
        clk = clocks.stop()           # never leave the nvidia-smi sampler running
    if args.dump_outputs and rank == 0:
        # every rank ends with the same vertices; the histories are those of the last block's solver object
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, a in (('vertices', cg.fs), ('tests', np.array(cg.tests, np.float64)), ('ress', np.array(cg.ress, np.float64))):
            np.save(os.path.join(args.dump_outputs, name + '.npy'), a)
    launches = int(h.lib.nw_launch_count(h.h) - launches0)
    dev_ms = allmax(dev_ms)
    stage_ms = (ctypes.c_double * 16)()
    stage_l = (ctypes.c_int64 * 16)()
    h.call('nw_get_profile', stage_ms, stage_l, None)
    h.call('nw_set_profile', 0)
    # the timed region is every device-side piece of the K steps: the CG iterations (inside nw_search) AND the per-block
    # octree build of nw_set_topology (the reference rebuilds its cKDTree every iteration, mesh_conj_grad.py:445)
    dev_ms += allmax(stage_ms[9])
    value = P * world * K / (dev_ms * 1e-3)

    # ---- roofline of the dominant kernel, measured live over the timed region ----
    peaks_path = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(peaks_path):
        peak, peak_src = float(json.load(open(peaks_path))['hbm_gbs']), 'measured (MEASURED_PEAKS.json hbm_gbs)'
    else:
        peak, peak_src = 6650.0, 'fallback (B200_PROFILING.md)'
    alg_bytes = {
        'sweep1': 76.0 * P + 24.0 * F + 12.0 * M,          # NN + weights + residual in one kernel (SURVEY 8d)
        'sweep2': 36.0 * P + 12.0 * 3 * M,                 # multi-RHS Gram pass, n = 3
        'mesh_prior': 120.0 * M,                           # _ncc
        'apply_A': 36.0 * P + 12.0 * M,
        'apply_AH': 36.0 * P + 12.0 * M,
        'adjoint': 36.0 * P + 12.0 * M,                    # AH res + AH 1 in one pass (the scatter of the iteration)
    }
    stage = {STAGES[k]: {'ms_total': stage_ms[k], 'launches': int(stage_l[k])} for k in range(len(STAGES))}
    dom = max(('sweep1', 'sweep2', 'mesh_prior'), key=lambda k: stage[k]['ms_total'])
    dom_ms = stage[dom]['ms_total'] / K
    achieved = alg_bytes[dom] / (dom_ms * 1e-3) / 1e9
    tpath = os.path.join(ROOT, 'profiles', 'traffic.json')
    try:
        traffic_tab = json.load(open(tpath)).get(args.workload, {}) if os.path.exists(tpath) else {}
    except Exception:
        traffic_tab = {}

    def traffic_of(name):          # DRAM bytes per launch from the committed ncu captures (profiles/traffic.json), or None
        return traffic_tab.get(name)
    traffic = traffic_of(dom)
    roofline = {'bound': 'hbm', 'kernel': dom, 'achieved': achieved, 'peak': peak, 'unit': 'GB/s', 'frac': achieved / peak,
                'traffic': traffic, 'peak_source': peak_src, 'frac_of_nominal_8000_gbs': achieved / 8000.0, 'ms_per_launch': dom_ms, 'algorithmic_bytes_per_launch': alg_bytes[dom],
                'share_of_step': stage[dom]['ms_total'] / dev_ms}
    # isolated single-operator kernels (device resident, CUDA events)
    kernels = {}
    ms = ctypes.c_float(0.0)
    for name in ('apply_A', 'apply_AH', 'adjoint', 'sweep2', 'mesh_prior', 'sweep1'):
        try:
            h.call('nw_bench_kernel', name.encode(), 10, ctypes.byref(ms))
            gbs = alg_bytes[name] / (ms.value * 1e-3) / 1e9
            kernels[name] = {'ms': ms.value, 'achieved_gbs': gbs, 'frac': gbs / peak, 'traffic': traffic_of(name)}
        except Exception as e:      # noqa
            kernels[name] = {'error': str(e)}

    # curvature: once through the C ABI with host buffers (what remove_necks / the recipe's final step call), then the
    # kernel alone on the device-resident copies
    alg_bytes['curvature'] = 184.0 * M
    try:
        from ch_shrinkwrap_b200.membrane_mesh import curvature_grad
        mesh.update_geometry()
        t0 = time.perf_counter()
        cout = curvature_grad(mesh, kc=1.0)
        curv_first = time.perf_counter() - t0         # first call on this handle: allocates the device copies and the pinned staging
        t0 = time.perf_counter()
        curvature_grad(mesh, kc=1.0, out=cout)        # what remove_necks pays once per remesh block (_membrane_mesh.pyx:1212)
        curv_wall = time.perf_counter() - t0
        h.call('nw_bench_kernel', b'curvature', 10, ctypes.byref(ms))
        gbs = alg_bytes['curvature'] / (ms.value * 1e-3) / 1e9
        fp64_ms = traffic_of('curvature_fp64_pipe_busy_ms')
        kernels['curvature'] = {'ms': ms.value, 'achieved_gbs': gbs, 'frac': gbs / peak, 'traffic': traffic_of('curvature'),
                                # against the fp64 pipe instead of HBM: the time that pipe is busy for this arithmetic (ncu) / the kernel's time
                                'fp64_bound': None if not fp64_ms else {'bound': 'fp64', 'pipe_busy_ms': fp64_ms, 'frac': fp64_ms / ms.value},
                                'c_abi_call_ms_host_buffers': 1e3 * curv_wall, 'c_abi_first_call_ms': 1e3 * curv_first,
                                'vertices_per_s': M / (ms.value * 1e-3)}
    except Exception as e:      # noqa
        kernels['curvature'] = {'error': str(e)}
    # every rank holds the whole mesh and must end the timed run with the very same vertices: the adjoint accumulates in
    # integers (order-free) and the mesh-side kernels are replicated, so anything but bit identity is a bug
    ranks_identical = None
    if dist is not None:
        import zlib
        import torch
        crc = zlib.crc32(np.ascontiguousarray(mesh._vertices['position']).tobytes())
        t = torch.tensor([crc], dtype=torch.int64, device='cuda')
        allc = [torch.zeros_like(t) for _ in range(world)]
        dist.all_gather(allc, t)
        ranks_identical = bool(all(int(c.item()) == crc for c in allc))
        # how evenly the sweep is spread: every rank's own total of the two per-point stages over the timed window
        ts = torch.tensor([stage_ms[2] + stage_ms[10], stage_ms[5]], dtype=torch.float64, device='cuda')
        allt = [torch.zeros_like(ts) for _ in range(world)]
        dist.all_gather(allt, ts)
        sweep_by_rank = [round(float(t[0].item()) / K, 4) for t in allt]
        sweep2_by_rank = [round(float(t[1].item()) / K, 4) for t in allt]
        dist.barrier()
        dist.destroy_process_group()
    if rank != 0:
        return
    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        # bounded sample (config 1 is the same shape at 1/10 the size); the full-size CPU number is the reference arm's
        r = cpu_reference_run(CPU_SAMPLE if args.workload in ('c3', 'c4', 'c5') else args.workload, args.cpu_steps, 1, args.seed)
        cpu = {'value': r['value'], 'unit': unit, 'cores': r['cores'], 'kind': r['kind'], 'sample': r['sample'],
               'cg_iters_per_s_on_sample': args.cpu_steps / r['seconds'],
               'curvature': cpu_curvature_run(mesh)}      # the bench mesh itself (full size), one host core
    line = {
        'metric': metric, 'value': value, 'unit': unit, 'n_gpus': world, 'steps': K, 'warmup': W, 'ms_per_step': dev_ms / K,
        'higher_is_better': True, 'scaling': 'strong' if strong else 'weak', 'vs_baseline': None,
        'dtype': 'f32 (fp64 nearest-face compare and Gram sums, int64 fixed-point adjoint)', 'data': 'synthetic',
        'config': {'workload': cfg['desc'] + ('' if strong else ' per GPU'), 'points_per_gpu': P, 'points_total': P * world, 'vertices': M, 'faces': F, 'lam': lam,
                   'block_iterations': block, 'parallelism': 'points sharded x%d%s, mesh replicated' % (world, ' (interleaved spatial blocks)' if (strong and world > 1 and not args.random_shards) else ''),
                   'l2': 'inputs larger than L2: per-point streams %.0f MB vs 126 MB L2' % (52.0 * P / 1e6)},
        'cg_iters_per_s': K / (dev_ms * 1e-3),
        'e2e': e2e, 'gpu_launches': launches, 'clocks': {k: clk[k] for k in ('sm_mhz', 'sm_max_mhz', 'reasons')},
        'roofline': roofline, 'cpu_baseline': cpu, 'stages': stage, 'kernels': kernels,
    }
    if ranks_identical is not None:
        line['ranks_bit_identical'] = ranks_identical
        line['per_rank_ms_per_step'] = {'sweep1_plus_adjoint': sweep_by_rank, 'sweep2': sweep2_by_rank}
    print(json.dumps(line))


if __name__ == '__main__':
    main()
