"""bench.py -- particle-pair interactions/s on the 3D WCSPH dam break.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--dump-outputs DIR]
    python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...
    python bench.py --impl reference ...      # the CPU arm (oracle, all threads)

One "step" = one EPEC time step of pysph/examples/dam_break_3d.py with
--kernel CubicSpline: 2 x (cell-list build + EOS + fused pair kernel) + the
WCSPHStep stages + the adaptive-dt reduction.  N = 1 runs BASELINE.json
configs[1] (dx = 0.00877: ~1.0 M fluid + ~0.23 M wall/obstacle particles);
N > 1 keeps ~1.2 M particles per GPU (dx = 0.00877 / N^(1/3); N = 8 is
configs[2], ~10 M) with x-slabs and a NCCL halo exchange before every
evaluation.  Prints ONE JSON line (rank 0).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

BASE_DX = 0.00877
C3_DX = 0.00407         # BASELINE configs[2] as quoted: ~11.3 M particles
BYTES_PER_PAIR = 45.0   # SURVEY.md 8(d): 44 B gathered source state + ~1.1 B dest I/O
METRIC = 'particle_pair_interactions_per_s'


def dam_break_dx(args, world):
    """weak scaling (default): ~1.2 M particles per GPU; strong: BASELINE configs[2]'s
    10 M-particle case (dx = 0.00407) on however many GPUs there are"""
    if args.dx:
        return args.dx
    if args.scaling == 'strong':
        return C3_DX
    return BASE_DX / world ** (1.0 / 3.0)


def dam_break_workload(dx, world):
    """ONE string for both arms (the driver compares them)."""
    cfg = 2 if (world > 1 or abs(dx - C3_DX) < 1e-9) else 1
    return 'dam_break_3d (BASELINE configs[%d]) EPEC CubicSpline dx=%.6f hdx=1.3' % (cfg, dx)


def peaks():
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d['hbm_gbs']), 'measured (MEASURED_PEAKS.json hbm_gbs)'
    return 6650.0, 'fallback (B200_PROFILING.md 6.65 TB/s)'


class ClockSampler(object):
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ('clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,'
         'clocks_event_reasons.hw_thermal_slowdown,'
         'clocks_event_reasons.sw_thermal_slowdown,'
         'clocks_event_reasons.sw_power_cap')

    def __init__(self, index=0):
        self.lines = []
        self.proc = None
        self.index = index

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ['nvidia-smi', '-i', str(self.index), '--query-gpu=' + self.Q,
                 '--format=csv,noheader,nounits', '-lms', '200'],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
            # its start-up (NVML initialises every GPU of the box) stalls running kernels for
            # tens of ms: nothing is timed before the first line has arrived
            t0 = time.time()
            while not self.lines and time.time() - t0 < 15.0 and self.proc.poll() is None:
                time.sleep(0.01)
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self, first=0):
        """first: number of lines printed before the timed region began; the line
        in flight then (index first - 1) is kept when the region was shorter than
        one sampling period."""
        if self.proc is None:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['unavailable']}
        time.sleep(0.21)                     # let the sample covering the region's end arrive
        if len(self.lines) > first:
            self.lines = self.lines[first:]
        else:
            self.lines = self.lines[-1:]
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown',
                 'sw_power_cap']
        for ln in self.lines:
            f = [x.strip() for x in ln.split(',')]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
            except ValueError:
                continue
            for n, v in zip(names, f[3:7]):
                if v.lower().startswith('active'):
                    reasons.add(n)
        return {'sm_mhz': float(np.median(sm)) if sm else None,
                'sm_max_mhz': float(np.max(mx)) if mx else None,
                'samples': len(sm), 'reasons': sorted(reasons)}


def copy_arrays(pas):
    import pysph_b200 as pb
    out = []
    for pa in pas:
        q = pb.get_particle_array_wcsph(
            name=pa.name, **dict((k, v.copy()) for k, v in pa.properties.items()))
        q.set_num_real_particles(pa.num_real_particles)
        out.append(q)
    return out


def cpu_leg(pas, params, threads, budget_s, max_steps, warmup=0):
    """Time the fp64 oracle (the CPU restatement of the reference path) on the
    same workload: EPEC steps until the budget is used.  Returns a dict."""
    from oracle import oracle as orc
    s = orc.WCSPHOracleSolver(pas, params, 'CubicSpline', threads=threads)
    s.initialise()
    for _ in range(warmup):
        s.step()
    s.pairs_total = 0
    t0 = time.perf_counter()
    n = 0
    while n < max_steps:
        s.step()
        n += 1
        if time.perf_counter() - t0 > budget_s:
            break
    el = time.perf_counter() - t0
    return dict(pairs_per_s=s.pairs_total / el, steps=n, seconds=el,
                pairs_per_step=s.pairs_total / n)


def cpu_model():
    try:
        for ln in open('/proc/cpuinfo'):
            if ln.startswith('model name'):
                return ln.split(':', 1)[1].strip()
    except Exception:
        pass
    return 'unknown'


def _oracle_steps(solver, budget_s, max_steps, warmup):
    """EPEC / PEC steps of an oracle solver until the budget is used; pairs counted per
    evaluation through pairs_last_eval (one evaluate() call = every group once)."""
    total = [0]
    orig = solver.evaluate

    def counting(*a, **kw):
        r = orig(*a, **kw)
        total[0] += solver.pairs_last_eval
        return r
    solver.evaluate = counting
    solver.initialise()
    for _ in range(warmup):
        solver.step()
    total[0] = 0
    t0 = time.perf_counter()
    n = 0
    while n < max_steps:
        solver.step()
        n += 1
        if time.perf_counter() - t0 > budget_s:
            break
    el = time.perf_counter() - t0
    return dict(pairs_per_s=total[0] / el, steps=n, seconds=el, pairs_per_step=total[0] / n)


def run_reference(args, rank, world):
    """--impl reference: the CPU arm.  /root/reference cannot be built without
    cyarray/compyle/mako (DESIGN.md), so this times the oracle port with all
    host threads on the same config; rank 0 only."""
    if rank != 0:
        return
    from pysph_b200 import geometry as geo
    from oracle import oracle as orc
    ncores = os.cpu_count() or 1
    # torchrun exports OMP_NUM_THREADS=1: size the pool from the affinity mask instead
    try:
        ncores = len(os.sched_getaffinity(0))
    except Exception:
        pass
    threads = max(1, min(ncores, 64))
    budget = args.cpu_budget if args.cpu_budget != 20.0 else 150.0
    # the same W as the GPU arm reports (max(W, 3)); CPU steps cost ~0.5 s each here, so the
    # warm-up is capped where it would eat the budget
    ref_warmup = min(max(args.warmup, 3), 10)
    if args.workload == 'rings':
        dx = args.dx or 0.00028
        lz = args.lz * world
        dt = args.dt or 1e-8 * dx / 0.0005
        pas = [geo.rings_3d_particles(dx=dx, lz=lz)]
        o = orc.ElasticOracleSolver(pas, dict(dim=3, dt=dt, eps=0.3, alpha=1.0, beta=1.0,
                                              eps_xsph=0.5, grad3d=True),
                                    'CubicSpline', threads=threads)
        r = _oracle_steps(o, budget, max(1, args.steps), ref_warmup)
        workload = 'rings 3-D (BASELINE configs[4]) elastic dynamics EPEC CubicSpline ' \
                   'hdx=1.5 dx=%g lz=%g' % (dx, lz)
        what = 'full EPEC steps (two evaluations of both elastic-dynamics groups)'
    elif args.workload == 'taylor_green':
        p = geo.taylor_green_params(args.nx, dim=3)
        pas = [geo.taylor_green_particles(args.nx, dim=3)]
        o = orc.EDACOracleSolver(pas, p, 'QuinticSpline', threads=threads,
                                 domain=([0, 0, 0], [1, 1, 1], [1, 1, 1]))
        r = _oracle_steps(o, budget, max(1, args.steps), ref_warmup)
        workload = 'taylor_green 3-D (BASELINE configs[3]) EDAC/TVF PEC QuinticSpline ' \
                   'nx=%d hdx=1.0 periodic' % args.nx
        what = 'full PEC steps (one evaluation of both EDAC groups, materialised periodic ghosts)'
    else:
        dx = dam_break_dx(args, world)
        pas = geo.dam_break_3d_particles(dx=dx)
        params = geo.dam_break_3d_params(dx)
        r = cpu_leg(pas, params, threads, budget_s=budget,
                    max_steps=max(1, args.steps), warmup=ref_warmup)
        workload = dam_break_workload(dx, world)
        what = 'full EPEC steps'
    ntot = sum(pa.get_number_of_particles(real=True) for pa in pas)
    ms = 1e3 * r['seconds'] / r['steps']
    line = {
        'impl': 'reference', 'metric': METRIC, 'value': r['pairs_per_s'],
        'unit': 'pairs/s', 'n_gpus': world, 'steps': r['steps'],
        'warmup': max(args.warmup, 3), 'cpu_warmup_steps': ref_warmup, 'ms_per_step': ms,
        'steps_per_s': 1e3 / ms, 'higher_is_better': True, 'scaling': args.scaling,
        'vs_baseline': None, 'dtype': 'f64', 'data': 'synthetic',
        'config': {'workload': workload,
                   'particles': ntot, 'pairs_per_step': r['pairs_per_step']},
        'cpu_baseline': {'value': r['pairs_per_s'], 'unit': 'pairs/s',
                         'cores': threads, 'kind': 'port',
                         'cpu': cpu_model(),
                         'sample': '%d %s of the same %d-particle '
                                   'state (time budget %.0f s)' % (r['steps'], what, ntot,
                                                                   budget)},
        'e2e': {'value': r['pairs_per_s'], 'unit': 'pairs/s',
                'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
    }
    print(json.dumps(line))


def run_taylor_green(args, emit):
    """--workload taylor_green: BASELINE configs[3] -- 3-D Taylor-Green vortex, EDAC
    scheme (transport-velocity branch), QuinticSpline, 126^3 = 2.0 M particles in the
    periodic unit cube, PEC + EDACTVFStep at the example's fixed dt, one B200.  Same
    JSON line as the default workload; one step = one evaluation = two pair passes."""
    import torch
    import pysph_b200 as pb
    from pysph_b200 import geometry as geo
    torch.cuda.set_device(0)
    nx = args.nx
    p = geo.taylor_green_params(nx, dim=3)
    pa = geo.taylor_green_particles(nx, dim=3)
    host_copy = None
    if not args.no_cpu:
        host_copy = pb.get_particle_array_edac(
            name='fluid', **dict((k, v.copy()) for k, v in pa.properties.items()))
    keep = pinned_arrays([pa])
    dm = pb.DomainManager(xmin=0, xmax=1, ymin=0, ymax=1, zmin=0, zmax=1,
                          periodic_in_x=True, periodic_in_y=True, periodic_in_z=True)
    sch = pb.EDACScheme(['fluid'], [], dim=3, c0=p['c0'], nu=p['nu'], rho0=p['rho0'],
                        pb=p['pb'], h=p['h'])
    solver = pb.make_edac_solver([pa], sch, pb.QuinticSpline(dim=3), dt=p['dt'], domain=dm)
    be = solver.backend
    stream = torch.cuda.current_stream()
    be.use_torch_stream(stream)
    W, K = max(args.warmup, 3), args.steps
    sampler = ClockSampler(0)
    sampler.start()
    solver.initialise()
    for _ in range(W):
        solver.step()
    solver.a_eval.count_pairs = True
    solver.step()
    pairs_step = solver.a_eval.last_pairs          # both passes
    solver.a_eval.count_pairs = False
    be.ctx.call('b200sph_reset_stats')
    be.ctx.call('b200sph_set_profiling', 2)
    torch.cuda.synchronize()
    n_s0 = len(sampler.lines)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record(stream)
    for _ in range(K):
        solver.step()
    ev1.record(stream)
    torch.cuda.synchronize()
    clocks = sampler.stop(n_s0)
    ms_step = ev0.elapsed_time(ev1) / K
    st = be.stats()
    DIAG = 20
    be.ctx.call('b200sph_reset_stats')
    be.ctx.call('b200sph_set_profiling', 1)
    for _ in range(DIAG):
        solver.step()
    torch.cuda.synchronize()
    st_diag = be.stats()
    be.ctx.call('b200sph_set_profiling', 0)
    # e2e: host state in, result out, every step
    state = ['x', 'y', 'z', 'u', 'v', 'w', 'p', 'h', 'm']
    outp = ['x', 'y', 'z', 'u', 'v', 'w', 'rho', 'p']
    n = pa.get_number_of_particles()
    be.ctx.call('b200sph_set_async_copies', 1)

    def e2e_step():
        be.push_real(state)
        solver.step()
        be.pull_real(outp)
        be.synchronize()
    for _ in range(2):
        e2e_step()
    torch.cuda.synchronize()
    ev0.record(stream)
    for _ in range(args.e2e_steps):
        e2e_step()
    ev1.record(stream)
    torch.cuda.synchronize()
    be.ctx.call('b200sph_set_async_copies', 0)
    ms_e2e = ev0.elapsed_time(ev1) / args.e2e_steps
    peak, peak_src = peaks()
    ms_p2 = st['ms_pair'] / max(st['pair_launches'], 1)
    pairs_p2 = pairs_step / 2.0
    B2 = 64.0        # group 2 gathers {A,B} 32 B + C2 16 B + Dv 16 B per pair
    achieved = pairs_p2 * B2 / (ms_p2 * 1e-3) / 1e9
    cpu = None
    if host_copy is not None:
        from oracle import oracle as orc
        o = orc.EDACOracleSolver([host_copy], p, 'QuinticSpline', threads=1,
                                 domain=([0, 0, 0], [1, 1, 1], [1, 1, 1]))
        t0 = time.perf_counter()
        pairs_cpu = o.evaluate()
        el = time.perf_counter() - t0
        cpu = {'value': pairs_cpu / el, 'unit': 'pairs/s', 'cores': 1, 'kind': 'port',
               'cpu': cpu_model(),
               'sample': 'one full evaluation (both EDAC groups) of the same %d-particle '
                         'state with materialised periodic ghosts, fp64 oracle, 1 thread '
                         '(%.1f s)' % (n, el)}
    emit({
        'metric': METRIC, 'value': pairs_step / (ms_step * 1e-3), 'unit': 'pairs/s',
        'n_gpus': 1, 'steps': K, 'warmup': W, 'ms_per_step': ms_step,
        'steps_per_s': 1e3 / ms_step, 'higher_is_better': True, 'scaling': 'weak',
        'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
        'config': {'workload': 'taylor_green 3-D (BASELINE configs[3]) EDAC/TVF PEC '
                               'QuinticSpline nx=%d hdx=1.0 periodic' % nx,
                   'particles_rank0': n, 'pairs_per_step': pairs_step,
                   'parallelism': 'single GPU', 'dt': p['dt'],
                   'l2': 'no flush: > 126 MB working set per step, state advances',
                   'precision': 'fp32 pair arithmetic on cell-relative coordinates, '
                                'fp64 integrated state (x u p uhat)'},
        'clocks': clocks,
        'e2e': {'value': pairs_step / (ms_e2e * 1e-3), 'unit': 'pairs/s',
                'ms_per_step': ms_e2e, 'steps': args.e2e_steps,
                'h2d_bytes_per_step': 8 * len(state) * n,
                'd2h_bytes_per_step': 8 * len(outp) * n},
        'gpu_launches': int(st['kernel_launches']),
        'roofline': {'bound': 'hbm', 'kernel': 'k_tvf_pass2<QuinticSpline,3>',
                     'achieved': achieved, 'peak': peak, 'unit': 'GB/s',
                     'frac': achieved / peak, 'traffic': None, 'peak_source': peak_src,
                     'algorithmic_bytes_per_pair': B2, 'pairs_per_launch': pairs_p2,
                     'avg_launch_ms': ms_p2,
                     'share_of_step': st['ms_pair'] / K / ms_step,
                     'ms_nnps_per_step': st_diag['ms_nnps'] / DIAG,
                     'ms_other_per_step': st_diag['ms_other'] / DIAG,
                     'note': 'other = k_pack_tvf + k_tvf_pass1 + stages',
                     'nnps': {'full_builds': st['full_builds'],
                              'light_updates': st['light_updates'],
                              'list_builds': st['list_builds'],
                              'list_entries_per_particle': st['list_entries_per_particle']}},
        'cpu_baseline': cpu,
    })


def run_rings(args, emit, rank=0, local_rank=0, world=1):
    """--workload rings: BASELINE configs[4] -- 3-D elastic dynamics (Gray, Monaghan &
    Swift), the colliding rings of rings.py extruded along z, CubicSpline hdx=1.5,
    EPEC + SolidMechStep at a fixed dt.  dx = 0.00028; lz = 0.005 per GPU (1.0 M particles
    per GPU, 4 GPUs = the 4 M case: weak scaling along z, x-slabs with a two-support halo
    that carries the deviatoric stress).  One step = two evaluations = four pair passes
    (velocity gradient; continuity + momentum with stress + AV + XSPH)."""
    import torch
    import torch.distributed as dist
    import pysph_b200 as pb
    from pysph_b200 import geometry as geo
    torch.cuda.set_device(local_rank)
    dx = args.dx or 0.00028
    lz = args.lz * world
    dt = args.dt or 1e-8 * dx / 0.0005      # rings.py:36 (dt = 1e-8 at dx = 0.0005), same dt / h
    host_copy = None
    if world == 1:
        pa = geo.rings_3d_particles(dx=dx, lz=lz)
        if not args.no_cpu:
            host_copy = geo.rings_3d_particles(dx=dx, lz=lz)
        keep = pinned_arrays([pa])
        sch = pb.ElasticSolidsScheme(['solid'], [], dim=3)
        solver = pb.make_elastic_solver([pa], sch, pb.CubicSpline(dim=3), dt=dt,
                                        device=local_rank)
        pm = None
    else:
        from pysph_b200.parallel import make_rings_slab_solver
        solver, pm, pas = make_rings_slab_solver(dx, lz, rank, world, device=local_rank, dt=dt)
        pa = pas[0]
    be = solver.backend
    stream = torch.cuda.current_stream()
    be.use_torch_stream(stream)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def reduce(v, op):
        if world == 1:
            return v
        t = torch.tensor([float(v)], dtype=torch.float64, device='cuda')
        dist.all_reduce(t, op=op)
        return float(t.item())
    W, K = max(args.warmup, 3), args.steps
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    solver.initialise()
    for _ in range(W):
        solver.step()
    solver.a_eval.count_pairs = True
    solver.step()
    pairs_eval = solver.a_eval.last_pairs          # both passes of the step's last evaluation
    solver.a_eval.count_pairs = False
    pairs_step = int(reduce(2 * pairs_eval, dist.ReduceOp.SUM))   # EPEC: two evaluations per step
    be.ctx.call('b200sph_reset_stats')
    be.ctx.call('b200sph_set_profiling', 2)
    barrier()
    n_s0 = len(sampler.lines)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record(stream)
    for _ in range(K):
        solver.step()
    ev1.record(stream)
    barrier()
    clocks = sampler.stop(n_s0) if rank == 0 else None
    ms_step = reduce(ev0.elapsed_time(ev1), dist.ReduceOp.MAX) / K
    st = be.stats()
    DIAG = 20
    be.ctx.call('b200sph_reset_stats')
    be.ctx.call('b200sph_set_profiling', 1)
    for _ in range(DIAG):
        solver.step()
    torch.cuda.synchronize()
    st_diag = be.stats()
    be.ctx.call('b200sph_set_profiling', 0)
    state = ['x', 'y', 'z', 'u', 'v', 'w', 'rho', 'h', 'm',
             's00', 's01', 's02', 's11', 's12', 's22']
    outp = ['x', 'y', 'z', 'u', 'v', 'w', 'rho', 'p']
    if world > 1:
        # host mirrors hold this rank's real particles (migration may have changed the
        # count): refresh them once, then pin
        solver.pull()
        nr = pa.get_number_of_particles(real=True)
        for k in list(pa.properties):
            pa.properties[k] = pa.properties[k][:nr].copy()
        pa._n = nr
        keep = pinned_arrays([pa])
    n = be.sizes(0)[1]
    n_total = int(reduce(n, dist.ReduceOp.SUM))
    be.ctx.call('b200sph_set_async_copies', 1)

    def e2e_step():
        be.push_real(state)
        solver.step()
        be.pull_real(outp)
        be.synchronize()
    for _ in range(2):
        e2e_step()
    barrier()
    ev0.record(stream)
    for _ in range(args.e2e_steps):
        e2e_step()
    ev1.record(stream)
    barrier()
    be.ctx.call('b200sph_set_async_copies', 0)
    ms_e2e = reduce(ev0.elapsed_time(ev1), dist.ReduceOp.MAX) / args.e2e_steps
    peak, peak_src = peaks()
    ms_p2 = st['ms_pair'] / max(st['pair_launches'], 1)
    pairs_p2 = pairs_eval / 2.0
    B2 = 96.0        # pass 2 gathers {A,B} 32 B + C 16 B + stress records 48 B per pair
    achieved = pairs_p2 * B2 / (ms_p2 * 1e-3) / 1e9
    cpu = None
    if host_copy is not None:
        from oracle import oracle as orc
        o = orc.ElasticOracleSolver([host_copy], dict(dim=3, dt=dt, eps=0.3, alpha=1.0,
                                                      beta=1.0, eps_xsph=0.5, grad3d=True),
                                    'CubicSpline', threads=1)
        t0 = time.perf_counter()
        pairs_cpu = o.evaluate()
        el = time.perf_counter() - t0
        cpu = {'value': pairs_cpu / el, 'unit': 'pairs/s', 'cores': 1, 'kind': 'port',
               'cpu': cpu_model(),
               'sample': 'one full evaluation (both elastic-dynamics groups) of the same '
                         '%d-particle initial state, fp64 oracle, 1 thread (%.1f s)' % (n, el)}
    if rank != 0:
        return
    emit({
        'metric': METRIC, 'value': pairs_step / (ms_step * 1e-3), 'unit': 'pairs/s',
        'n_gpus': world, 'steps': K, 'warmup': W, 'ms_per_step': ms_step,
        'steps_per_s': 1e3 / ms_step, 'higher_is_better': True, 'scaling': 'weak',
        'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
        'config': {'workload': 'rings 3-D (BASELINE configs[4]) elastic dynamics EPEC '
                               'CubicSpline hdx=1.5 dx=%g lz=%g' % (dx, lz),
                   'particles': n_total, 'particles_rank0': n, 'pairs_per_step': pairs_step,
                   'parallelism': 'single GPU' if world == 1 else
                                  'x-slabs x%d, two-support halo (16 fields), peer-memory '
                                  'refresh' % world,
                   'dt': dt,
                   'l2': 'no flush: > 126 MB working set per step, state advances',
                   'precision': 'fp32 pair arithmetic on cell-relative coordinates, '
                                'fp64 integrated state (x u rho s)'},
        'clocks': clocks,
        'e2e': {'value': pairs_step / (ms_e2e * 1e-3), 'unit': 'pairs/s',
                'ms_per_step': ms_e2e, 'steps': args.e2e_steps,
                'h2d_bytes_per_step': 8 * len(state) * n_total,
                'd2h_bytes_per_step': 8 * len(outp) * n_total},
        'gpu_launches': int(st['kernel_launches']),
        'roofline': {'bound': 'hbm', 'kernel': 'k_solid_pass2<CubicSpline,3>',
                     'achieved': achieved, 'peak': peak, 'unit': 'GB/s',
                     'frac': achieved / peak, 'traffic': None, 'peak_source': peak_src,
                     'algorithmic_bytes_per_pair': B2, 'pairs_per_launch': pairs_p2,
                     'avg_launch_ms': ms_p2,
                     'share_of_step': st['ms_pair'] / K / ms_step,
                     'ms_nnps_per_step': st_diag['ms_nnps'] / DIAG,
                     'ms_other_per_step': st_diag['ms_other'] / DIAG,
                     'note': 'rank 0; other = k_pack_solid + k_solid_pass1 + stages',
                     'nnps': {'full_builds': st['full_builds'],
                              'light_updates': st['light_updates'],
                              'list_builds': st['list_builds'],
                              'list_entries_per_particle': st['list_entries_per_particle']}},
        'cpu_baseline': cpu,
        'halo': None if pm is None else {'full_updates': pm.n_full, 'refreshes': pm.n_refresh,
                                         'peer_refreshes': pm.n_peer_refresh},
    })


DUMP_FIELDS = ('x', 'y', 'z', 'u', 'v', 'w', 'rho', 'p', 'arho', 'au', 'av', 'aw')
DUMP_SAMPLE = 131072     # particles per array: 3 arrays x 13 fp64 columns stay under 64 MB


def dump_outputs(be, out_dir):
    """--dump-outputs: what a caller of the timed steps receives after the last of them --
    every array's real particles, pulled from the device, as DIR/<array>_<field>.npy
    (float64) with DIR/<array>_gid.npy naming the particles.  Rows are in gid order, so the
    files do not depend on how the device orders particles; an array of more than
    DUMP_SAMPLE particles is sampled at fixed, seeded positions of that order.  The host
    mirrors are left as they are (the e2e loop pushes them)."""
    from pysph_b200 import _lib
    os.makedirs(out_dir, exist_ok=True)
    for i, pa in enumerate(be.particle_arrays):
        n = be.sizes(i)[1]
        gid = np.empty(n, dtype=np.uint32)
        be.ctx.call('b200sph_pull_u32', i, _lib.INT_PROP_IDS['gid'], gid.ctypes.data, 0, n)
        rows = np.argsort(gid, kind='stable')
        if n > DUMP_SAMPLE:
            rows = rows[np.sort(np.random.RandomState(i).choice(n, DUMP_SAMPLE, replace=False))]
        np.save(os.path.join(out_dir, '%s_gid.npy' % pa.name), gid[rows].astype(np.float64))
        for f in DUMP_FIELDS:
            col = np.empty(n, dtype=np.float64)
            be.ctx.call('b200sph_pull_f64', i, be.prop_ids[i][f], col.ctypes.data, 0, n)
            np.save(os.path.join(out_dir, '%s_%s.npy' % (pa.name, f)), col[rows])


def pinned_arrays(pas):
    """Re-home every property of the ParticleArrays in pinned host memory."""
    import torch
    keep = []
    for pa in pas:
        for k, a in list(pa.properties.items()):
            t = torch.from_numpy(a.copy()).pin_memory()
            keep.append(t)
            pa.properties[k] = t.numpy()
    return keep


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=100)
    ap.add_argument('--warmup', type=int, default=50)
    ap.add_argument('--impl', default='b200')
    ap.add_argument('--dx', type=float, default=None)
    ap.add_argument('--e2e-steps', type=int, default=10)
    ap.add_argument('--cpu-budget', type=float, default=20.0)
    ap.add_argument('--no-cpu', action='store_true')
    ap.add_argument('--workload', default='dam_break',
                    choices=['dam_break', 'taylor_green', 'rings'])
    ap.add_argument('--nx', type=int, default=126)
    ap.add_argument('--lz', type=float, default=0.005)
    ap.add_argument('--dt', type=float, default=None)
    ap.add_argument('--scaling', default='weak', choices=['weak', 'strong'],
                    help='weak: ~1.2 M particles per GPU (default); strong: the 10 M-particle '
                         'case of BASELINE configs[2] (dx = 0.00407) on N GPUs')
    ap.add_argument('--no-parity', action='store_true',
                    help='N > 1: skip the N-rank == 1-process check that precedes the timed region')
    ap.add_argument('--no-developed', action='store_true',
                    help='skip the second timed region (developed flow: list rebuilds inside)')
    ap.add_argument('--no-extras', action='store_true',
                    help='skip the sub-records of BASELINE configs[3] / [4] (and configs[2] as '
                         'quoted at N = 8) appended to the dam-break line')
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help='single-GPU dam break: after the timed steps, write the particle fields '
                         'of their last step to DIR/<array>_<field>.npy (float64, gid order, at '
                         'most %d particles per array, sampled with a fixed seed) to compare '
                         'two builds output for output' % DUMP_SAMPLE)
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')

    rank = int(os.environ.get('RANK', '0'))
    local_rank = int(os.environ.get('LOCAL_RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    if args.dump_outputs and (args.impl != 'b200' or args.workload != 'dam_break' or world > 1):
        ap.error('--dump-outputs: only the single-GPU dam break (--impl b200 --workload '
                 'dam_break --gpus 1) writes its outputs')
    if world == 1 and args.gpus > 1:
        print('bench.py: --gpus %d needs torch.distributed.run with '
              '--nproc-per-node %d' % (args.gpus, args.gpus), file=sys.stderr)
        sys.exit(2)

    if args.impl == 'reference':
        run_reference(args, rank, world)
        return

    # stdout must carry exactly ONE JSON line: NCCL (and anything else native) may
    # print banners there, so fd 1 points at stderr until the result is ready
    sys.stdout.flush()
    saved_stdout = os.dup(1)
    os.dup2(2, 1)

    def emit(line):
        sys.stdout.flush()
        os.dup2(saved_stdout, 1)
        print(json.dumps(line))
        sys.stdout.flush()
    if args.workload == 'taylor_green' and world > 1:
        print('bench.py: --workload taylor_green is a single-GPU workload', file=sys.stderr)
        sys.exit(2)
    if world > 1:
        import torch
        import torch.distributed as dist
        torch.cuda.set_device(local_rank)
        dist.init_process_group('nccl', device_id=torch.device('cuda', local_rank))
    try:
        if args.workload == 'taylor_green':
            run_taylor_green(args, emit)
        elif args.workload == 'rings':
            run_rings(args, emit, rank, local_rank, world)
        else:
            line = run_dam_break(args, rank, local_rank, world)
            # BASELINE configs[3] (Taylor-Green, EDAC, one GPU) and configs[4] (colliding
            # rings, 4 GPUs; also on one) under the same clock, as sub-records
            extra = {}
            if not args.no_extras and not args.dx and args.scaling == 'weak':
                sub = argparse.Namespace(**vars(args))
                sub.steps, sub.warmup = min(args.steps, 20), min(args.warmup, 5)
                sub.e2e_steps = min(args.e2e_steps, 3)

                def grab(key):
                    def _emit(d):
                        extra[key] = d
                    return _emit
                if world == 1:
                    run_taylor_green(sub, grab('taylor_green'))
                if world in (1, 4):
                    run_rings(sub, grab('rings'), rank, local_rank, world)
            if rank == 0:
                if extra:
                    line['extra'] = extra
                emit(line)
    finally:
        if world > 1:
            import torch.distributed as dist
            if dist.is_initialized():
                dist.destroy_process_group()



def _timed_steps(solver, stream, K, barrier, reduce_max):
    """K steps bracketed by barrier + synchronize; device time, max over ranks"""
    import torch
    barrier()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record(stream)
    for _ in range(K):
        solver.step()
    ev1.record(stream)
    barrier()
    return reduce_max(ev0.elapsed_time(ev1)) / K


def multi_gpu_parity(rank, local_rank, world, kernel, steps=12, dx=0.03):
    """The N-rank slab run against ONE process on the same small dam break (dx = 0.03,
    ~60 k particles), matched by gid: the decomposition-invariance check of
    pysph/parallel/tests/test_parallel_run.py:36-49 inside the bench, so that the driver's
    scaling run carries multi-GPU field parity itself.  Returns a dict (rank 0) or None."""
    import torch
    import torch.distributed as dist
    import pysph_b200 as pb
    from pysph_b200 import geometry as geo
    from pysph_b200.parallel import make_slab_solver
    params = geo.dam_break_3d_params(dx)
    solver, pm, pas = make_slab_solver(dx, params, kernel, rank, world, device=local_rank)
    rs = np.random.RandomState(7)
    for _ in range(steps):
        solver.step()
    solver.pull()
    fields = ('x', 'y', 'z', 'u', 'v', 'w', 'rho')
    mine = []
    for pa in pas:
        nr = pa.get_number_of_particles(real=True)
        mine.append(np.column_stack([pa.properties['gid'][:nr].astype(np.float64)] +
                                    [pa.properties[k][:nr] for k in fields]))
    mine = np.concatenate(mine) if mine else np.zeros((0, 8))
    gathered = [None] * world
    dist.all_gather_object(gathered, mine)
    st = solver.backend.stats()
    stats = dict(full_updates=pm.n_full, refreshes=pm.n_refresh, peer_refreshes=pm.n_peer_refresh,
                 overlapped_evaluations=int(st.get('overlapped', 0) or 0),
                 ctas_interior=int(st.get('chunks_interior', 0) or 0),
                 ctas_boundary=int(st.get('chunks_boundary', 0) or 0),
                 fused_stages=int(st.get('fused_stages', 0) or 0))
    del solver, pm
    if rank != 0:
        return None
    allp = np.concatenate(gathered)
    allp = allp[np.argsort(allp[:, 0], kind='stable')]
    ref = geo.dam_break_3d_particles(dx=dx)
    s1 = pb.make_wcsph_solver(ref, dict(params), kernel, device=local_rank)
    for _ in range(steps):
        s1.step()
    s1.pull()
    one = np.concatenate([np.column_stack([pa.properties['gid'].astype(np.float64)] +
                                          [pa.properties[k] for k in fields]) for pa in ref])
    one = one[np.argsort(one[:, 0], kind='stable')]
    del s1
    ok = allp.shape == one.shape and np.array_equal(allp[:, 0], one[:, 0])
    err = {}
    if ok:
        h0, c0, rho0 = params['h0'], params['c0'], params['rho0']
        scale = dict(x=h0, y=h0, z=h0, u=c0, v=c0, w=c0, rho=rho0)
        for j, k in enumerate(fields):
            err[k] = float(np.max(np.abs(allp[:, j + 1] - one[:, j + 1])) / scale[k])
        ok = max(err.values()) <= 1e-9
    return dict(ok=bool(ok), particles=int(one.shape[0]), steps=steps, dx=dx,
                max_scaled_error=err, tolerance=1e-9, halo=stats,
                what='N-rank slabs vs one process, matched by gid; errors in units of '
                     'h0 (positions), c0 (velocities), rho0 (density)')


def run_dam_break(args, rank, local_rank, world):
    import torch
    import torch.distributed as dist
    import pysph_b200 as pb
    from pysph_b200 import geometry as geo

    torch.cuda.set_device(local_rank)
    dx = dam_break_dx(args, world)
    params = geo.dam_break_3d_params(dx)
    kernel = pb.CubicSpline(dim=3)
    W = max(args.warmup, 3)
    K = args.steps

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def reduce(v, op=None):
        if world == 1:
            return v
        t = torch.tensor([float(v)], dtype=torch.float64, device='cuda')
        dist.all_reduce(t, op=op or dist.ReduceOp.MAX)
        return float(t.item())

    parity = None
    if world > 1 and not args.no_parity:
        parity = multi_gpu_parity(rank, local_rank, world, kernel)
        if rank == 0 and not parity['ok']:
            sys.stderr.write('bench.py: MULTI-GPU PARITY FAILED: %r\n' % (parity,))
        flag = torch.tensor([1.0 if (parity is None or parity['ok']) else 0.0],
                            dtype=torch.float64, device='cuda')
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        if float(flag.item()) < 0.5:
            sys.exit(3)

    if world == 1:
        pas = geo.dam_break_3d_particles(dx=dx)
        host_copy = copy_arrays(pas) if not args.no_cpu else None
        keep = pinned_arrays(pas)
        solver = pb.make_wcsph_solver(pas, dict(params), kernel, device=local_rank)
        pm = None
    else:
        from pysph_b200.parallel import make_slab_solver
        solver, pm, pas = make_slab_solver(dx, params, kernel, rank, world,
                                           device=local_rank)
        host_copy = None
    be = solver.backend
    # run on torch's current stream so torch events / NCCL order with our kernels
    stream = torch.cuda.current_stream()
    be.use_torch_stream(stream)

    n_local = sum(be.sizes(i)[1] for i in range(len(pas)))

    def count_pairs_of_one_step():
        """one step with the device pair counter on (untimed); an evaluation that had to
        be repeated after a failed deferred drift check counts once (the repeat)"""
        total = [0]
        integ = solver.integrator
        orig_ca = integ.compute_accelerations

        def counting_ca(*a, **kw):
            orig_ca(*a, **kw)
            total[0] += solver.a_eval.last_pairs
        solver.a_eval.count_pairs = True
        integ.compute_accelerations = counting_ca
        solver.step()
        del integ.compute_accelerations
        solver.a_eval.count_pairs = False
        loc = total[0]
        if world > 1:
            t = torch.tensor([loc], dtype=torch.int64, device='cuda')
            dist.all_reduce(t)
            return loc, int(t.item())
        return loc, loc

    # nvidia-smi is started BEFORE the warm-up: its start-up (NVML init over every GPU
    # of the box) perturbs running kernels for tens of ms; only the lines it prints
    # during the timed region are used
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    solver.initialise()
    for _ in range(W):
        solver.step()
    pairs_local, pairs_total = count_pairs_of_one_step()

    # ---- timed region: exactly K steps, device resident ----------------------
    import gc

    def timed_steps():
        be.ctx.call('b200sph_reset_stats')
        be.ctx.call('b200sph_set_profiling', 2)      # events around the pair kernels only
        barrier()
        first_line = len(sampler.lines)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        if pm is not None and getattr(pm, '_prof', None) is not None:
            pm.profile_summary()
        # the host runs at most one evaluation ahead of the GPU (it reads the list-validity
        # answer of every evaluation), so a host pause is GPU idle time: no garbage
        # collection in here
        gc.collect()
        gc.disable()
        t0 = time.perf_counter()
        e0.record(stream)
        for _ in range(K):
            solver.step()
        e1.record(stream)
        cpu_ms = 1e3 * (time.perf_counter() - t0)
        gc.enable()
        barrier()
        return e0.elapsed_time(e1), be.stats(), cpu_ms, first_line

    ms_total, st, cpu_enqueue_ms, n_s0 = timed_steps()
    # the first K timed steps, not a re-measured region: the dump depends on the arguments only
    if args.dump_outputs:
        dump_outputs(be, args.dump_outputs)
    if os.environ.get('B200SPH_PM_PROFILE') and pm is None:
        sys.stderr.write('[pm-profile rank 0] per step: cpu_loop %.3f ms\n' % (cpu_enqueue_ms / K))
    if pm is not None and getattr(pm, '_prof', None) is not None:
        ps = pm.profile_summary()
        sys.stderr.write('[pm-profile rank %d] per step: cpu_loop %.3f ms; %s\n' % (
            rank, cpu_enqueue_ms / K,
            ', '.join('%s %.3f' % (k, v / K) for k, v in sorted(ps.items()))))
    # phase breakdown (diagnostic, NOT part of the timed region): every phase bracketed
    # by events, which costs ~25 event records per step
    DIAG = 20
    be.ctx.call('b200sph_reset_stats')
    be.ctx.call('b200sph_set_profiling', 1)
    ev2, ev3 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev2.record(stream)
    for _ in range(DIAG):
        solver.step()
    ev3.record(stream)
    torch.cuda.synchronize()
    st_diag = be.stats()
    be.ctx.call('b200sph_set_profiling', 0)
    ms_step = reduce(ms_total) / K
    ms_diag_step = reduce(ev2.elapsed_time(ev3)) / DIAG
    # The diagnostic pass runs the SAME steps right afterwards with MORE overhead (an event pair
    # around every phase).  If the timed steps took over 1.5 x as long, the GPU sat idle for a
    # third of the region: the host was stalled from outside (seen once in ~20 runs on these
    # shared boxes: 25 ms inside 20 steps, profiles/r02_summary.md).  Like a throttled run it
    # is taken again, once, and the line says so with both numbers.
    remeasured = None
    if ms_step > 1.5 * ms_diag_step:
        first = {'ms_per_step': ms_step, 'host_loop_ms_per_step': cpu_enqueue_ms / K,
                 'diagnostic_pass_ms_per_step': ms_diag_step,
                 'reason': 'the timed steps took > 1.5 x the diagnostic pass of the same steps '
                           '(GPU idle: host stalled)'}
        ms_total, st, cpu_enqueue_ms, n_s0 = timed_steps()
        be.ctx.call('b200sph_set_profiling', 0)
        ms_step = reduce(ms_total) / K
        remeasured = first
    clocks = sampler.stop(n_s0) if rank == 0 else None
    value = pairs_total / (ms_step * 1e-3)

    # ---- e2e: the same step through the host-buffer API ----------------------
    # every step: H2D of the state the step consumes (pinned host ParticleArray
    # buffers), the step, D2H of the output properties; one wait per step.  h and m do
    # not change in this scheme (no update_h): they went up once with the arrays.
    state = ['x', 'y', 'z', 'u', 'v', 'w', 'rho']
    outp = ['x', 'y', 'z', 'u', 'v', 'w', 'rho', 'p']
    if world > 1:
        # host mirrors hold this rank's real particles (sizes may have changed by
        # migration): refresh them once, then pin
        solver.pull()
        for pa in pas:
            nr = pa.get_number_of_particles(real=True)
            for k in list(pa.properties):
                pa.properties[k] = pa.properties[k][:nr].copy()
            pa._n = nr
        keep = pinned_arrays(pas)
    be.ctx.call('b200sph_set_async_copies', 1)
    n_full0 = pm.n_full if pm is not None else 0

    def e2e_step():
        be.push_real(state)      # H2D from pinned host ParticleArray buffers
        solver.step()
        be.pull_real(outp)       # D2H of the step's result
        be.synchronize()         # the host sees the result of every step
    ms_e2e, e2e_note = None, None
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    try:
        for _ in range(2):
            e2e_step()
        barrier()
        ev0.record(stream)
        for _ in range(args.e2e_steps):
            e2e_step()
        ev1.record(stream)
        barrier()
        ms_e2e = ev0.elapsed_time(ev1) / args.e2e_steps
    except ValueError as e:
        # a migration changed a rank's particle count under the host mirrors (push_real /
        # pull_real refuse to run past them): no e2e number rather than a wrong one
        e2e_note = 'skipped: %s' % e
    be.ctx.call('b200sph_set_async_copies', 0)
    nreal = sum(be.sizes(i)[1] for i in range(len(pas)))
    h2d, d2h = 8 * len(state) * nreal, 8 * len(outp) * nreal
    if world > 1:
        t = torch.tensor([ms_e2e if ms_e2e is not None else -1.0,
                          0.0 if ms_e2e is not None else 1.0], dtype=torch.float64, device='cuda')
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_e2e = None if float(t[1].item()) > 0.5 else float(t[0].item())
        t2 = torch.tensor([float(h2d), float(d2h)], dtype=torch.float64, device='cuda')
        dist.all_reduce(t2)
        h2d, d2h = int(t2[0].item()), int(t2[1].item())
    e2e = {'value': pairs_total / (ms_e2e * 1e-3) if ms_e2e else None, 'unit': 'pairs/s',
           'ms_per_step': ms_e2e, 'steps': args.e2e_steps,
           'h2d_bytes_per_step': h2d, 'd2h_bytes_per_step': d2h,
           'host_api': 'B200Backend.push_real(x y z u v w rho) -> B200Solver.step() -> '
                       'pull_real(x y z u v w rho p), pinned host ParticleArray buffers'}
    if e2e_note:
        e2e['note'] = e2e_note

    # ---- developed flow: the same steps from a state with 1-3 m/s random velocities -----
    # the timed region above starts from the t = 0 lattice ("quiet water": the neighbour
    # lists live for hundreds of evaluations); here they expire every few steps, so list
    # rebuilds, repeated evaluations after failed deferred checks and (N > 1) migration
    # and ghost re-import are inside the timed steps
    developed = None
    if not args.no_developed:
        rs = np.random.RandomState(1234 + rank)
        fl = pas[0]
        solver.pull()
        nr = fl.get_number_of_particles(real=True)
        if world > 1:
            for k in list(fl.properties):
                fl.properties[k] = fl.properties[k][:be.sizes(0)[0]]
        for k in ('u', 'v', 'w'):
            fl.properties[k][:nr] += rs.normal(scale=2.0, size=nr)
        be.push_real_array(0, ['u', 'v', 'w'])
        Wd, Kd = 10, max(min(K, 40), 10)
        for _ in range(Wd):
            solver.step()
        pl, pt = count_pairs_of_one_step()
        be.ctx.call('b200sph_reset_stats')
        be.ctx.call('b200sph_set_profiling', 1)
        pm_full0 = pm.n_full if pm is not None else 0
        pm_fail0 = pm.n_deferred_failed if pm is not None else 0
        ms_dev = _timed_steps(solver, stream, Kd, barrier, reduce)
        std = be.stats()
        be.ctx.call('b200sph_set_profiling', 0)
        developed = {
            'value': pt / (ms_dev * 1e-3), 'unit': 'pairs/s', 'ms_per_step': ms_dev,
            'steps': Kd, 'warmup': Wd, 'pairs_per_step': pt,
            'state': 'the timed state + N(0, 2 m/s) on every fluid velocity component, '
                     '%d steps later' % Wd,
            'full_builds': int(std['full_builds']), 'list_builds': int(std['list_builds']),
            'light_updates': int(std['light_updates']),
            'deferred_failed': int(std['deferred_failed']),
            'proactive_builds': int(std.get('proactive_builds', 0) or 0),
            'ms_nnps_per_step': std['ms_nnps'] / Kd,
            'ms_per_rebuild': (std['ms_nnps'] / max(int(std['full_builds']), 1))
            if std['full_builds'] else None,
            'note': 'events around every phase are on in this region (ms_nnps needs them): '
                    'ms_per_step is ~2 % pessimistic',
        }
        if pm is not None:
            developed['halo_full_updates'] = pm.n_full - pm_full0
            developed['halo_deferred_failed'] = pm.n_deferred_failed - pm_fail0
            developed['halo_proactive'] = pm.n_proactive

    # ---- roofline of the dominant kernel (k_pair_list), from the timed region -----
    peak, peak_src = peaks()
    ms_pair = st['ms_pair'] / max(st['pair_launches'], 1)
    pairs_per_launch = pairs_local / 2.0     # EPEC: two evaluations per step
    achieved = pairs_per_launch * BYTES_PER_PAIR / (ms_pair * 1e-3) / 1e9
    lists = bool(st['list_builds'] or st['light_updates'])
    roofline = {'bound': 'hbm',      # the contract's class (memory, not tensor) = the denominator used
                'limiter_ncu': 'L1/TEX gather path 85 % (LSU data-pipe wavefronts) + long-scoreboard latency '
                               '(issue active 73 %, 41 % warps active; profiles/r02e_lb_raw.csv); DRAM at '
                               '15 % of peak -- NOT HBM-bound: "achieved" charges every gathered '
                               'record to HBM as SURVEY 8d defines it, the records are served by L1/L2',
                'kernel': 'k_pair_list<CubicSpline,3>' if lists else 'k_pair<CubicSpline,3>',
                'achieved': achieved, 'peak': peak, 'unit': 'GB/s',
                'frac': achieved / peak, 'traffic': None,
                'peak_source': peak_src,
                'algorithmic_bytes_per_pair': BYTES_PER_PAIR,
                'pairs_per_launch': pairs_per_launch,
                'avg_launch_ms': ms_pair,
                'share_of_step': st['ms_pair'] / K / ms_step,
                'ms_nnps_per_step': st_diag['ms_nnps'] / DIAG,
                'ms_other_per_step': st_diag['ms_other'] / DIAG,
                'breakdown': 'nnps/other: separate %d-step pass after the timed region' % DIAG,
                'nnps': {'full_builds': st['full_builds'],
                         'light_updates': st['light_updates'],
                         'list_builds': st['list_builds'],
                         'list_entries_per_particle': st['list_entries_per_particle'],
                         'fused_stages': st.get('fused_stages')}}
    if world > 1:
        roofline['note'] = ('rank 0; with the halo in flight the pair work is two launches '
                            '(ghost-free CTAs, then the rest behind the halo): avg_launch_ms '
                            'spans both and whatever wait lies between them')
    prof = os.path.join(ROOT, 'profiles', 'pair_traffic.json')
    if world == 1 and abs(dx - BASE_DX) < 1e-9 and os.path.exists(prof):
        # measured DRAM bytes of this kernel on THIS workload (ncu --set full, N = 1,
        # dx = 0.00877; profiles/): the per-pair gathers are served by L1/L2 (records of
        # one cell neighbourhood are re-read ~80x), DRAM streams the neighbour lists
        try:
            roofline['traffic'] = json.load(open(prof)).get('dram_bytes_per_launch')
        except Exception:
            pass
    if roofline['traffic']:
        roofline['dram_gbs'] = roofline['traffic'] / (ms_pair * 1e-3) / 1e9
        roofline['dram_frac'] = roofline['dram_gbs'] / peak
    per_rank = None
    if world > 1:
        nov = max(int(st.get('overlapped', 0) or 0), 1)
        mine = torch.tensor([st['ms_pair'] / K, st_diag['ms_nnps'] / DIAG, st_diag['ms_other'] / DIAG,
                             float(n_local), float(pairs_local),
                             float(st.get('ms_halo_chain', 0.0)) / nov, float(st.get('ms_pair_wall', 0.0)) / nov,
                             float(st.get('ms_halo_sent', 0.0)) / nov, float(st.get('ms_halo_reduced', 0.0)) / nov],
                            dtype=torch.float64, device='cuda')
        allr = [torch.zeros_like(mine) for _ in range(world)]
        dist.all_gather(allr, mine)
        # ms_pair: the main-stream launch (the ghost-free CTAs) per STEP; ms_halo_chain /
        # ms_pair_wall: per EVALUATION, from the fork of the communication stream to the end of
        # the ghost scatter / to the end of both pair launches
        per_rank = [dict(zip(('ms_pair', 'ms_nnps', 'ms_other', 'n_real', 'pairs', 'ms_halo_chain',
                              'ms_pair_wall', 'ms_halo_sent', 'ms_halo_reduced'),
                             [round(float(v), 4) for v in r.tolist()])) for r in allr]
    n_total = int(reduce(n_local, dist.ReduceOp.SUM)) if world > 1 else n_local
    halo = None
    if pm is not None:
        halo = {'full_updates': pm.n_full, 'refreshes': pm.n_refresh,
                'peer_refreshes': pm.n_peer_refresh, 'peer_sync': bool(getattr(pm, '_peer_sync', False)),
                'overlapped_evaluations': int(st.get('overlapped', 0) or 0),
                'ctas_interior': int(st.get('chunks_interior', 0) or 0),
                'ctas_boundary': int(st.get('chunks_boundary', 0) or 0)}

    # ---- BASELINE configs[2] exactly as quoted (dx = 0.00407, ~11.3 M particles) on the
    #      same N = 8 GPUs: the weak-scaling series above stops at 9.1 M ----------------
    c3 = None
    if world == 8 and args.scaling == 'weak' and not args.dx and not args.no_extras:
        del solver, pm
        from pysph_b200.parallel import make_slab_solver
        p3 = geo.dam_break_3d_params(C3_DX)
        s3, pm3, pas3 = make_slab_solver(C3_DX, p3, kernel, rank, world, device=local_rank)
        s3.backend.use_torch_stream(stream)
        solver = s3
        for _ in range(W):
            s3.step()
        be3 = s3.backend
        n3 = int(reduce(sum(be3.sizes(i)[1] for i in range(len(pas3))), dist.ReduceOp.SUM))
        total = [0]
        orig = s3.integrator.compute_accelerations

        def cca(*a, **kw):
            orig(*a, **kw)
            total[0] += s3.a_eval.last_pairs
        s3.a_eval.count_pairs = True
        s3.integrator.compute_accelerations = cca
        s3.step()
        del s3.integrator.compute_accelerations
        s3.a_eval.count_pairs = False
        p3t = int(reduce(total[0], dist.ReduceOp.SUM))
        ms3 = _timed_steps(s3, stream, K, barrier, reduce)
        c3 = {'workload': dam_break_workload(C3_DX, world), 'particles': n3,
              'pairs_per_step': p3t, 'ms_per_step': ms3, 'steps': K, 'warmup': W,
              'value': p3t / (ms3 * 1e-3), 'unit': 'pairs/s',
              'halo': {'full_updates': pm3.n_full, 'refreshes': pm3.n_refresh}}

    if rank != 0:
        return None

    # ---- CPU baseline (rank 0, N = 1): the oracle on a bounded sample --------
    cpu = None
    if world == 1 and not args.no_cpu:
        try:
            r = cpu_leg(host_copy, params, 1, budget_s=args.cpu_budget, max_steps=1)
            cpu = {'value': r['pairs_per_s'], 'unit': 'pairs/s', 'cores': 1,
                   'kind': 'port', 'cpu': cpu_model(),
                   'sample': '%d full EPEC step(s) of the same %d-particle state from '
                             't=0, fp64 oracle, 1 thread (%.1f s)'
                             % (r['steps'], sum(p.get_number_of_particles()
                                                for p in host_copy), r['seconds'])}
        except Exception as e:      # the CPU leg must not cost the measured GPU line
            cpu = {'value': None, 'unit': 'pairs/s', 'cores': 1, 'kind': 'port',
                   'error': '%s: %s' % (type(e).__name__, e)}

    line = {
        'metric': METRIC, 'value': value, 'unit': 'pairs/s', 'n_gpus': world,
        'steps': K, 'warmup': W, 'ms_per_step': ms_step,
        'steps_per_s': 1e3 / ms_step, 'higher_is_better': True,
        'scaling': args.scaling, 'vs_baseline': None, 'dtype': 'f32',
        'data': 'synthetic',
        'config': {'workload': dam_break_workload(dx, world),
                   'regime': 'from the t = 0 lattice (quiet water: no list rebuild inside the '
                             'timed steps); see "developed" for the same steps with rebuilds',
                   'particles': n_total,
                   'particles_rank0': n_local,
                   'pairs_per_step': pairs_total,
                   'per_rank': per_rank,
                   'deferred_failed': int(st['deferred_failed']),
                   'parallelism': 'single GPU' if world == 1 else
                                  'x-slabs x%d, halo over peer memory (NVLink) under the '
                                  'interior pair work' % world,
                   'multi_gpu_parity': parity,
                   'halo': halo,
                   'l2': 'no flush: per-step working set (~220 B/particle state '
                         '+ 48 B/particle packed records, > 126 MB L2 at 1.2 M '
                         'particles) and the state advances every step',
                   'precision': 'fp32 pair arithmetic on cell-relative '
                                'coordinates, fp64 integrated state'},
        'clocks': clocks,
        'e2e': e2e,
        'gpu_launches': int(st['kernel_launches']),
        'launches_per_step': st['kernel_launches'] / float(K),
        # wall time of the host loop that enqueued the timed steps (it waits for the GPU once per
        # evaluation): ~ ms_per_step when the GPU is the bottleneck, larger when the host was
        'host_loop_ms_per_step': cpu_enqueue_ms / float(K),
        # not None: the first K timed steps were disturbed from outside and taken again (see there)
        'remeasured': remeasured,
        'roofline': roofline,
    }
    if developed:
        line['developed'] = developed
    if c3:
        line['configs2_as_quoted'] = c3
    if cpu:
        line['cpu_baseline'] = cpu
    return line


if __name__ == '__main__':
    main()
