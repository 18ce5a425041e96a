"""Slab re-cut (SURVEY.md 8e "re-cut every K steps"): `b200sph_column_counts` /
`k_column_counts` and `SlabParallelManager._recut`.  Also covered on the host emulation of
the library (tests/test_library_on_cpu.py: slab decomposition with lb_freq=2 on 3 ranks)
and with the numpy test double (tests/test_parallel_gloo.py: test_slab_recut_gloo).  The
2-GPU test skips on a machine with one GPU."""
import numpy as np
import pytest

pytestmark = [pytest.mark.gpu,
              pytest.mark.timeout(300)]


def test_column_counts_match_numpy(gpu_device):
    import pysph_b200 as pb
    from pysph_b200.parallel import DeviceHaloOps
    rs = np.random.RandomState(3)
    pas = []
    for name, n in (('fluid', 70001), ('wall', 3333), ('empty', 0)):
        x = np.sort(rs.uniform(-0.2, 3.4, n)) if name == 'fluid' else rs.uniform(-0.2, 3.4, n)
        pas.append(pb.get_particle_array_wcsph(name=name, x=x, y=x * 0, z=x * 0,
                                               h=0.1, m=1.0, rho=1.0))
    be = pb.B200Backend(pas, extra_capacity=100)
    ops = DeviceHaloOps(be, 0)
    x0, width, nbins = 0.0, 0.05, 64          # particles below / above go to the end bins
    weights = [1.0, 0.45, 7.0]
    got = ops.column_weights(x0, width, nbins, weights).cpu().numpy()
    want = np.zeros(nbins)
    for pa, w in zip(pas, weights):
        b = np.clip(np.floor((pa.x - x0) / width).astype(int), 0, nbins - 1)
        want += w * np.bincount(b, minlength=nbins)
    assert np.array_equal(got, want)
    # ghosts are not counted
    buf = ops.new_buffer(9 * 10)
    buf[:] = 1.0
    ops.append(0, buf, 0, 10, 9, False)
    got2 = ops.column_weights(x0, width, nbins, weights).cpu().numpy()
    assert np.array_equal(got2, want)


def _worker(rank, world, port, q):
    import os
    import torch
    import torch.distributed as dist
    import pysph_b200 as pb
    from pysph_b200 import geometry as geo
    from pysph_b200.parallel import make_slab_solver
    import test_gpu_multi as M
    os.environ['MASTER_ADDR'] = '127.0.0.1'
    os.environ['MASTER_PORT'] = str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group('nccl', rank=rank, world_size=world,
                            device_id=torch.device('cuda', rank))
    try:
        params = geo.dam_break_3d_params(M.DX)
        solver, pm, pas = make_slab_solver(M.DX, params, pb.CubicSpline(dim=3), rank, world,
                                           device=rank, adaptive_timestep=False, n_damp=0,
                                           lb_freq=2)
        pm.lb_weights = [1.0] + [0.1] * (len(pas) - 1)    # != the 0.45 the cuts were made with
        M._perturb(pas)
        solver.backend.push_all()
        solver.backend.use_torch_stream()
        for _ in range(M.NSTEPS):
            solver.step()
        solver.pull()
        q.put((rank, M._collect(pas), pm.n_recut, list(pm.cuts)))
    finally:
        dist.destroy_process_group()


def test_recut_slabs_match_single_gpu():
    import torch
    import torch.multiprocessing as mp
    import pysph_b200 as pb
    from pysph_b200 import geometry as geo, parallel
    import test_gpu_multi as M
    if torch.cuda.device_count() < 2:
        pytest.skip('needs >= 2 GPUs')
    world = 2
    params = geo.dam_break_3d_params(M.DX)
    pas = geo.dam_break_3d_particles(dx=M.DX)
    M._perturb(pas)
    s = pb.make_wcsph_solver(pas, dict(params), pb.CubicSpline(dim=3),
                             adaptive_timestep=False, n_damp=0)
    for _ in range(M.NSTEPS):
        s.step()
    s.pull()
    ref = M._collect(pas)
    ctx = mp.get_context('spawn')
    q = ctx.Queue()
    port = M._free_port()
    procs = [ctx.Process(target=_worker, args=(r, world, port, q)) for r in range(world)]
    for p in procs:
        p.start()
    out = [q.get(timeout=240) for _ in range(world)]
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    static = parallel.balanced_cuts(*parallel.dam_break_column_weights(M.DX, solid_weight=0.45),
                                    world, M.DX)
    assert all(o[2] >= 1 for o in out) and out[0][3] == out[1][3] != static
    h0, c0 = params['h0'], params['c0']
    for name in ref:
        g_all = np.concatenate([o[1][name]['gid'] for o in out])
        assert np.array_equal(np.sort(g_all), np.sort(ref[name]['gid'])), name
        order_ref, order = np.argsort(ref[name]['gid']), np.argsort(g_all)
        for k, tol in (('x', 2e-6 * h0), ('y', 2e-6 * h0), ('z', 2e-6 * h0), ('u', 2e-6 * c0),
                       ('v', 2e-6 * c0), ('w', 2e-6 * c0), ('rho', 2e-4)):
            a = np.concatenate([o[1][name][k] for o in out])[order]
            assert np.max(np.abs(a - ref[name][k][order_ref])) <= tol, (name, k)
