"""Multi-GPU parity (needs >= 2 CUDA devices): the slab decomposition with the
NCCL halo exchange reproduces the single-GPU run, matched by gid -- the mirror
of the reference's serial-vs-4-ranks dam_break_3d test
(pysph/parallel/tests/test_parallel_run.py:36-49, example_test_case.py:146-166).
"""
import os
import socket

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

DX = 0.04
NSTEPS = 25


def _ngpus():
    try:
        import torch
        return torch.cuda.device_count()
    except Exception:
        return 0


def _free_port():
    s = socket.socket()
    s.bind(('127.0.0.1', 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _perturb(pas):
    """Deterministic (gid based) velocity field so that particles migrate and
    the ghost values change every evaluation."""
    f = pas[0]
    g = f.gid.astype(np.float64)
    f.u[:] = 2.0 * np.sin(0.37 * g) + 1.5
    f.v[:] = 1.0 * np.cos(0.11 * g)
    f.w[:] = 0.5 * np.sin(0.05 * g)
    f.rho[:] = 1000.0 * (1.0 + 0.005 * np.sin(0.23 * g))


def _collect(pas):
    out = {}
    for pa in pas:
        nr = pa.get_number_of_particles(real=True)
        out[pa.name] = dict((k, pa.properties[k][:nr].copy())
                            for k in ('gid', 'x', 'y', 'z', 'u', 'v', 'w', 'rho'))
    return out


def _worker(rank, world, port, q):
    import torch
    import torch.distributed as dist
    import pysph_b200 as pb
    from pysph_b200 import geometry as geo
    from pysph_b200.parallel import make_slab_solver
    os.environ['MASTER_ADDR'] = '127.0.0.1'
    os.environ['MASTER_PORT'] = str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group('nccl', rank=rank, world_size=world,
                            device_id=torch.device('cuda', rank))
    try:
        params = geo.dam_break_3d_params(DX)
        solver, pm, pas = make_slab_solver(DX, params, pb.CubicSpline(dim=3), rank,
                                           world, device=rank,
                                           adaptive_timestep=False, n_damp=0)
        _perturb(pas)
        solver.backend.push_all()
        solver.backend.use_torch_stream()
        for _ in range(NSTEPS):
            solver.step()
        solver.pull()
        q.put((rank, _collect(pas), pm.n_full, pm.n_refresh,
               solver.backend.stats(), pm.n_peer_refresh))
    finally:
        dist.destroy_process_group()


@pytest.mark.skipif(_ngpus() < 2, reason='needs >= 2 GPUs')
@pytest.mark.parametrize('world', [2])
def test_slab_decomposition_matches_single_gpu(world):
    import torch.multiprocessing as mp
    import pysph_b200 as pb
    from pysph_b200 import geometry as geo

    # single-GPU reference run
    params = geo.dam_break_3d_params(DX)
    pas = geo.dam_break_3d_particles(dx=DX)
    _perturb(pas)
    s = pb.make_wcsph_solver(pas, dict(params), pb.CubicSpline(dim=3),
                             adaptive_timestep=False, n_damp=0)
    for _ in range(NSTEPS):
        s.step()
    s.pull()
    ref = _collect(pas)

    ctx = mp.get_context('spawn')
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, world, port, q))
             for r in range(world)]
    for p in procs:
        p.start()
    out = [q.get(timeout=300) for _ in range(world)]
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    n_full = [o[2] for o in out]
    n_refresh = [o[3] for o in out]
    # the ghost sets were reused (refresh path) and rebuilt (fast particles)
    assert min(n_refresh) > 0 and min(n_full) >= 2, (n_full, n_refresh)
    # the refreshes went over peer memory (NVLink stores), not NCCL send/recv
    assert min(o[5] for o in out) > 0, [o[5] for o in out]
    h0, c0 = params['h0'], params['c0']
    for name in ref:
        g_all = np.concatenate([o[1][name]['gid'] for o in out])
        assert np.array_equal(np.sort(g_all), np.sort(ref[name]['gid'])), name
        order_ref = np.argsort(ref[name]['gid'])
        order = np.argsort(g_all)
        for k, tol in (('x', 2e-6 * h0), ('y', 2e-6 * h0), ('z', 2e-6 * h0),
                       ('u', 2e-6 * c0), ('v', 2e-6 * c0), ('w', 2e-6 * c0),
                       ('rho', 2e-4)):
            a = np.concatenate([o[1][name][k] for o in out])[order]
            b = ref[name][k][order_ref]
            assert np.max(np.abs(a - b)) <= tol, (name, k, np.max(np.abs(a - b)))
