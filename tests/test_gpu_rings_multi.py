"""Elastic-dynamics slab decomposition (BASELINE configs[4] is a 4-GPU case): the
16-field ghost message, the 30-field migration message and group 1 on a two-support halo.
The same comparison runs on the library emulation over gloo with 3 ranks
(tests/test_library_on_cpu.py::test_rings_slab_decomposition_on_the_emulated_library);
here it runs on 2 GPUs with the peer-memory refresh and skips on a machine with one GPU;
the layout tests run on one."""
import os

import numpy as np
import pytest

from test_gpu_multi import _free_port, _ngpus
from test_library_on_cpu import RINGS, RING_FIELDS, _rings_collect, _rings_perturb

pytestmark = [pytest.mark.gpu, pytest.mark.timeout(300)]


def _worker(rank, world, port, q):
    import torch
    import torch.distributed as dist
    from pysph_b200.parallel import make_rings_slab_solver
    os.environ['MASTER_ADDR'] = '127.0.0.1'
    os.environ['MASTER_PORT'] = str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group('nccl', rank=rank, world_size=world,
                            device_id=torch.device('cuda', rank))
    try:
        solver, pm, pas = make_rings_slab_solver(RINGS['dx'], RINGS['lz'], rank, world,
                                                 device=rank, dt=RINGS['dt'],
                                                 geometry_kw=dict(u_f=RINGS['u_f']))
        _rings_perturb(pas[0])
        solver.backend.push_all()
        solver.backend.use_torch_stream()
        for _ in range(RINGS['steps']):
            solver.step()
        solver.pull()
        q.put((rank, _rings_collect(pas[0]), pm.n_full, pm.n_refresh, pm.n_peer_refresh))
    finally:
        dist.destroy_process_group()


@pytest.mark.skipif(_ngpus() < 2, reason='needs >= 2 GPUs')
def test_rings_slabs_match_single_gpu():
    import torch.multiprocessing as mp
    import pysph_b200 as pb
    from pysph_b200 import geometry as geo
    world = 2
    pa = geo.rings_3d_particles(dx=RINGS['dx'], lz=RINGS['lz'], u_f=RINGS['u_f'])
    _rings_perturb(pa)
    s = pb.make_elastic_solver([pa], pb.ElasticSolidsScheme(['solid'], [], dim=3),
                               pb.CubicSpline(dim=3), dt=RINGS['dt'])
    for _ in range(RINGS['steps']):
        s.step()
    s.pull()
    ref = _rings_collect(pa)
    ctx = mp.get_context('spawn')
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, world, port, q)) for r in range(world)]
    for p in procs:
        p.start()
    out = [q.get(timeout=240) for _ in range(world)]
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    assert min(o[2] for o in out) >= 2
    g_all = np.concatenate([o[1]['gid'] for o in out])
    assert np.array_equal(np.sort(g_all), np.sort(ref['gid']))
    order_ref, order = np.argsort(ref['gid']), np.argsort(g_all)
    c0 = pa.cs[0]
    smax = np.max(np.abs(ref['s00']))
    tols = dict(x=1e-7 * 0.08, y=1e-7 * 0.08, z=1e-7 * 0.08, u=2e-6 * c0, v=2e-6 * c0,
                w=2e-6 * c0, rho=5e-6)
    for k in RING_FIELDS:
        a = np.concatenate([o[1][k] for o in out])[order]
        assert np.max(np.abs(a - ref[k][order_ref])) <= tols.get(k, 2e-4 * smax), k


S6 = ['s00', 's01', 's02', 's11', 's12', 's22']
F9 = ['x', 'y', 'z', 'u', 'v', 'w', 'rho', 'h', 'm']
F16 = F9 + ['x0', 'y0', 'z0', 'u0', 'v0', 'w0', 'rho0']


def test_elastic_halo_and_migration_layout(gpu_device):
    """One GPU: with elastic-dynamics arrays b200sph_halo_layout reports 16 / 30 fields, the
    ghost message is x y z u v w rho h m s00 s01 s02 s11 s12 s22 cs, the migration message
    the 16 fp64 state properties, gid, s00..s22, s000..s220, cs -- field-major, exact."""
    import pysph_b200 as pb
    from pysph_b200.parallel import DeviceHaloOps
    rs = np.random.RandomState(5)
    n = 400
    props = dict((k, rs.uniform(0.1, 1.0, n)) for k in F16 + S6 + [k + '0' for k in S6])
    props['x'] = rs.uniform(0.0, 3.0, n)
    props['cs'] = rs.uniform(10.0, 20.0, n)
    mk = lambda name: pb.get_particle_array_elastic_dynamics(
        name=name, constants=dict(E=1e7, nu=0.3, rho_ref=1.0, c0_ref=5.0), **props)
    a, b = mk('solid'), mk('other')
    a.gid[:] = np.arange(n) + 7
    ref = dict((k, v.copy()) for k, v in a.properties.items())
    cs32 = ref['cs'].astype(np.float32).astype(np.float64)      # cs is fp32 on the device
    be = pb.B200Backend([a, b], extra_capacity=2000)
    ops = DeviceHaloOps(be, 0)
    assert (ops.halo_nf, ops.migrate_nf) == (16, 30)
    lo, hi = 1.0, 1.6
    buf = ops.new_buffer(16 * n)
    cnt = ops.pack(0, 1, lo, hi, buf, 0)
    sel = np.where((ref['x'] >= lo) & (ref['x'] < hi))[0]
    assert cnt == sel.size and cnt > 20
    got = buf[:16 * cnt].cpu().numpy().reshape(16, cnt)
    for f, k in enumerate(F9 + S6):
        assert np.array_equal(got[f], ref[k][sel]), k
    assert np.array_equal(got[15], cs32[sel])
    ops.append(1, buf, 0, cnt, 16, False)
    assert be.sizes(1) == (n + cnt, n)
    be.pull(1)
    for k in F9 + S6:
        assert np.array_equal(b.properties[k][n:], ref[k][sel]), k
    assert np.array_equal(b.cs[n:], cs32[sel]) and np.all(b.s000[n:] == 0.0)
    assert np.all(b.tag[n:] == 1)
    # the refresh message of ALL arrays in one kernel (what the peer-memory path sends) and
    # its scatter onto the existing ghosts: same layout, current values
    a.s01[:] = ref['s01'] + 3.0
    a.cs[:] = ref['cs'] * 2.0
    be.push(0, ['s01', 'cs'])
    buf2 = ops.new_buffer(16 * n)
    nd = ops.pack_selected_all(1, buf2.data_ptr(), buf2.numel())
    assert nd == 16 * cnt
    got2 = buf2[:nd].cpu().numpy().reshape(16, cnt)
    assert np.array_equal(got2[10], ref['s01'][sel] + 3.0) and np.array_equal(got2[0], ref['x'][sel])
    assert np.array_equal(got2[15], (ref['cs'] * 2.0).astype(np.float32).astype(np.float64)[sel])
    ops.overwrite_all([0, 0], [0, cnt], buf2.data_ptr())
    be.pull(1, ['s01', 'cs', 'x'])
    assert np.array_equal(b.s01[n:], ref['s01'][sel] + 3.0)
    assert np.array_equal(b.cs[n:], (ref['cs'] * 2.0).astype(np.float32).astype(np.float64)[sel])
    assert np.array_equal(b.x[n:], ref['x'][sel])
    a.s01[:] = ref['s01']
    a.cs[:] = ref['cs']
    be.push(0, ['s01', 'cs'])
    ops.drop_ghosts(1)
    mbuf = ops.new_buffer(30 * n)
    n_lo, n_hi = ops.migrate_out(0, 0.5, 2.5, mbuf, 0)
    s_lo = np.where(ref['x'] < 0.5)[0]
    keep = np.where((ref['x'] >= 0.5) & (ref['x'] < 2.5))[0]
    assert n_lo == s_lo.size > 0 and n_hi > 0
    blk = mbuf[:30 * n_lo].cpu().numpy().reshape(30, n_lo)
    names = F16 + ['gid'] + S6 + [k + '0' for k in S6]
    for f, k in enumerate(names):
        assert np.array_equal(blk[f], ref[k][s_lo].astype(float)), k
    assert np.array_equal(blk[29], cs32[s_lo])
    be.pull(0)
    for k in F16 + S6 + [k + '0' for k in S6]:
        assert np.array_equal(a.properties[k], ref[k][keep]), k
    assert np.array_equal(a.cs, cs32[keep]) and np.array_equal(a.gid, ref['gid'][keep])
    ops.append(1, mbuf, 0, n_lo, 30, True)
    assert be.sizes(1) == (n + n_lo, n + n_lo)
    be.pull(1)
    for k in F16 + S6 + [k + '0' for k in S6]:
        assert np.array_equal(b.properties[k][n:], ref[k][s_lo]), k
    assert np.array_equal(b.cs[n:], cs32[s_lo]) and np.array_equal(b.gid[n:], ref['gid'][s_lo])
    assert np.all(b.tag[n:] == 0)


def test_empty_elastic_array_agrees_on_the_message_layout(gpu_device):
    """A rank whose slab holds no particle must still report the 16 / 30-field layout (its
    neighbours size their messages with it): pushing an EMPTY elastic array allocates the
    elastic-dynamics pool."""
    import ctypes as C
    import pysph_b200 as pb
    pa = pb.get_particle_array_elastic_dynamics(name='solid', x=np.zeros(0))
    be = pb.B200Backend([pa], extra_capacity=64)
    be.push_all()
    h, m = C.c_int(), C.c_int()
    be.ctx.call('b200sph_halo_layout', C.byref(h), C.byref(m))
    assert (h.value, m.value) == (16, 30)
    q = pb.get_particle_array_wcsph(name='fluid', x=np.zeros(0))
    be2 = pb.B200Backend([q], extra_capacity=64)
    be2.push_all()
    be2.ctx.call('b200sph_halo_layout', C.byref(h), C.byref(m))
    assert (h.value, m.value) == (9, 17)
