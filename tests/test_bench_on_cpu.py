"""bench.py's GPU arms end to end on the CPU: the library emulation stands in for
libb200sph.so (tests/test_library_on_cpu.py) and a few lines of fake `torch.cuda` (events
that read the wall clock, no-op synchronize / set_device, pin_memory = identity) stand in
for the device.  This checks the code NO CPU test otherwise executes -- workload set-up,
pair counting, the timed loop, the e2e loop, the roofline / cpu_baseline arithmetic and the
JSON line's keys -- at sizes that take seconds.  The numbers it produces mean nothing."""
import importlib
import io
import json
import os
import sys
import time

import pytest

from test_library_on_cpu import emulated_library  # noqa: F401  (fixture)

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


class _Event(object):
    def __init__(self, enable_timing=False):
        self.t = None

    def record(self, stream=None):
        self.t = time.perf_counter()

    def synchronize(self):
        pass

    def elapsed_time(self, other):
        return max(1e3 * (other.t - self.t), 1e-3)


class _Stream(object):
    cuda_stream = 0


@pytest.fixture
def fake_cuda(monkeypatch):
    import torch
    monkeypatch.setattr(torch.cuda, 'Event', _Event)
    monkeypatch.setattr(torch.cuda, 'synchronize', lambda *a, **k: None)
    monkeypatch.setattr(torch.cuda, 'set_device', lambda *a, **k: None)
    monkeypatch.setattr(torch.cuda, 'current_stream', lambda *a, **k: _Stream())
    monkeypatch.setattr(torch.Tensor, 'pin_memory', lambda self, *a, **k: self)
    return torch


CONTRACT = ['metric', 'value', 'unit', 'n_gpus', 'steps', 'warmup', 'ms_per_step',
            'higher_is_better', 'scaling', 'vs_baseline', 'dtype', 'data', 'config', 'clocks',
            'e2e', 'gpu_launches', 'roofline', 'cpu_baseline']


def _bench_line(monkeypatch, capfd, argv):
    """bench.main() in this process; returns its one JSON line"""
    sys.path.insert(0, ROOT)
    bench = importlib.import_module('bench')
    monkeypatch.setattr(sys, 'argv', ['bench.py', '--steps', '3', '--warmup', '3',
                                      '--e2e-steps', '2', '--cpu-budget', '5'] + argv)
    for k in ('RANK', 'LOCAL_RANK', 'WORLD_SIZE'):
        monkeypatch.delenv(k, raising=False)
    saved = os.dup(1)
    try:
        bench.main()
    finally:
        os.dup2(saved, 1)           # bench points fd 1 at stderr until its line is ready
        os.close(saved)
    out = capfd.readouterr().out
    lines = [ln for ln in out.splitlines() if ln.startswith('{')]
    assert len(lines) == 1, out[-2000:]
    return json.loads(lines[0])


@pytest.mark.parametrize('argv', [
    ['--dx', '0.08'],
    ['--workload', 'taylor_green', '--nx', '10'],
    ['--workload', 'rings', '--dx', '0.0025', '--lz', '0.0075'],
], ids=['dam_break', 'taylor_green', 'rings'])
def test_bench_gpu_arm_on_the_emulated_library(emulated_library, fake_cuda, monkeypatch,  # noqa: F811
                                               capfd, argv):
    d = _bench_line(monkeypatch, capfd, argv)
    for k in CONTRACT:
        assert k in d, k
    assert d['unit'] == 'pairs/s' and d['n_gpus'] == 1 and d['steps'] == 3 and d['warmup'] == 3
    assert d['value'] > 0 and d['ms_per_step'] > 0 and d['higher_is_better'] is True
    assert d['gpu_launches'] > 0 and d['config']['pairs_per_step'] > 0
    assert 'workload' in d['config'] and 'model' not in d['config']
    e = d['e2e']
    assert e['value'] > 0 and e['h2d_bytes_per_step'] > 0 and e['d2h_bytes_per_step'] > 0
    r = d['roofline']
    for k in ('bound', 'achieved', 'peak', 'unit', 'frac', 'traffic'):
        assert k in r, k
    assert r['bound'] == 'hbm' and r['unit'] == 'GB/s' and r['peak'] > 0
    c = d['cpu_baseline']
    assert c['kind'] == 'port' and c['cores'] == 1 and c['value'] > 0 and c['sample']


def test_bench_dump_outputs_on_the_emulated_library(emulated_library, fake_cuda,  # noqa: F811
                                                    monkeypatch, capfd, tmp_path):
    """--dump-outputs DIR: the same arguments write the same files (float64, rows in gid order,
    arrays above the sample size sampled), and --steps sets how far the dumped state got."""
    import numpy as np
    sys.path.insert(0, ROOT)
    bench = importlib.import_module('bench')
    monkeypatch.setattr(bench, 'DUMP_SAMPLE', 200)
    base = ['--dx', '0.08', '--no-cpu', '--no-developed', '--no-extras']
    runs = {}
    for tag, steps in (('a', 3), ('b', 3), ('c', 4)):
        d = _bench_line(monkeypatch, capfd, base + ['--steps', str(steps),
                                                    '--dump-outputs', str(tmp_path / tag)])
        assert d['steps'] == steps
        runs[tag] = dict((p.name[:-4], np.load(p)) for p in (tmp_path / tag).iterdir())
    a = runs['a']
    names = ('fluid', 'boundary', 'obstacle')
    assert sorted(a) == sorted('%s_%s' % (n, f) for n in names for f in ('gid',) + bench.DUMP_FIELDS)
    for k, v in a.items():
        assert v.dtype == np.float64 and v.ndim == 1 and np.all(np.isfinite(v)), k
        assert np.array_equal(v, runs['b'][k]), k
    for n in names:
        g = a[n + '_gid']
        assert 0 < len(g) <= 200 and np.all(np.diff(g) > 0), n
    assert len(a['fluid_gid']) == 200            # the fluid is larger than the sample
    assert not np.array_equal(a['fluid_w'], runs['c']['fluid_w'])


def _rank_main(rank, world, port, so, argv, q):
    """one rank of `torchrun bench.py --gpus N` without GPUs: gloo for nccl, host tensors
    for device tensors, the library emulation for libb200sph.so"""
    import torch
    import torch.distributed as dist
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, 'tests'))
    from pysph_b200 import _lib, parallel
    _lib.LIB_PATH, _lib._lib = so, None
    torch.cuda.Event = _Event
    torch.cuda.synchronize = lambda *a, **k: None
    torch.cuda.set_device = lambda *a, **k: None
    torch.cuda.current_stream = lambda *a, **k: _Stream()
    torch.Tensor.pin_memory = lambda self, *a, **k: self
    real_tensor, real_init = torch.tensor, dist.init_process_group

    def tensor(*a, **k):
        if str(k.get('device', 'cpu')).startswith('cuda'):
            k['device'] = 'cpu'
        return real_tensor(*a, **k)
    torch.tensor = tensor
    dist.init_process_group = lambda backend=None, **k: real_init(
        'gloo', rank=rank, world_size=world)
    init = parallel.DeviceHaloOps.__init__

    def host_init(self, backend, device):
        init(self, backend, 0)
        self.device = torch.device('cpu')

    def read_later(self, t):
        v = float(t[0])
        return lambda: v
    parallel.DeviceHaloOps.__init__ = host_init
    parallel.DeviceHaloOps.read_later = read_later
    os.environ.update(RANK=str(rank), LOCAL_RANK='0', WORLD_SIZE=str(world),  # one emulated device per process
                      MASTER_ADDR='127.0.0.1', MASTER_PORT=str(port))
    sys.argv = ['bench.py', '--gpus', str(world), '--steps', '3', '--warmup', '3',
                '--e2e-steps', '2', '--no-cpu'] + argv
    import tempfile
    tmp = tempfile.TemporaryFile()
    saved = os.dup(1)
    os.dup2(tmp.fileno(), 1)        # what bench prints on fd 1 (it parks fd 1 on stderr itself)
    try:
        bench = importlib.import_module('bench')
        bench.main()
        sys.stdout.flush()
    except BaseException:
        import traceback
        os.dup2(saved, 1)
        q.put((rank, 'error', traceback.format_exc()))
        raise
    os.dup2(saved, 1)
    tmp.seek(0)
    q.put((rank, 'ok', tmp.read().decode()))


@pytest.mark.timeout(400)
@pytest.mark.parametrize('argv', [['--dx', '0.07'],
                                  ['--workload', 'rings', '--dx', '0.0025', '--lz', '0.005']],
                         ids=['dam_break', 'rings'])
def test_bench_two_ranks_on_the_emulated_library(emulated_library, argv):  # noqa: F811
    """`torchrun --nproc-per-node 2 bench.py --gpus 2 ...` on the CPU: rank 0 prints ONE line
    with the whole-job aggregate, the other rank prints nothing."""
    import socket
    import torch.multiprocessing as mp
    from pysph_b200 import _lib
    sock = socket.socket()
    sock.bind(('127.0.0.1', 0))
    port = sock.getsockname()[1]
    sock.close()
    ctx = mp.get_context('spawn')
    q = ctx.Queue()
    procs = [ctx.Process(target=_rank_main, args=(r, 2, port, _lib.LIB_PATH, argv, q))
             for r in range(2)]
    for p in procs:
        p.start()
    out = dict()
    for _ in range(2):
        rank, status, text = q.get(timeout=240)
        assert status == 'ok', text[-3000:]
        out[rank] = text
    for p in procs:
        p.join(timeout=120)
        assert p.exitcode == 0
    lines = [ln for ln in out[0].splitlines() if ln.startswith('{')]
    assert len(lines) == 1 and not [ln for ln in out[1].splitlines() if ln.startswith('{')]
    d = json.loads(lines[0])
    assert d['n_gpus'] == 2 and d['scaling'] == 'weak' and d['value'] > 0
    assert d['e2e']['value'] > 0 and d['e2e']['h2d_bytes_per_step'] > 0
    assert d['gpu_launches'] > 0 and d['roofline']['frac'] > 0
    if argv[0] == '--dx':
        # the slab run inside the bench reproduced one process (by gid), the peer protocol
        # carried the refreshes and pair passes ran their ghost-free CTAs under the halo
        par = d['config']['multi_gpu_parity']
        assert par['ok'] is True and max(par['max_scaled_error'].values()) <= 1e-9, par
        # ... on a problem where pair passes DID run ghost-free CTAs under the halo in flight
        assert par['halo']['overlapped_evaluations'] > 0 and par['halo']['ctas_interior'] > 0 \
            and par['halo']['fused_stages'] > 0, par
        halo = d['config']['halo']
        assert halo['peer_sync'] is True and halo['peer_refreshes'] > 0, halo
        # (slabs this thin have a ghost in every CTA's neighbourhood: the overlap needs
        # ghost-free CTAs, which the bench's own parity problem at dx = 0.03 has)
        assert halo['ctas_boundary'] > 0 and (halo['overlapped_evaluations'] > 0) == \
            (halo['ctas_interior'] > 0), halo
        dev = d['developed']
        assert dev['value'] > 0 and dev['full_builds'] >= 1, dev
        assert d['launches_per_step'] > 0
        # the disturbed-run guard: the keys exist; on a quiet run nothing was taken again
        assert d['host_loop_ms_per_step'] > 0 and 'remeasured' in d
