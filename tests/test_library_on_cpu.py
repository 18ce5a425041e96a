"""The WHOLE library on the CPU (no GPU): pysph_b200/csrc/b200sph.cu -- host C-ABI code and
kernels -- is transformed (tests/cpu_emul/transform.py: kernel launches become emu::launch
calls, nothing else changes), compiled with g++ against a host stand-in for the CUDA runtime and
device intrinsics (tests/cpu_emul/cuda_shim.h: blocks run in order; threads of a block in order,
or lock-stepped -- as fibers, or with B200SPH_EMUL_THREADS=1 as OS threads -- with real __syncthreads / shuffles / ballots / atomics) and loaded
in place of libb200sph.so.  The GPU parity tests of this repository are then run against it.

This is TEST INFRASTRUCTURE: the product never loads this library (pysph_b200/_lib.py knows only
libb200sph.so and raises without it); it exists so that the host logic -- pool layout, list
builds and rebuilds, deferred drift checks, device-resident dt, periodic wrap, EDAC and
elastic-dynamics entry points -- can be exercised where no GPU is available, with the same
tests and tolerances.  It proves nothing about performance or about GPU-specific behaviour
(memory spaces, launch limits, real concurrency).
"""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
EMUL = os.path.join(HERE, 'cpu_emul')
BUILD = os.path.join(EMUL, '_build')
sys.path.insert(0, EMUL)


def _build():
    import transform
    os.makedirs(BUILD, exist_ok=True)
    from pysph_b200 import build as lib_build
    cpp = os.path.join(BUILD, 'b200sph_emul.cpp')
    text, modes = transform.transform(lib_build.read_source())
    assert modes['k_list_build'] == 'emu::BLOCK' and modes['k_pair_list'] == 'emu::WARP' \
        and modes['k_stage'] == 'emu::SEQ' and modes['k_stage_pack'] == 'emu::BLOCK'
    if not os.path.exists(cpp) or open(cpp).read() != text:
        open(cpp, 'w').write(text)
    so = os.path.join(BUILD, 'libb200sph_emul.so')
    deps = [cpp, os.path.join(EMUL, 'cuda_shim.h'), os.path.join(EMUL, 'cuda_shim.cpp'),
            os.path.join(ROOT, 'include', 'b200sph.h')]
    if not os.path.exists(so) or os.path.getmtime(so) < max(os.path.getmtime(d) for d in deps):
        cxx = '/usr/bin/g++' if os.path.exists('/usr/bin/g++') else 'g++'
        subprocess.check_call([cxx, '-O1', '-std=c++17', '-shared', '-fPIC', '-w', '-pthread',
                               '-I', os.path.join(ROOT, 'include'), '-I', EMUL, cpp,
                               os.path.join(EMUL, 'cuda_shim.cpp'), '-o', so])
    return so


_NVRTC_OK, _REAL_COMPILE = set(), []


def host_compile_image(source, name='generated.cu', arch=None):
    """Stands in for pysph_b200.codegen.compile_image (NVRTC) while the emulated library is
    loaded: the SAME generated source, compiled for the host against cuda_shim.h; the "image"
    handed to b200sph_generic_load is the path of the shared object."""
    import hashlib
    tag = hashlib.sha1(source.encode()).hexdigest()[:16]
    cpp = os.path.join(BUILD, 'gen_%s.cpp' % tag)
    so = os.path.join(BUILD, 'gen_%s.so' % tag)
    if tag not in _NVRTC_OK:
        # ... and the real thing must accept the same text: NVRTC needs no GPU to compile
        image = _REAL_COMPILE[0](source)
        assert image[:4] == b'\x7fELF'
        _NVRTC_OK.add(tag)
    if not os.path.exists(so):
        open(cpp, 'w').write('#include "cuda_shim.h"\n#include <cmath>\n' + source)
        cxx = '/usr/bin/g++' if os.path.exists('/usr/bin/g++') else 'g++'
        subprocess.check_call([cxx, '-O1', '-std=c++17', '-shared', '-fPIC', '-w', '-I', EMUL, cpp,
                               '-L', BUILD, '-l:libb200sph_emul.so', '-Wl,-rpath,' + BUILD, '-o', so])
    return so.encode() + b'\0'


@pytest.fixture(scope='module')
def emulated_library():
    """libb200sph_emul.so stands in for libb200sph.so while this module runs."""
    from pysph_b200 import _lib, codegen
    so = _build()
    saved = (_lib.LIB_PATH, _lib._lib, codegen.compile_image)
    _lib.LIB_PATH, _lib._lib = so, None
    if not _REAL_COMPILE:
        _REAL_COMPILE.append(codegen.compile_image)
    codegen.compile_image = host_compile_image
    _lib.load()
    yield 0
    _lib.LIB_PATH, _lib._lib, codegen.compile_image = saved


def test_every_entry_point_is_exported(emulated_library):
    from pysph_b200 import _lib
    lib = _lib.load()
    for name in _lib.SIGNATURES:
        assert hasattr(lib, name), name
    assert lib.b200sph_abi_version() == 5


# ---- the GPU tests of this repository, run against the emulated library --------------------
# (module, test, kwargs).  The default selection takes ~1.5 minutes (lock-stepped lanes are
# fibers, cuda_shim.cpp); the rest runs with B200SPH_EMUL_FULL=1 (another ~2 minutes).
# B200SPH_EMUL_THREADS=1 makes every lane a real OS thread instead (the cross-check: ~5x slower).
FAST = [
    ('test_gpu_parity', 'test_density_1d_fixture', {}),
    ('test_gpu_parity', 'test_nnps_equals_brute_force', {}),
    ('test_gpu_parity', 'test_nnps_corner_cases', {}),
    ('test_gpu_parity', 'test_steppers_and_eos_vs_reference_bodies', {}),
    ('test_gpu_parity', 'test_push_pull_roundtrip_and_errors', {}),
] + [('test_gpu_parity', 'test_wcsph_evaluation_vs_reference_bodies', {'idx': i}) for i in range(6)] + [
    ('test_gpu_parity', 'test_monaghan_av_vs_reference_bodies', {'idx': i}) for i in range(2)] + [
    ('test_gpu_parity', 'test_laminar_viscosity_vs_reference_bodies', {'idx': i}) for i in range(2)] + [
    ('test_gpu_periodic', 'test_periodic_lattice_density', {'dim': d, 'n': n, 'shift': sh})
    for d, n in ((1, 20), (2, 10), (3, 5)) for sh in (0.0, 0.35)
] + [
    ('test_gpu_periodic', 'test_sph_evaluator_periodic_fixture', {}),
    ('test_gpu_periodic', 'test_periodic_errors', {}),
    ('test_gpu_periodic', 'test_periodic_wcsph_steps_vs_oracle', {'dim': 2, 'n': 24, 'pattern': (1, 1, 0)}),
    ('test_gpu_periodic', 'test_periodic_wcsph_steps_vs_oracle', {'dim': 3, 'n': 10, 'pattern': (1, 0, 1)}),
] + [('test_gpu_edac', 'test_edac_evaluation_matches_reference_bodies', {'idx': i}) for i in range(4)] + [
    ('test_gpu_edac', 'test_edac_tvf_step_matches_reference_bodies', {}),
    ('test_gpu_edac', 'test_taylor_green_steps_vs_oracle', {'dim': 2, 'nx': 32, 'kernel': 'QuinticSpline'}),
    ('test_gpu_edac', 'test_edac_setup_errors', {}),
    ('test_gpu_edac', 'test_edac_channel_with_walls_steps_vs_oracle', {}),
    ('test_gpu_edac', 'test_edac_periodic_channel_with_walls_vs_oracle', {}),
    ('test_gpu_edac', 'test_edac_step_matches_reference_bodies', {}),
    ('test_gpu_edac', 'test_edac_external_flow_steps_vs_oracle', {}),
] + [('test_gpu_edac', 'test_edac_external_flow_evaluation_matches_reference_bodies', {'idx': i})
     for i in range(4)] + [
] + [('test_gpu_edac', 'test_edac_solid_wall_evaluation_matches_reference_bodies', {'idx': i})
     for i in range(4)] + [('test_gpu_solid', 'test_elastic_evaluation_matches_reference_bodies', {'idx': i})
     for i in range(6)] + [
    ('test_gpu_solid', 'test_solid_mech_step_matches_reference_bodies', {}),
    ('test_gpu_solid', 'test_rings_steps_vs_oracle', {}),
    ('test_gpu_solid', 'test_rings_3d_steps_vs_oracle', {}),
    ('test_gpu_solid', 'test_bar_hits_rigid_wall_vs_oracle', {}),
    ('test_gpu_solid', 'test_rings_3d_momentum_and_symmetry_at_size',
     {'dx': 0.0025, 'lz': 0.01, 'steps': 6, 'min_particles': 1000}),
    ('test_gpu_parity', 'test_kernels_via_two_particle_density', {}),
    ('test_gpu_parity', 'test_dam_break_3d_small_eval_and_steps', {}),
    ('test_gpu_parity', 'test_dam_break_2d_gate', {}),
    ('test_gpu_parity', 'test_determinism', {}),
    ('test_gpu_parity', 'test_deferred_drift_check_protocol', {}),
    ('test_gpu_parity', 'test_zorder_rows_give_the_same_neighbours_and_fields', {'monkeypatch': None}),
    ('test_gpu_parity', 'test_fused_stage_kernel_is_bitwise_the_separate_kernels', {'monkeypatch': None, 'device_dt': True, 'dx': 0.08}),
    ('test_gpu_parity', 'test_fused_stage_kernel_is_bitwise_the_separate_kernels', {'monkeypatch': None, 'device_dt': False, 'dx': 0.08}),
    ('test_gpu_periodic', 'test_periodic_wcsph_steps_vs_oracle', {'dim': 3, 'n': 10, 'pattern': (1, 1, 1)}),
    ('test_gpu_periodic', 'test_periodic_wcsph_steps_vs_oracle', {'dim': 2, 'n': 24, 'pattern': (0, 1, 0)}),
    ('test_output', 'test_dump_and_restart_on_device', {'tmp_path': None}),
    ('test_gpu_mirror', 'test_mirror_wcsph_steps_vs_oracle', {'dim': 2, 'n': 24, 'pattern': (1, 1, 0)}),
    ('test_gpu_mirror', 'test_mirror_wcsph_steps_vs_oracle', {'dim': 3, 'n': 10, 'pattern': (1, 0, 1)}),
    ('test_gpu_mirror', 'test_mirror_wcsph_steps_vs_oracle', {'dim': 3, 'n': 10, 'pattern': (1, 1, 1)}),
    ('test_gpu_mirror', 'test_mirror_errors', {}),
    ('test_gpu_rings_multi', 'test_elastic_halo_and_migration_layout', {}),
    ('test_gpu_rings_multi', 'test_empty_elastic_array_agrees_on_the_message_layout', {}),
    ('test_gpu_groups', 'test_group_honors_condition', {}),
    ('test_gpu_groups', 'test_iterated_groups', {}),
    ('test_gpu_groups', 'test_pre_post_order', {}),
    ('test_gpu_groups', 'test_start_stop_idx', {'as_str': False}),
    ('test_gpu_groups', 'test_start_stop_idx', {'as_str': True}),
    ('test_gpu_groups', 'test_start_stop_idx_three_arrays', {}),
    ('test_gpu_generic', 'test_simple_equation', {}),
    ('test_gpu_generic', 'test_iterated_generic_groups', {}),
    ('test_gpu_generic', 'test_mixed_type_arrays_and_time', {}),
    ('test_gpu_generic', 'test_generic_group_controls', {}),
    ('test_gpu_generic', 'test_user_property_and_kernel_symbol', {}),
    ('test_gpu_generic', 'test_untranslatable_bodies_fail_at_setup', {}),
    ('test_gpu_generic', 'test_generic_kernel_symbols_vs_reference_kernels', {}),
    ('test_gpu_generic', 'test_host_callbacks_and_helpers', {}),
    ('test_gpu_generic', 'test_mixed_and_aliased_groups', {}),
] + [('test_gpu_generic', 'test_generic_wcsph_group_equals_golden', {'idx': i}) for i in (0, 1, 2, 5)]
FULL = [
    ('test_gpu_parity', 'test_device_resident_dt_is_bitwise_the_host_path', {}),
    ('test_gpu_gate_25k', 'test_dam_break_2d_gate_25k', {}),
]


def _id(t):
    return t[1].replace('test_', '') + ''.join('-%s' % (v,) for v in t[2].values()
                                               if v is not None).replace(' ', '')


def _call(t, emulated_library):
    import torch
    from pysph_b200 import parallel
    mod = __import__(t[0])
    fn = getattr(mod, t[1])
    fn = getattr(fn, '__wrapped__', fn)
    kw = dict(t[2])
    if 'tmp_path' in kw:
        import pathlib
        import tempfile
        kw['tmp_path'] = pathlib.Path(tempfile.mkdtemp())
    init = parallel.DeviceHaloOps.__init__

    def host_init(self, backend, device):
        init(self, backend, 0)
        self.device = torch.device('cpu')
    with pytest.MonkeyPatch.context() as mp:
        # halo buffers in host memory: under the emulation device memory IS host memory, also
        # on a machine where torch sees a GPU
        mp.setattr(parallel.DeviceHaloOps, '__init__', host_init)
        if 'monkeypatch' in kw:
            kw['monkeypatch'] = mp
        return fn(emulated_library, **kw)


@pytest.mark.parametrize('t', FAST, ids=_id)
def test_gpu_test_on_the_emulated_library(emulated_library, t):
    _call(t, emulated_library)


@pytest.mark.skipif(not os.environ.get('B200SPH_EMUL_FULL'),
                    reason='long (minutes each): set B200SPH_EMUL_FULL=1')
@pytest.mark.parametrize('t', FULL, ids=_id)
def test_gpu_test_on_the_emulated_library_full(emulated_library, t):
    _call(t, emulated_library)


@pytest.mark.skipif(not os.environ.get('B200SPH_EMUL_FULL'),
                    reason='long: set B200SPH_EMUL_FULL=1')
def test_pair_kernel_variants_on_the_emulated_library(emulated_library, monkeypatch):
    import test_gpu_parity
    test_gpu_parity.test_all_pair_kernels_agree(emulated_library, monkeypatch)


def _small_dam_break(dx=0.08, vscale=1.0):
    from pysph_b200 import geometry as geo
    pas = geo.dam_break_3d_particles(dx=dx)
    rs = np.random.RandomState(9)
    f = pas[0]
    for k in ('u', 'v', 'w'):
        f.properties[k][:] = rs.normal(scale=vscale, size=f.u.size)
    f.rho[:] *= 1 + 0.01 * rs.uniform(-1, 1, f.u.size)
    return pas, geo.dam_break_3d_params(dx)


def test_small_dam_break_host_logic(emulated_library):
    """What the long tests check, on a 3.5 k-particle dam break: adaptive EPEC steps against
    the oracle (pair counts equal), device-resident dt bitwise == the host path, the deferred
    drift check forces repeats (fast particles use up the skin)."""
    import pysph_b200 as pb
    from helpers import copy_arrays
    from oracle import oracle as orc
    out = {}
    for mode in (True, False):
        pas, params = _small_dam_break(vscale=3.0)
        params = dict(params, n_damp=4)
        if mode:
            opas = copy_arrays(pas)
            o = orc.WCSPHOracleSolver(opas, params, 'CubicSpline', threads=2)
        s = pb.make_wcsph_solver(pas, dict(params), pb.CubicSpline(dim=3), device_dt=mode)
        s.a_eval.count_pairs = True
        s.initialise()
        if mode:
            o.initialise()
            assert s.a_eval.last_pairs == o.pairs_last_eval
        s.a_eval.count_pairs = False
        for _ in range(14):
            s.step()
        for _ in range(4):
            s.step()
        s.pull()
        st = s.backend.stats()
        out[mode] = (s.t, s.dt, dict((k, pas[0].properties[k].copy()) for k in ('x', 'u', 'rho')), st)
        if mode:
            for _ in range(18):
                o.step()
            assert abs(s.t - o.t) <= 1e-5 * o.t
            for k, tol in (('x', 2e-6), ('u', 2e-5), ('rho', 1e-6)):
                want = opas[0].properties[k]
                scale = max(np.max(np.abs(want)), 1.0 if k == 'x' else 1e-12)
                assert np.max(np.abs(pas[0].properties[k] - want)) <= tol * scale, k
    a, b = out[True], out[False]
    assert a[:2] == b[:2]
    for k in a[2]:
        assert np.array_equal(a[2][k], b[2][k]), k
    st = a[3]
    # the skin was used up on the way: either a deferred check failed (evaluation repeated)
    # or the extrapolated drift made the library rebuild one evaluation early
    assert st['light_updates'] > 10 and st['deferred_failed'] + st['proactive_builds'] >= 1 \
        and st['list_builds'] >= 2, st


def test_final_time_small(emulated_library):
    """The last step lands on the final time (solver.py:756-776): dt = tf - t when the next
    step would overshoot, the loop stops within the reference's tolerance; device-resident
    clock (k_dt_commit) == host clock bitwise == the oracle's step count and time."""
    import pysph_b200 as pb
    from helpers import copy_arrays
    from oracle import oracle as orc
    pas, params = _small_dam_break(vscale=0.3)
    params = dict(params, n_damp=3)
    probe = pb.make_wcsph_solver(pas, dict(params), pb.CubicSpline(dim=3))
    for _ in range(5):
        probe.step()
    tf = probe.t + 0.4 * probe.dt             # inside the 6th step
    out = {}
    for mode in (True, False):
        pas, _ = _small_dam_break(vscale=0.3)
        if mode:
            opas = copy_arrays(pas)
            o = orc.WCSPHOracleSolver(opas, dict(params, tf=tf), 'CubicSpline', threads=2)
            o.initialise()
            while (tf - o.t) > np.finfo(float).eps * 2 * tf * max(o.count, 1):
                o.step()
        s = pb.make_wcsph_solver(pas, dict(params), pb.CubicSpline(dim=3), device_dt=mode,
                                 tf=tf)
        s.solve(100)
        s.pull()
        assert s.count == 6 and abs(s.t - tf) <= 4 * np.finfo(float).eps * tf, (s.count, s.t, tf)
        out[mode] = (s.t, s.dt, pas[0].x.copy(), pas[0].u.copy())
        s.solve(100)                           # nothing left to do
        assert s.count == 6
        if mode:
            assert o.count == 6 and abs(o.t - s.t) <= 1e-12 * tf and abs(o.dt - s.dt) <= 1e-5 * o.dt
            assert np.max(np.abs(pas[0].x - opas[0].x)) <= 2e-6
    a, b = out[True], out[False]
    assert a[:2] == b[:2] and np.array_equal(a[2], b[2]) and np.array_equal(a[3], b[3])


def test_deferred_protocol_small(emulated_library):
    """nnps_update_deferred / nnps_confirm on the small case (the GPU version of this check is
    tests/test_gpu_parity.py::test_deferred_drift_check_protocol)."""
    import pysph_b200 as pb
    pas, params = _small_dam_break(vscale=0.5)
    s = pb.make_wcsph_solver(pas, dict(params), pb.CubicSpline(dim=3))
    s.initialise()
    be, nn, ae = s.backend, s.nnps, s.a_eval
    f = pas[0]
    f.x[:] += 1e-4 * params['h0']
    be.push(0, ['x'])
    nn.update(deferred=True)
    ae.compute(0.0, 0.0)
    assert nn.confirm() is False
    rs = np.random.RandomState(1)
    f.x[:] += params['h0'] * rs.uniform(-1, 1, f.x.size)
    be.push(0, ['x'])
    nn.update(deferred=True)
    ae.compute(0.0, 0.0)
    assert nn.confirm() is True and nn.confirm() is False
    nn.update()
    ae.compute(0.0, 0.0)
    f.x[:] += params['h0'] * rs.uniform(-1, 1, f.x.size)
    be.push(0, ['x'])
    nn.update(deferred=True)
    ae.compute(0.0, 0.0)
    with pytest.raises(RuntimeError, match='never confirmed'):
        be.pull(0, ['au'])
    assert be.stats()['deferred_failed'] == 2


def test_dump_and_restart_small(emulated_library, tmp_path):
    """Solver.dump_output / load_output on the small case (GPU version:
    tests/test_output.py::test_dump_and_restart_on_device).  A restart re-runs
    initial_acceleration (solver.py:454), whose TaitEOSHGCorrection clamps the solids'
    density IN PLACE (wc/basic.py:119-120): like in the reference, a restarted run is therefore
    not bitwise the uninterrupted one -- it is compared with the oracle restarted the same way."""
    import pysph_b200 as pb
    from helpers import copy_arrays
    from oracle import oracle as orc
    from pysph_b200 import output
    pas, params = _small_dam_break(vscale=0.2)
    params = dict(params, n_damp=8)          # the dump falls INTO the damping window
    s = pb.make_wcsph_solver(pas, dict(params), pb.CubicSpline(dim=3))
    for _ in range(6):
        s.step()
    f = s.dump_output(str(tmp_path), 'db')
    data = output.load(f)
    assert int(data['solver_data']['count']) == 6 and float(data['solver_data']['t']) == s.t
    t6, dt6 = s.t, float(data['solver_data']['dt'])
    # the file holds the undamped dt (solver.py:747-753)
    assert abs(dt6 - s.dt / s._damping_factor) <= 1e-15 * dt6 and 0.9 < s._damping_factor < 1.0
    # the restarted run ...
    pas2, _ = _small_dam_break(vscale=0.2)
    s2 = pb.make_wcsph_solver(pas2, dict(params), pb.CubicSpline(dim=3))
    s2.load_output(f)
    assert (s2.count, s2.t, s2.dt) == (6, t6, dt6)
    # ... and the oracle, started from the same file the same way
    opas = [data['arrays'][pa.name] for pa in pas]
    for q, pa in zip(opas, pas):                 # the oracle wants every WCSPH property
        for k in pa.properties:
            if k not in q.properties:
                q.add_property(k)
    o = orc.WCSPHOracleSolver(opas, dict(params), 'CubicSpline', threads=2)
    o.t, o.dt, o.count = t6, dt6, 6
    o.initialise()
    s2.initialise()
    assert abs(s2.dt - o.dt) <= 1e-6 * o.dt
    for _ in range(4):
        s2.step()
        o.step()
    s2.pull()
    assert s2.count == 10 and abs(s2.t - o.t) <= 1e-6 * o.t
    for a, b in zip(pas2, opas):
        for k, tol in (('x', 2e-6), ('y', 2e-6), ('z', 2e-6), ('u', 2e-5), ('v', 2e-5),
                       ('w', 2e-5), ('rho', 1e-6)):
            scale = max(np.max(np.abs(b.properties[k])), 1.0 if k in 'xyz' else 1e-3)
            assert np.max(np.abs(a.properties[k] - b.properties[k])) <= tol * scale, (a.name, k)


def test_async_output_small(emulated_library, tmp_path):
    """solve(pfreq=...) with asynchronous dumps (b200sph_snapshot_take / fetch / release +
    the writer thread) writes the same files as synchronous dumps, for the device-resident
    and the host-side time step; a file written asynchronously restarts."""
    import pysph_b200 as pb
    from pysph_b200 import output
    files = {}
    for mode, asyn, device_dt in (('async', True, True), ('sync', False, True),
                                  ('async_host_dt', True, False)):
        pas, params = _small_dam_break(vscale=0.5)
        s = pb.make_wcsph_solver(pas, dict(params, n_damp=5), pb.CubicSpline(dim=3),
                                 device_dt=device_dt)
        d = tmp_path / mode
        s.solve(7, pfreq=3, output_directory=str(d), fname='db', asynchronous=asyn,
                detailed_output=(mode != 'async_host_dt'))
        assert sorted(os.listdir(str(d))) == ['db_00000.npz', 'db_00003.npz', 'db_00006.npz',
                                              'db_00007.npz']
        files[mode] = dict((f, output.load(str(d / f))) for f in os.listdir(str(d)))
        assert s.count == 7
    for f, want in files['sync'].items():
        for mode in ('async', 'async_host_dt'):
            got = files[mode][f]
            for k in ('t', 'dt', 'count'):
                assert float(got['solver_data'][k]) == float(want['solver_data'][k]), (f, k)
            for name, pa in want['arrays'].items():
                q = got['arrays'][name]
                assert q.get_number_of_particles() == pa.get_number_of_particles()
                props = q.output_property_arrays if mode == 'async_host_dt' else pa.properties
                assert len(props) > 10
                for k in props:
                    assert q.properties[k].dtype == pa.properties[k].dtype, (f, name, k)
                    assert np.array_equal(q.properties[k], pa.properties[k]), (f, name, k)
    # something moved between the dumps, and integer properties came through
    a, b = files['async']['db_00003.npz'], files['async']['db_00006.npz']
    assert np.max(np.abs(a['arrays']['fluid'].x - b['arrays']['fluid'].x)) > 0
    assert np.array_equal(a['arrays']['fluid'].gid, b['arrays']['fluid'].gid)
    assert a['arrays']['fluid'].gid.dtype == np.uint32 and len(set(a['arrays']['fluid'].gid)) > 100
    # misuse: a second snapshot while one is open
    pas, params = _small_dam_break()
    s = pb.make_wcsph_solver(pas, dict(params), pb.CubicSpline(dim=3))
    s.initialise()
    import ctypes as C
    args = (1, (C.c_int * 1)(0), (C.c_int * 1)(0), (C.c_int64 * 1)(10))
    s.backend.ctx.call('b200sph_snapshot_take', *args)
    with pytest.raises(Exception, match='not released'):
        s.backend.ctx.call('b200sph_snapshot_take', *args)
    buf = np.empty(10)
    with pytest.raises(Exception, match='does not hold'):
        s.backend.ctx.call('b200sph_snapshot_fetch', 0, buf.ctypes.data, 11)
    s.backend.ctx.call('b200sph_snapshot_fetch', 0, buf.ctypes.data, 10)
    s.pull()
    assert np.array_equal(buf, pas[0].x[:10])
    s.backend.ctx.call('b200sph_snapshot_release')


# ---- the slab decomposition: real halo / migration kernels of the (emulated) library, the
#      real SlabParallelManager, gloo instead of NCCL, host tensors as "device" buffers ---------
def test_column_counts_on_the_emulated_library(emulated_library):
    """b200sph_column_counts (the slab re-cut's histogram) against numpy: clamped end
    bins, real particles only, run-merged atomics."""
    import pysph_b200 as pb
    rs = np.random.RandomState(3)
    x = np.sort(rs.uniform(-0.2, 3.4, 5001))
    pa = pb.get_particle_array_wcsph(name='fluid', x=x, y=x * 0, z=x * 0, h=0.1, m=1.0, rho=1.0)
    pb2 = pb.get_particle_array_wcsph(name='wall', x=rs.uniform(-0.2, 3.4, 777), h=0.1, m=1.0,
                                      rho=1.0)
    pb2.set_num_real_particles(700)              # 77 ghosts at the end: not counted
    pb2.tag[700:] = 1
    be = pb.B200Backend([pa, pb2])
    for arr, p, n in ((0, pa, 5001), (1, pb2, 700)):
        cnt = np.zeros(64, dtype=np.uint64)
        be.ctx.call('b200sph_column_counts', arr, 0.0, 1.0 / 0.05, 64, cnt.ctypes.data)
        b = np.clip(np.floor(p.x[:n] / 0.05).astype(int), 0, 63)
        assert np.array_equal(cnt.astype(np.int64), np.bincount(b, minlength=64)), arr
        assert cnt.sum() == n


SLAB_DX, SLAB_STEPS = 0.07, 8


def _slab_worker(rank, world, port, so, q, lb_freq=0):
    import torch
    import torch.distributed as dist
    from pysph_b200 import _lib
    _lib.LIB_PATH, _lib._lib = so, None
    import pysph_b200 as pb
    from pysph_b200 import geometry as geo, parallel
    import test_gpu_multi as M

    Base = parallel.DeviceHaloOps

    class HostHaloOps(Base):
        """DeviceHaloOps with CPU tensors: under the emulation device memory IS host memory"""

        def __init__(self, backend, device):
            Base.__init__(self, backend, 0)
            self.device = torch.device('cpu')

        def read_later(self, tensor):
            v = float(tensor[0])
            return lambda: v
    parallel.DeviceHaloOps = HostHaloOps
    os.environ['MASTER_ADDR'] = '127.0.0.1'
    os.environ['MASTER_PORT'] = str(port)
    # lb_freq runs take the send / recv refresh, the others the peer-memory refresh (the shim
    # emulates cudaIpc with shared memory between the worker processes)
    os.environ['B200SPH_PEER_HALO'] = '0' if lb_freq else '1'
    dist.init_process_group('gloo', rank=rank, world_size=world)
    try:
        params = geo.dam_break_3d_params(SLAB_DX)
        solver, pm, pas = parallel.make_slab_solver(SLAB_DX, params, pb.CubicSpline(dim=3),
                                                    rank, world, device=0, n_damp=0,
                                                    lb_freq=lb_freq)
        if lb_freq:         # the planes were balanced with solids at 0.45: re-cut with the
            pm.lb_weights = [1.0] + [0.1] * (len(pas) - 1)     # reference's 0.1 moves them
        M._perturb(pas)
        solver.backend.push_all()
        for _ in range(SLAB_STEPS):
            solver.step()
        t, dt = solver.t, solver.dt
        solver.pull()
        q.put((rank, M._collect(pas), pm.n_full, pm.n_refresh, pm.n_deferred_failed, t, dt,
               pm.use_peer, pm.n_recut, list(pm.cuts), pm.n_peer_refresh))
    except Exception:
        import traceback
        q.put(('error', rank, traceback.format_exc()))
        raise
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize('world,lb_freq', [
    (3, 0), (3, 2),
    pytest.param(2, 0, marks=pytest.mark.skipif(not os.environ.get('B200SPH_EMUL_FULL'),
                                                reason='set B200SPH_EMUL_FULL=1'))])
def test_slab_decomposition_on_the_emulated_library(emulated_library, world, lb_freq):
    """tests/test_gpu_multi.py without GPUs: x-slabs with ADAPTIVE dt (device-resident dt +
    all-reduce MIN on the time-control block), deferred refresh / confirm, full path with
    migration; world 3 has a rank with two neighbours.  Matches the one-process run by gid."""
    import socket
    import torch.multiprocessing as mp
    import pysph_b200 as pb
    from pysph_b200 import geometry as geo, _lib, parallel
    import test_gpu_multi as M
    params = geo.dam_break_3d_params(SLAB_DX)
    pas = geo.dam_break_3d_particles(dx=SLAB_DX)
    M._perturb(pas)
    s = pb.make_wcsph_solver(pas, dict(params, n_damp=0), pb.CubicSpline(dim=3))
    for _ in range(SLAB_STEPS):
        s.step()
    t_ref, dt_ref = s.t, s.dt
    s.pull()
    ref = M._collect(pas)
    sock = socket.socket()
    sock.bind(('127.0.0.1', 0))
    port = sock.getsockname()[1]
    sock.close()
    ctx = mp.get_context('spawn')
    q = ctx.Queue()
    procs = [ctx.Process(target=_slab_worker, args=(r, world, port, _lib.LIB_PATH, q, lb_freq))
             for r in range(world)]
    for p in procs:
        p.start()
    out = [q.get(timeout=900) for _ in range(world)]
    assert not any(o[0] == 'error' for o in out), [o[2] for o in out if o[0] == 'error'][:1]
    for p in procs:
        p.join(timeout=120)
        assert p.exitcode == 0
    assert min(o[3] for o in out) > 0 and min(o[2] for o in out) >= 1      # refreshes and full paths
    if lb_freq:         # refresh through send / recv (B200SPH_PEER_HALO=0)
        assert not any(o[7] for o in out) and not any(o[10] for o in out)
    elif any(o[7] for o in out):   # refresh through the neighbours' staging buffers ("NVLink stores")
        assert all(o[7] for o in out) and min(o[10] for o in out) > 0
    else:               # shared mappings unavailable in this sandbox: the manager fell back, collectively
        assert not any(o[10] for o in out)
    if lb_freq:         # the slabs were re-cut on the way (k_column_counts + migration)
        static = parallel.balanced_cuts(*parallel.dam_break_column_weights(
            SLAB_DX, solid_weight=0.45), world, SLAB_DX)
        assert all(o[8] >= 1 for o in out) and all(o[9] == out[0][9] for o in out)
        assert out[0][9] != static, (out[0][9], static)
    for o in out:
        assert abs(o[5] - t_ref) <= 1e-6 * t_ref and abs(o[6] - dt_ref) <= 1e-5 * dt_ref
    h0, c0 = params['h0'], params['c0']
    for name in ref:
        g_all = np.concatenate([o[1][name]['gid'] for o in out])
        assert np.array_equal(np.sort(g_all), np.sort(ref[name]['gid'])), name
        order_ref, order = np.argsort(ref[name]['gid']), np.argsort(g_all)
        for k, tol in (('x', 5e-6 * h0), ('y', 5e-6 * h0), ('z', 5e-6 * h0), ('u', 5e-6 * c0),
                       ('v', 5e-6 * c0), ('w', 5e-6 * c0), ('rho', 5e-4)):
            a = np.concatenate([o[1][name][k] for o in out])[order]
            assert np.max(np.abs(a - ref[name][k][order_ref])) <= tol, (name, k)


@pytest.mark.parametrize('name', ['test_halo_pack_append_overwrite_migrate',
                                  'test_evaluation_with_ghosts_equals_one_array'])
def test_halo_entry_points_on_the_emulated_library(emulated_library, monkeypatch, name):
    """tests/test_gpu_halo.py (pack / append / overwrite / migrate through the C-ABI, and an
    evaluation with imported ghosts) with the buffers in host memory -- under the emulation
    device memory IS host memory; the product's DeviceHaloOps knows only CUDA tensors."""
    import torch
    import test_gpu_halo
    from pysph_b200 import parallel
    init = parallel.DeviceHaloOps.__init__

    def host_init(self, backend, device):
        init(self, backend, 0)
        self.device = torch.device('cpu')
    monkeypatch.setattr(parallel.DeviceHaloOps, '__init__', host_init)
    getattr(test_gpu_halo, name)(emulated_library)


RINGS = dict(dx=0.0025, lz=0.0075, dt=2e-7, steps=10, u_f=0.25)
RING_FIELDS = ('x', 'y', 'z', 'u', 'v', 'w', 'rho', 's00', 's01', 's02', 's11', 's12', 's22')


def _rings_perturb(pa):
    """pressure and shear everywhere (not only at the contact), the same function of
    position whatever the decomposition"""
    pa.rho[:] *= 1.0 + 0.01 * np.sin(300.0 * pa.x + 170.0 * pa.y + 90.0 * pa.z)
    pa.v[:] += 0.02 * pa.cs * np.sin(250.0 * pa.x)
    pa.w[:] += 0.02 * pa.cs * np.cos(200.0 * pa.y)


def _rings_collect(pa):
    nr = pa.get_number_of_particles(real=True)
    return dict((k, pa.properties[k][:nr].copy()) for k in ('gid',) + RING_FIELDS)


def _rings_worker(rank, world, port, so, q):
    import torch
    import torch.distributed as dist
    from pysph_b200 import _lib
    _lib.LIB_PATH, _lib._lib = so, None
    from pysph_b200 import parallel

    Base = parallel.DeviceHaloOps

    class HostHaloOps(Base):
        def __init__(self, backend, device):
            Base.__init__(self, backend, 0)
            self.device = torch.device('cpu')

        def read_later(self, tensor):
            v = float(tensor[0])
            return lambda: v
    parallel.DeviceHaloOps = HostHaloOps
    os.environ['MASTER_ADDR'] = '127.0.0.1'
    os.environ['MASTER_PORT'] = str(port)
    dist.init_process_group('gloo', rank=rank, world_size=world)
    try:
        solver, pm, pas = parallel.make_rings_slab_solver(
            RINGS['dx'], RINGS['lz'], rank, world, dt=RINGS['dt'],
            geometry_kw=dict(u_f=RINGS['u_f']))
        assert pm.ops.halo_nf == 16 and pm.ops.migrate_nf == 30
        _rings_perturb(pas[0])
        solver.backend.push_all()
        n0 = pas[0].get_number_of_particles()
        for _ in range(RINGS['steps']):
            solver.step()
        solver.pull()
        q.put((rank, _rings_collect(pas[0]), pm.n_full, pm.n_refresh, n0,
               pas[0].get_number_of_particles(real=True), pm.use_peer, pm.n_peer_refresh))
    except Exception:
        import traceback
        q.put(('error', rank, traceback.format_exc()))
        raise
    finally:
        dist.destroy_process_group()


def test_rings_slab_decomposition_on_the_emulated_library(emulated_library):
    """BASELINE configs[4] across ranks, without GPUs: the 3-D colliding rings cut into 3
    x-slabs (the ghost message carries the deviatoric stress, migration the stress and its
    stage copy, group 1 runs on a two-support halo) against the one-process run, by gid.
    The rings move fast enough (u_f = 0.25) that lists are rebuilt, particles migrate
    and the bodies are in contact within the 10 steps."""
    import socket
    import torch.multiprocessing as mp
    import pysph_b200 as pb
    from pysph_b200 import geometry as geo, _lib
    world = 3
    pa = geo.rings_3d_particles(dx=RINGS['dx'], lz=RINGS['lz'], u_f=RINGS['u_f'])
    _rings_perturb(pa)
    s = pb.make_elastic_solver([pa], pb.ElasticSolidsScheme(['solid'], [], dim=3),
                               pb.CubicSpline(dim=3), dt=RINGS['dt'])
    for _ in range(RINGS['steps']):
        s.step()
    s.pull()
    ref = _rings_collect(pa)
    assert np.max(np.abs(ref['s00'])) > 1.0
    sock = socket.socket()
    sock.bind(('127.0.0.1', 0))
    port = sock.getsockname()[1]
    sock.close()
    ctx = mp.get_context('spawn')
    q = ctx.Queue()
    procs = [ctx.Process(target=_rings_worker, args=(r, world, port, _lib.LIB_PATH, q))
             for r in range(world)]
    for p in procs:
        p.start()
    out = [q.get(timeout=900) for _ in range(world)]
    assert not any(o[0] == 'error' for o in out), [o[2] for o in out if o[0] == 'error'][:1]
    for p in procs:
        p.join(timeout=120)
        assert p.exitcode == 0
    assert min(o[2] for o in out) >= 2                  # full paths (rebuild + migration)
    assert any(o[4] != o[5] for o in out)               # somebody gained / lost particles
    # refreshes went through the neighbours' staging buffers (k_halo_gather_all / scatter_all<16>)
    # (if shared mappings are unavailable in this sandbox the manager falls back, collectively)
    if any(o[6] for o in out):
        assert all(o[6] for o in out) and min(o[7] for o in out) > 0, [(o[6], o[7]) for o in out]
    g_all = np.concatenate([o[1]['gid'] for o in out])
    assert np.array_equal(np.sort(g_all), np.sort(ref['gid']))
    order_ref, order = np.argsort(ref['gid']), np.argsort(g_all)
    c0 = pa.cs[0]
    smax = np.max(np.abs(ref['s00']))
    tols = dict(x=1e-7 * 0.08, y=1e-7 * 0.08, z=1e-7 * 0.08, u=2e-6 * c0, v=2e-6 * c0,
                w=2e-6 * c0, rho=5e-6)
    for k in RING_FIELDS:
        a = np.concatenate([o[1][k] for o in out])[order]
        tol = tols.get(k, 2e-4 * smax)
        assert np.max(np.abs(a - ref[k][order_ref])) <= tol, (k, np.max(np.abs(a - ref[k][order_ref])), tol)


def test_solver_configuration_surface(emulated_library, tmp_path):
    """The reference Solver's set_* / add_*_callback methods (solver.py:231-384) drive the
    same loop: callbacks see the solver before / after every step (t not yet advanced in the
    post-step callback, solver.py:480-487), a post-stage callback moves the clock to the
    host, solve() without arguments uses what was configured."""
    import pysph_b200 as pb
    from pysph_b200 import output
    seen = {'pre': [], 'post': [], 'stage': []}
    pas, params = _small_dam_break(vscale=0.3)
    s = pb.make_wcsph_solver(pas, dict(params, n_damp=2), pb.CubicSpline(dim=3))
    s.add_pre_step_callback(lambda sv: seen['pre'].append((sv.count, sv.t, sv.dt)))
    s.add_post_step_callback(lambda sv: seen['post'].append((sv.count, sv.t, sv.dt)))
    s.set_max_steps(4)
    s.set_print_freq(2)
    s.set_output_directory(str(tmp_path))
    s.set_output_fname('cfg')
    s.set_output_printing_level(True)
    s.set_arrays_to_print(['fluid'])
    with pytest.raises(RuntimeError, match='not availabe'):
        s.set_arrays_to_print(['nope'])
    s.solve()
    assert s.count == 4 and s.integrator.device_dt
    assert sorted(os.listdir(str(tmp_path))) == ['cfg_%05d.npz' % k for k in (0, 2, 4)]
    assert 'au' in output.load(str(tmp_path / 'cfg_00004.npz'))['arrays']['fluid'].properties
    assert [c for c, _, _ in seen['pre']] == [0, 1, 2, 3] == [c for c, _, _ in seen['post']]
    for (c0, t0, d0), (c1, t1, d1) in zip(seen['pre'], seen['post']):
        assert (t0, d0) == (t1, d1)                      # t advances after the callbacks
    ts = [t for _, t, _ in seen['pre']] + [s.t]
    for k in range(4):
        assert abs(ts[k] + seen['pre'][k][2] - ts[k + 1]) <= 1e-15
    # the same run with a post-stage callback: host clock, same trajectory
    pas2, _ = _small_dam_break(vscale=0.3)
    s2 = pb.make_wcsph_solver(pas2, dict(params, n_damp=2), pb.CubicSpline(dim=3))
    s2.add_post_stage_callback(lambda t, dt, stage: seen['stage'].append((t, dt, stage)))
    s2.set_final_time(1e9)
    s2.solve(4)
    assert not s2.integrator.device_dt and (s2.t, s2.dt) == (s.t, s.dt)
    assert [st for _, _, st in seen['stage']] == [1, 2] * 4
    s.pull()
    s2.pull()
    assert np.array_equal(pas[0].x, pas2[0].x)
    assert not os.path.exists(str(tmp_path / 'b200_00000.npz'))      # s2 wrote nothing


def test_output_at_times_small(emulated_library, tmp_path):
    """set_output_at_times (solver.py:706-742): a step is cut so that it lands on each
    requested time, a file is written there, and the time step resumes from the uncut one."""
    import pysph_b200 as pb
    from pysph_b200 import output
    pas, params = _small_dam_break(vscale=0.3)
    probe = pb.make_wcsph_solver(pas, dict(params, n_damp=0), pb.CubicSpline(dim=3))
    for _ in range(8):
        probe.step()
    dt_typ = probe.dt
    times = [2.5 * dt_typ, 4.2 * dt_typ]
    log = []
    pas, _ = _small_dam_break(vscale=0.3)
    s = pb.make_wcsph_solver(pas, dict(params, n_damp=0), pb.CubicSpline(dim=3),
                             tf=6.1 * dt_typ)
    s.set_output_at_times(times)
    s.set_output_directory(str(tmp_path))
    s.set_print_freq(1000)
    s.add_pre_step_callback(lambda sv: log.append((sv.count, sv.t, sv.dt)))
    s.solve(asynchronous=False)
    assert not s.integrator.device_dt                      # host clock
    ts = [t for _, t, _ in log] + [s.t]
    eps = 4 * np.finfo(float).eps * s.tf * s.count
    for want in times + [s.tf]:
        assert min(abs(t - want) for t in ts) <= eps, (want, ts)
    # a cut step is shorter than its neighbours, the one after it is a full step again
    dts = [d for _, _, d in log]
    cut = [k for k in range(len(ts) - 1) if any(abs(ts[k + 1] - w) <= eps for w in times)]
    assert len(cut) == 2
    for k in cut:
        assert dts[k] < 0.9 * dts[k - 1] and dts[k + 1] > 0.9 * dts[k - 1]
    files = sorted(os.listdir(str(tmp_path)))
    assert len(files) == 4                                 # initial, two output times, final
    got = sorted(float(output.load(str(tmp_path / f))['solver_data']['t']) for f in files)
    for want, t in zip([0.0] + times + [s.tf], got):
        assert abs(t - want) <= eps
    # the file at an output time holds the UNCUT dt (solver.py:747-750)
    d1 = output.load(str(tmp_path / files[1]))['solver_data']
    assert abs(float(d1['dt']) - dts[cut[0] - 1]) <= 0.2 * dts[cut[0] - 1]


@pytest.mark.parametrize('empty', ['obstacle', 'fluid', 'boundary'])
def test_empty_arrays_small(emulated_library, empty):
    """Ragged inputs: a whole particle array with zero particles (as a source only, as the
    only fluid, as the only wall) goes through NNPS, evaluation, EPEC steps and the adaptive
    time step like in the oracle."""
    import pysph_b200 as pb
    from helpers import copy_arrays
    from oracle import oracle as orc
    pas, params = _small_dam_break(vscale=0.5)
    keep = []
    for pa in pas:
        if pa.name == empty:
            pa = pb.get_particle_array_wcsph(name=pa.name, x=np.zeros(0))
        keep.append(pa)
    pas = keep
    assert [pa.name for pa in pas] == ['fluid', 'boundary', 'obstacle']
    opas = copy_arrays(pas)
    params = dict(params, n_damp=2)
    s = pb.make_wcsph_solver(pas, dict(params), pb.CubicSpline(dim=3))
    o = orc.WCSPHOracleSolver(opas, params, 'CubicSpline', threads=2)
    s.a_eval.count_pairs = True
    s.initialise()
    o.initialise()
    assert s.a_eval.last_pairs == o.pairs_last_eval
    for _ in range(5):
        s.step()
        o.step()
    s.pull()
    assert abs(s.t - o.t) <= 1e-6 * o.t
    for a, b in zip(pas, opas):
        assert a.get_number_of_particles() == b.get_number_of_particles()
        for k, tol in (('x', 2e-6), ('u', 2e-5), ('rho', 1e-6), ('au', 1e-4), ('arho', 1e-4)):
            want = b.properties[k]
            if want.size:
                scale = max(np.max(np.abs(want)), 1.0 if k == 'x' else 1e-3)
                assert np.max(np.abs(a.properties[k] - want)) <= tol * scale, (a.name, k)
