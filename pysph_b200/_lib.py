"""ctypes binding of libb200sph.so (the C-ABI declared in include/b200sph.h).

Loading fails loudly if the shared library is missing -- there is no CPU or
PyTorch fallback for any entry point.
"""
import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, 'libb200sph.so')

MAX_ARRAYS = 8

# property ids (include/b200sph.h)
PROP_IDS = {}
for _i, _n in enumerate(['x', 'y', 'z', 'u', 'v', 'w', 'rho', 'h', 'm',
                         'x0', 'y0', 'z0', 'u0', 'v0', 'w0', 'rho0',
                         'p', 'cs', 'arho', 'au', 'av', 'aw', 'ax', 'ay', 'az',
                         'dt_cfl', 'dt_force']):
    PROP_IDS[_n] = _i
# transport-velocity / EDAC extension (B200SPH_UHAT ...)
PROP_IDS.update(uhat=27, vhat=28, what=29, V=32, pavg=33, auhat=34, avhat=35,
                awhat=36, ap=37)
# arrays of the EDAC scheme (they own 'ap') integrate p: it lives in the fp64
# B200SPH_PF / B200SPH_PF0 instead of the derived fp32 B200SPH_P
EDAC_PROP_IDS = dict(PROP_IDS, p=30, p0=31)
# a solid wall of the EDAC scheme (wc/edac.py:752-753): what the wall equations compute is
# kept in the transport-velocity slots a wall does not otherwise use (include/b200sph.h)
EDAC_WALL_PROP_IDS = dict(PROP_IDS)
EDAC_WALL_PROP_IDS.update(ug=27, vg=28, wg=29, V=32, wij=33, uf=34, vf=35, wf=36)
for _n in ('uhat', 'vhat', 'what', 'pavg', 'auhat', 'avhat', 'awhat', 'ap'):
    EDAC_WALL_PROP_IDS.pop(_n, None)
# elastic-dynamics extension (B200SPH_S00 ...); arrays that own 's00' use these
_SYM = ('00', '01', '02', '11', '12', '22')
ELASTIC_PROP_IDS = dict(PROP_IDS)
ELASTIC_PROP_IDS.update(('s' + k, 70 + i) for i, k in enumerate(_SYM))
ELASTIC_PROP_IDS.update(('s' + k + '0', 76 + i) for i, k in enumerate(_SYM))
ELASTIC_PROP_IDS.update(('v%d%d' % (i, j), 82 + 3 * i + j) for i in range(3) for j in range(3))
ELASTIC_PROP_IDS.update(('r' + k, 91 + i) for i, k in enumerate(_SYM))
ELASTIC_PROP_IDS.update(('as' + k, 97 + i) for i, k in enumerate(_SYM))
INT_PROP_IDS = {'gid': 64, 'tag': 65, 'pid': 66}
USER_PROP0, MAX_USER_PROPS = 110, 16     # B200SPH_USER0, B200SPH_MAX_USER
F64_DEVICE_PROPS = ('x', 'y', 'z', 'u', 'v', 'w', 'rho', 'h', 'm',
                    'x0', 'y0', 'z0', 'u0', 'v0', 'w0', 'rho0')

EQ_SUMMATION_DENSITY = 1
EQ_CONTINUITY = 2
EQ_MOMENTUM = 4
EQ_XSPH = 8
EQ_MONAGHAN_AV = 16
EQ_LAMINAR = 32

HALO_FIELDS = 9
MIGRATE_FIELDS = 17
HALO_FIELD_NAMES = ('x', 'y', 'z', 'u', 'v', 'w', 'rho', 'h', 'm')


class PairProgram(C.Structure):
    _fields_ = [('eqmask', (C.c_uint32 * MAX_ARRAYS) * MAX_ARRAYS),
                ('real_only', C.c_int32),
                ('tensile_correction', C.c_int32),
                ('c0', C.c_double), ('alpha', C.c_double), ('beta', C.c_double),
                ('gx', C.c_double), ('gy', C.c_double), ('gz', C.c_double),
                ('eps_xsph', C.c_double), ('nu', C.c_double), ('eta', C.c_double)]


TVF_PGRAD, TVF_AV, TVF_VISC, TVF_ASTRESS, TVF_EDAC, TVF_NOSLIP = 1, 2, 4, 8, 16, 32
TVF_MOM, TVF_XSPH = 64, 128


class TvfProgram(C.Structure):
    _fields_ = [('fluid_mask', C.c_uint32), ('bql', C.c_int32),
                ('eqbits', C.c_uint32), ('passes', C.c_int32),
                ('pb', C.c_double), ('nu', C.c_double), ('edac_nu', C.c_double),
                ('c0', C.c_double), ('rho0', C.c_double), ('alpha', C.c_double),
                ('gx', C.c_double), ('gy', C.c_double), ('gz', C.c_double),
                ('tdamp', C.c_double), ('t', C.c_double), ('solid_mask', C.c_uint32),
                ('clamp_p', C.c_int32), ('eps_xsph', C.c_double)]


class SolidProgram(C.Structure):
    _fields_ = [('elastic_mask', C.c_uint32), ('grad3d', C.c_int32),
                ('passes', C.c_int32), ('ghost_group1', C.c_int32),
                ('eps', C.c_double), ('alpha', C.c_double), ('beta', C.c_double),
                ('eps_xsph', C.c_double),
                ('c0_ref', C.c_double * MAX_ARRAYS), ('rho_ref', C.c_double * MAX_ARRAYS),
                ('wdeltap', C.c_double * MAX_ARRAYS), ('n', C.c_double * MAX_ARRAYS),
                ('G', C.c_double * MAX_ARRAYS),
                ('source_mask', C.c_uint32), ('reserved', C.c_uint32)]


class GridInfo(C.Structure):
    _fields_ = [('cell_size', C.c_double), ('hmin', C.c_double),
                ('xmin', C.c_double * 3), ('xmax', C.c_double * 3),
                ('ncells', C.c_int32 * 3), ('n_cells', C.c_int64),
                ('n_particles', C.c_int64)]


class Stats(C.Structure):
    _fields_ = [('ms_nnps', C.c_double), ('ms_pair', C.c_double),
                ('ms_other', C.c_double), ('pair_launches', C.c_int64),
                ('kernel_launches', C.c_int64), ('pairs', C.c_int64),
                ('full_builds', C.c_int64), ('light_updates', C.c_int64),
                ('list_builds', C.c_int64),
                ('list_entries_per_particle', C.c_int64),
                ('deferred_failed', C.c_int64), ('fused_stages', C.c_int64),
                ('overlapped', C.c_int64), ('proactive_builds', C.c_int64),
                ('chunks_interior', C.c_int64),
                ('chunks_boundary', C.c_int64), ('ms_halo_chain', C.c_double),
                ('ms_pair_wall', C.c_double), ('ms_halo_sent', C.c_double),
                ('ms_halo_reduced', C.c_double)]


_ctx_p = C.c_void_p
_i64 = C.c_int64
_dp = C.POINTER(C.c_double)
_up = C.POINTER(C.c_uint32)

# name -> (restype, argtypes); must list every function of include/b200sph.h
SIGNATURES = {
    'b200sph_abi_version': (C.c_int, []),
    'b200sph_create': (C.c_int, [C.c_int, C.POINTER(_ctx_p)]),
    'b200sph_destroy': (C.c_int, [_ctx_p]),
    'b200sph_last_error': (C.c_char_p, [_ctx_p]),
    'b200sph_set_stream': (C.c_int, [_ctx_p, C.c_void_p]),
    'b200sph_synchronize': (C.c_int, [_ctx_p]),
    'b200sph_add_array': (C.c_int, [_ctx_p, C.c_char_p, _i64, _i64, _i64]),
    'b200sph_resize_array': (C.c_int, [_ctx_p, C.c_int, _i64, _i64]),
    'b200sph_get_array_size': (C.c_int, [_ctx_p, C.c_int, C.POINTER(_i64),
                                         C.POINTER(_i64)]),
    'b200sph_push_f64': (C.c_int, [_ctx_p, C.c_int, C.c_int, C.c_void_p, _i64, _i64]),
    'b200sph_pull_f64': (C.c_int, [_ctx_p, C.c_int, C.c_int, C.c_void_p, _i64, _i64]),
    'b200sph_push_u32': (C.c_int, [_ctx_p, C.c_int, C.c_int, C.c_void_p, _i64, _i64]),
    'b200sph_pull_u32': (C.c_int, [_ctx_p, C.c_int, C.c_int, C.c_void_p, _i64, _i64]),
    'b200sph_set_async_copies': (C.c_int, [_ctx_p, C.c_int]),
    'b200sph_device_ptr': (C.c_int, [_ctx_p, C.c_int, C.c_int,
                                     C.POINTER(C.c_void_p)]),
    'b200sph_set_kernel': (C.c_int, [_ctx_p, C.c_int, C.c_int]),
    'b200sph_set_domain': (C.c_int, [_ctx_p, _dp, _dp, C.POINTER(C.c_int)]),
    'b200sph_set_mirror': (C.c_int, [_ctx_p, C.POINTER(C.c_int), C.c_double]),
    'b200sph_update_domain': (C.c_int, [_ctx_p]),
    'b200sph_nnps_update': (C.c_int, [_ctx_p]),
    'b200sph_nnps_update_deferred': (C.c_int, [_ctx_p]),
    'b200sph_nnps_confirm': (C.c_int, [_ctx_p, C.POINTER(C.c_int)]),
    'b200sph_get_grid': (C.c_int, [_ctx_p, C.POINTER(GridInfo)]),
    'b200sph_get_neighbors': (_i64, [_ctx_p, C.c_int, C.c_int, _i64, C.c_void_p, _i64]),
    'b200sph_eos': (C.c_int, [_ctx_p, C.c_int, C.c_int, C.c_double, C.c_double,
                              C.c_double, C.c_double, C.c_int]),
    'b200sph_ferrari_h': (C.c_int, [_ctx_p, C.c_int, C.c_double, C.c_int, C.c_int]),
    'b200sph_set_hm_static': (C.c_int, [_ctx_p, C.c_int]),
    'b200sph_pair_pass': (C.c_int, [_ctx_p, C.POINTER(PairProgram),
                                    C.POINTER(_i64)]),
    'b200sph_set_dest_range': (C.c_int, [_ctx_p, C.c_int, _i64, _i64]),
    'b200sph_user_property': (C.c_int, [_ctx_p, C.c_int]),
    'b200sph_generic_load': (C.c_int, [_ctx_p, C.c_void_p, _i64]),
    'b200sph_generic_launch': (C.c_int, [_ctx_p, C.c_int, C.c_char_p, C.c_int, C.c_int, C.c_uint,
                                         C.c_int, C.c_double, C.c_double, C.c_int]),
    'b200sph_tvf_pass': (C.c_int, [_ctx_p, C.POINTER(TvfProgram), C.POINTER(_i64)]),
    'b200sph_stage_tvf': (C.c_int, [_ctx_p, C.c_int, C.c_int, C.c_double]),
    'b200sph_stage_tvf_dev': (C.c_int, [_ctx_p, C.c_int, C.c_int]),
    'b200sph_stage_edac': (C.c_int, [_ctx_p, C.c_int, C.c_int, C.c_double]),
    'b200sph_stage_edac_dev': (C.c_int, [_ctx_p, C.c_int, C.c_int]),
    'b200sph_solid_pass': (C.c_int, [_ctx_p, C.POINTER(SolidProgram), C.POINTER(_i64)]),
    'b200sph_stage_solid': (C.c_int, [_ctx_p, C.c_int, C.c_int, C.c_double]),
    'b200sph_stage_solid_dev': (C.c_int, [_ctx_p, C.c_int, C.c_int]),
    'b200sph_stage': (C.c_int, [_ctx_p, C.c_int, C.c_int, C.c_double]),
    'b200sph_dt_factors': (C.c_int, [_ctx_p, _dp]),
    'b200sph_time_control': (C.c_int, [_ctx_p, C.c_void_p, C.POINTER(C.c_void_p)]),
    'b200sph_time_set': (C.c_int, [_ctx_p, C.c_double, C.c_double]),
    'b200sph_time_get': (C.c_int, [_ctx_p, _dp]),
    'b200sph_stage_dev': (C.c_int, [_ctx_p, C.c_int, C.c_int]),
    'b200sph_dt_propose': (C.c_int, [_ctx_p, C.c_double, C.c_int]),
    'b200sph_dt_commit': (C.c_int, [_ctx_p, C.c_double, C.c_double, C.c_int, C.c_int, C.c_int, C.c_int]),
    'b200sph_dt_advance': (C.c_int, [_ctx_p, C.c_double, C.c_int, C.c_double, C.c_double, C.c_int, C.c_int, C.c_int]),
    'b200sph_peer_init': (C.c_int, [_ctx_p, C.c_int, C.c_int, C.c_void_p]),
    'b200sph_peer_connect': (C.c_int, [_ctx_p, C.c_void_p]),
    'b200sph_peer_begin': (C.c_int, [_ctx_p]),
    'b200sph_peer_publish': (C.c_int, [_ctx_p, C.c_int, C.c_int]),
    'b200sph_peer_send': (C.c_int, [_ctx_p, C.c_int, C.c_int, C.c_int, C.c_void_p, _i64]),
    'b200sph_peer_reduce': (C.c_int, [_ctx_p, C.c_int]),
    'b200sph_peer_recv': (C.c_int, [_ctx_p, C.c_int, C.POINTER(_i64), C.POINTER(_i64), C.c_void_p]),
    'b200sph_peer_commit_dt': (C.c_int, [_ctx_p, C.c_double, C.c_double, C.c_int, C.c_int, C.c_int]),
    'b200sph_peer_end': (C.c_int, [_ctx_p]),
    'b200sph_peer_decision': (C.c_int, [_ctx_p, _dp]),
    'b200sph_peer_allreduce_dt': (C.c_int, [_ctx_p]),
    'b200sph_time_snapshot': (C.c_int, [_ctx_p, C.c_int, _dp]),
    'b200sph_halo_pack': (C.c_int, [_ctx_p, C.c_int, C.c_int, C.c_double,
                                    C.c_double, C.c_void_p, _i64,
                                    C.POINTER(_i64)]),
    'b200sph_halo_pack_selected': (C.c_int, [_ctx_p, C.c_int, C.c_int, C.c_void_p,
                                             _i64, C.POINTER(_i64)]),
    'b200sph_halo_overwrite': (C.c_int, [_ctx_p, C.c_int, _i64, C.c_void_p, _i64,
                                         _i64]),
    'b200sph_halo_pack_selected_all': (C.c_int, [_ctx_p, C.c_int, C.c_void_p, _i64,
                                                 C.POINTER(_i64)]),
    'b200sph_halo_overwrite_all': (C.c_int, [_ctx_p, C.POINTER(_i64),
                                             C.POINTER(_i64), C.c_void_p]),
    'b200sph_ipc_alloc': (C.c_int, [_ctx_p, _i64, C.POINTER(C.c_void_p),
                                    C.c_void_p]),
    'b200sph_ipc_open': (C.c_int, [_ctx_p, C.c_void_p, C.POINTER(C.c_void_p)]),
    'b200sph_ipc_close': (C.c_int, [_ctx_p, C.c_void_p, C.c_int]),
    'b200sph_nnps_drift': (C.c_int, [_ctx_p, _dp]),
    'b200sph_nnps_drift_device': (C.c_int, [_ctx_p, C.c_void_p]),
    'b200sph_nnps_keep_build': (C.c_int, [_ctx_p]),
    'b200sph_halo_append': (C.c_int, [_ctx_p, C.c_int, C.c_void_p, _i64, _i64,
                                      C.c_int, C.c_int]),
    'b200sph_drop_ghosts': (C.c_int, [_ctx_p, C.c_int]),
    'b200sph_migrate_out': (C.c_int, [_ctx_p, C.c_int, C.c_double, C.c_double,
                                      C.c_void_p, _i64, C.POINTER(_i64)]),
    'b200sph_time_final': (C.c_int, [_ctx_p, C.c_double, C.c_double]),
    'b200sph_snapshot_take': (C.c_int, [_ctx_p, C.c_int, C.POINTER(C.c_int),
                                        C.POINTER(C.c_int), C.POINTER(_i64)]),
    'b200sph_snapshot_fetch': (C.c_int, [_ctx_p, C.c_int, C.c_void_p, _i64]),
    'b200sph_snapshot_release': (C.c_int, [_ctx_p]),
    'b200sph_halo_layout': (C.c_int, [_ctx_p, C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    'b200sph_column_counts': (C.c_int, [_ctx_p, C.c_int, C.c_double, C.c_double, C.c_int,
                                        C.c_void_p]),
    'b200sph_get_stats': (C.c_int, [_ctx_p, C.POINTER(Stats)]),
    'b200sph_reset_stats': (C.c_int, [_ctx_p]),
    'b200sph_get_pair_r32_launches': (C.c_int, [_ctx_p, C.POINTER(C.c_int64)]),
    'b200sph_set_profiling': (C.c_int, [_ctx_p, C.c_int]),
}

_lib = None


def load():
    """Load libb200sph.so (build it with `python -m pysph_b200.build`)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            'pysph_b200: %s is missing. Build it with `python -m '
            'pysph_b200.build` (needs nvcc). There is no CPU fallback.'
            % LIB_PATH)
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)   # AttributeError if the symbol is missing
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


class B200Error(RuntimeError):
    pass


class Context(object):
    """Thin RAII wrapper over a b200sph_ctx handle."""

    def __init__(self, device=0):
        self.lib = load()
        h = _ctx_p()
        rc = self.lib.b200sph_create(int(device), C.byref(h))
        if rc != 0 or not h:
            msg = ''
            if h:
                msg = self.lib.b200sph_last_error(h).decode()
                self.lib.b200sph_destroy(h)
            raise B200Error(
                'b200sph_create(device=%d) failed (rc=%d) %s -- a CUDA device '
                'is required, there is no CPU fallback' % (device, rc, msg))
        self.h = h

    def close(self):
        if getattr(self, 'h', None):
            self.lib.b200sph_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def check(self, rc):
        if rc < 0:
            raise B200Error(self.lib.b200sph_last_error(self.h).decode())
        return rc

    def call(self, name, *args):
        return self.check(getattr(self.lib, name)(self.h, *args))
