"""Device-resident mirror of a list of ParticleArrays on one B200.

``B200Backend`` owns the C-ABI context and plays the role the reference gives
to ``DeviceHelper`` (pysph/base/device_helper.py:47-250: push / pull / resize /
get_number_of_particles) for every array at once; ``B200DeviceHelper`` is the
per-array object installed as ``pa.gpu`` so that reference code paths which go
through ``pa.gpu`` (output pull particle_array.pyx:377-378, adaptive dt
integrator.py:62-81,146-159) find what they expect.
"""
import ctypes as C

import numpy as np

from . import _lib
from ._lib import (PROP_IDS, INT_PROP_IDS, EDAC_PROP_IDS, EDAC_WALL_PROP_IDS,
                   ELASTIC_PROP_IDS)


def _host_array(pa, name):
    """Zero-copy numpy view of ALL particles of a property (real + ghost)."""
    if hasattr(pa, 'get_carray'):       # real PySPH ParticleArray
        return pa.get_carray(name).get_npy_array()
    return pa.properties[name]


class _MinMax(object):
    def __init__(self, minimum, maximum):
        self.minimum = minimum
        self.maximum = maximum


class B200DeviceHelper(object):
    """``pa.gpu`` stand-in bound to one array of a B200Backend."""

    def __init__(self, backend, index):
        self._backend = backend
        self._index = index

    def push(self, *props):
        self._backend.push(self._index, props or None)

    def pull(self, *props):
        self._backend.pull(self._index, props or None)

    def resize(self, n):
        self._backend.resize(self._index, n)

    def get_number_of_particles(self, real=False):
        n, n_real = self._backend.sizes(self._index)
        return n_real if real else n

    def update_minmax_cl(self, props, only_max=False):
        # integrator.py:69-79 -> per-property maxima over the real particles
        f = self._backend.dt_factors()
        for name, val in (('dt_cfl', f[0]), ('dt_force', f[1])):
            if name in props:
                setattr(self, name, _MinMax(None, val))

    def get_device_array(self, name):
        if name != 'h':
            raise NotImplementedError('get_device_array(%r)' % name)
        return _MinMax(self._backend.dt_factors()[2], None)


class B200Backend(object):
    def __init__(self, particle_arrays, device=0, capacity_factor=1.0,
                 extra_capacity=0):
        if len(particle_arrays) > _lib.MAX_ARRAYS:
            raise ValueError('at most %d particle arrays' % _lib.MAX_ARRAYS)
        self.ctx = _lib.Context(device)
        self.device = device
        self.particle_arrays = list(particle_arrays)
        self.names = [pa.name for pa in particle_arrays]
        self.index = dict((n, i) for i, n in enumerate(self.names))
        # name -> device property id, per array: EDAC arrays evolve p (fp64 PF)
        # (a wall of the EDAC scheme may carry 'ap' too, wc/edac.py:46-47: walls first)
        self.prop_ids = [dict(EDAC_WALL_PROP_IDS if 'wij' in pa.properties and
                              'ug' in pa.properties else
                              (EDAC_PROP_IDS if 'ap' in pa.properties else
                               (ELASTIC_PROP_IDS if 's00' in pa.properties else PROP_IDS)))
                         for pa in particle_arrays]
        self.user_props = []      # names of the fp64 properties created for generic equations
        for pa in particle_arrays:
            n = pa.get_number_of_particles()
            n_real = pa.get_number_of_particles(real=True)
            cap = int(n * capacity_factor) + int(extra_capacity)
            i = self.ctx.call('b200sph_add_array', pa.name.encode(), n, n_real,
                              cap)
            assert i == self.index[pa.name]
            pa.gpu = B200DeviceHelper(self, i)
        self._dt_cache = None
        self.push_all()

    def add_user_property(self, name):
        """A property the device pool does not have (generic-equation fallback,
        pysph_b200/codegen.py): created as a zero-filled fp64 array for every particle
        array, filled from the host arrays that define it; push / pull carry it from now on."""
        if name in self.user_props:
            return _lib.USER_PROP0 + self.user_props.index(name)
        if len(self.user_props) >= _lib.MAX_USER_PROPS:
            raise NotImplementedError('at most %d user properties' % _lib.MAX_USER_PROPS)
        for pa in self.particle_arrays:
            if name in pa.properties and \
                    len(pa.properties[name]) != pa.get_number_of_particles():
                raise NotImplementedError(
                    'B200 generic equations: property %r of %r has a stride (%d values for %d '
                    'particles); user properties hold one value per particle'
                    % (name, pa.name, len(pa.properties[name]), pa.get_number_of_particles()))
        pid = _lib.USER_PROP0 + len(self.user_props)
        self.user_props.append(name)
        self.ctx.call('b200sph_user_property', pid)
        for i, pa in enumerate(self.particle_arrays):
            self.prop_ids[i][name] = pid
            if name in pa.properties:
                self.push(i, [name])
        return pid

    # -- sizes ----------------------------------------------------------------
    def sizes(self, i):
        n, nr = C.c_int64(), C.c_int64()
        self.ctx.call('b200sph_get_array_size', i, C.byref(n), C.byref(nr))
        return n.value, nr.value

    def resize(self, i, n, n_real=None):
        if n_real is None:
            n_real = min(self.sizes(i)[1], n)
        self.ctx.call('b200sph_resize_array', i, int(n), int(n_real))

    # -- host <-> device ------------------------------------------------------
    def _props_of(self, pa, props, ids=PROP_IDS):
        if props is None:
            props = [p for p in pa.properties
                     if p in ids or p in INT_PROP_IDS]
        return props

    def push(self, i, props=None):
        pa = self.particle_arrays[i]
        n = pa.get_number_of_particles()
        dn, _ = self.sizes(i)
        if dn != n:
            self.resize(i, n, pa.get_number_of_particles(real=True))
        ids = self.prop_ids[i]
        for name in self._props_of(pa, props, ids):
            a = _host_array(pa, name)
            if name in ids:
                a = np.ascontiguousarray(a, dtype=np.float64)
                self.ctx.call('b200sph_push_f64', i, ids[name],
                              a.ctypes.data, 0, n)
            elif name in INT_PROP_IDS:
                a = np.ascontiguousarray(a).view(np.uint32)
                self.ctx.call('b200sph_push_u32', i, INT_PROP_IDS[name],
                              a.ctypes.data, 0, n)
            # properties the hot path never touches (div, ...) stay host-only
        self._dt_cache = None

    def pull(self, i, props=None):
        pa = self.particle_arrays[i]
        n, n_real = self.sizes(i)
        if pa.get_number_of_particles() != n and hasattr(pa, 'resize'):
            pa.resize(n)
        # the real / ghost split can change while n stays the same (one particle
        # migrates out, one more ghost arrives): always take it from the device
        if hasattr(pa, 'set_num_real_particles'):
            pa.set_num_real_particles(n_real)
        ids = self.prop_ids[i]
        for name in self._props_of(pa, props, ids):
            a = _host_array(pa, name)
            if name in ids:
                if a.dtype == np.float64 and a.flags.c_contiguous:
                    self.ctx.call('b200sph_pull_f64', i, ids[name],
                                  a.ctypes.data, 0, n)
                else:
                    tmp = np.empty(n, dtype=np.float64)
                    self.ctx.call('b200sph_pull_f64', i, ids[name],
                                  tmp.ctypes.data, 0, n)
                    a[:] = tmp
            elif name in INT_PROP_IDS:
                tmp = np.empty(n, dtype=np.uint32)
                self.ctx.call('b200sph_pull_u32', i, INT_PROP_IDS[name],
                              tmp.ctypes.data, 0, n)
                a[:] = tmp.view(a.dtype) if a.dtype.itemsize == 4 else tmp

    def _real_view(self, pa, name, n_real, who):
        """A contiguous fp64 host buffer of at least n_real elements, or an error: the
        C-ABI takes a raw pointer and a count, so a host mirror shorter than the
        device's real-particle count (particles migrated in since it was sized) would
        be read / written past its end."""
        a = _host_array(pa, name)
        if a.dtype != np.float64 or not a.flags.c_contiguous:
            raise TypeError('%s: %s.%s must be a contiguous float64 array'
                            % (who, pa.name, name))
        if a.size < n_real:
            raise ValueError(
                '%s: the host mirror of %s.%s holds %d values but the device has %d '
                'real particles (migration changed the count): pull() / resize the '
                'host array first' % (who, pa.name, name, a.size, n_real))
        return a

    def push_real(self, props):
        """Push the REAL particles' values only (ghosts on the device, if any, keep
        theirs): the per-step host -> device path of a multi-GPU run.  The host
        mirrors must be in the device's particle order (true until a migration
        compacts the arrays: re-pull then)."""
        for i, pa in enumerate(self.particle_arrays):
            n_real = self.sizes(i)[1]
            for name in props:
                a = self._real_view(pa, name, n_real, 'push_real')
                self.ctx.call('b200sph_push_f64', i, self.prop_ids[i][name],
                              a.ctypes.data, 0, n_real)
        self._dt_cache = None

    def push_real_array(self, i, props):
        """push_real for one array"""
        pa = self.particle_arrays[i]
        n_real = self.sizes(i)[1]
        for name in props:
            a = self._real_view(pa, name, n_real, 'push_real_array')
            self.ctx.call('b200sph_push_f64', i, self.prop_ids[i][name],
                          a.ctypes.data, 0, n_real)
        self._dt_cache = None

    def pull_real(self, props):
        for i, pa in enumerate(self.particle_arrays):
            n_real = self.sizes(i)[1]
            for name in props:
                a = self._real_view(pa, name, n_real, 'pull_real')
                self.ctx.call('b200sph_pull_f64', i, self.prop_ids[i][name],
                              a.ctypes.data, 0, n_real)

    def push_all(self, props=None):
        for i in range(len(self.particle_arrays)):
            self.push(i, props)

    def pull_all(self, props=None):
        for i in range(len(self.particle_arrays)):
            self.pull(i, props)

    # -- reductions -----------------------------------------------------------
    def dt_factors(self):
        out = (C.c_double * 3)()
        self.ctx.call('b200sph_dt_factors', out)
        return out[0], out[1], out[2]

    def stats(self):
        s = _lib.Stats()
        self.ctx.call('b200sph_get_stats', C.byref(s))
        out = dict((k, getattr(s, k)) for k, _ in s._fields_)
        n = C.c_int64(0)
        self.ctx.call('b200sph_get_pair_r32_launches', C.byref(n))
        out['pair_r32_launches'] = n.value
        return out

    def synchronize(self):
        self.ctx.call('b200sph_synchronize')

    def use_torch_stream(self, stream=None):
        """Run the library on torch's current (or the given) CUDA stream so that
        torch.distributed collectives and torch events are ordered with our
        kernels.  torch's default stream has the handle 0, which the C-ABI reads
        as "own stream"; CUDA's explicit handle for it is cudaStreamLegacy = 1."""
        import torch
        if stream is None:
            stream = torch.cuda.current_stream()
        self.ctx.call('b200sph_set_stream', stream.cuda_stream or 1)
        return stream
