"""B200AccelerationEval: drop-in for the compiled AccelerationEval object.

Stands where ``SPHCompiler`` installs the generated Cython extension
(pysph/sph/sph_compiler.py:26-58, pysph/sph/acceleration_eval.py:228-248):
``compute(t, dt)``, ``set_nnps(nnps)``, ``update_particle_arrays(arrays)``.
The loop nest of acceleration_eval_cython.mako:262-363 becomes the op list
built by ``pysph_b200.program.build_program``, executed through the C-ABI.
"""
import ctypes as C

from . import _lib
from .kernels import kernel_id
from .program import build_program, index_value, _converged


class B200AccelerationEval(object):
    def __init__(self, particle_arrays, equations, kernel, backend=None,
                 mode='serial', device=0):
        from .backend import B200Backend
        self.particle_arrays = list(particle_arrays)
        self.kernel = kernel
        self.mode = mode
        self.backend = backend or B200Backend(self.particle_arrays,
                                              device=device)
        self.ctx = self.backend.ctx
        self.ctx.call('b200sph_set_kernel', kernel_id(kernel), int(kernel.dim))
        self.equation_groups = equations
        from . import codegen
        self._generic_props = codegen.PropertyTable(self.backend.user_props)
        self.ops = build_program(equations, self.backend.names, kernel.dim,
                                 particle_arrays=self.particle_arrays, kernel=kernel,
                                 generic=self._generic_props)
        # generated kernels address properties by NAME through the base table (x .. dt_force) and
        # the user properties: an array whose scheme keeps a name elsewhere (the EDAC fluids'
        # evolved p, a wall's ug ...) or a scheme-owned extension property would be aliased
        from ._lib import PROP_IDS
        base = set(codegen.F64_NAMES) | set(codegen.F32_NAMES) | set(codegen.U32_NAMES)
        for name in sorted(self._generic_props.used):
            for i, ids in enumerate(self.backend.prop_ids):
                if name in ids and name not in self.backend.user_props and \
                        (name not in base or ids[name] != PROP_IDS[name]):
                    raise NotImplementedError(
                        'B200 generic equations: property %r of array %r belongs to a hand-written '
                        'scheme (device id %d); generated kernels can only use the WCSPH base '
                        'properties and their own' % (name, self.backend.names[i], ids[name]))
        # properties the generated kernels use beyond the pool's own
        for name in self._generic_props.user:
            self.backend.add_user_property(name)
        # h and m stay what the host pushed unless an op writes them (UpdateSmoothingLengthFerrari,
        # a translated equation storing to h or m); with several evaluators on one backend, one
        # such op anywhere decides.  The library then may use uniform h / m as constants.
        self.backend.hm_static = getattr(self.backend, 'hm_static', True) and \
            not _writes_h_or_m(self.ops)
        self.ctx.call('b200sph_set_hm_static', int(self.backend.hm_static))
        self._range = None
        self.nnps = None
        self.count_pairs = False
        self.last_pairs = 0
        # reference API: AccelerationEval.c_acceleration_eval is "the compiled
        # object"; here the adapter is its own compiled object
        self.c_acceleration_eval = self

    # -- reference protocol ---------------------------------------------------
    def set_nnps(self, nnps):
        self.nnps = nnps

    def set_compiled_object(self, obj):
        self.c_acceleration_eval = obj

    def update_particle_arrays(self, particle_arrays):
        by_name = dict((pa.name, pa) for pa in particle_arrays)
        for i, name in enumerate(self.backend.names):
            if name in by_name:
                pa = by_name[name]
                self.backend.particle_arrays[i] = pa
                pa.gpu = self.particle_arrays[i].gpu
                self.particle_arrays[i] = pa
        self.backend.push_all()

    def compute(self, t, dt):
        self._pairs = 0
        self._run(self.ops, t, dt)
        self.last_pairs = self._pairs

    def _run(self, ops, t, dt):
        """The loop nest of acceleration_eval_cython.mako:262-363 over the op list."""
        ctx = self.ctx
        cnt = C.c_int64(0)
        for op in ops:
            kind = op[0]
            if kind == 'cond':
                if op[1](t, dt):
                    self._run(op[2], t, dt)
            elif kind == 'iterate':
                # helper:320-340: at least min_iterations, stop when every equation has
                # converged or after max_iterations
                _, min_it, max_it, group, body = op
                it = 1
                while True:
                    self._run(body, t, dt)
                    if it >= min_it and (_converged(group) or it == max_it):
                        break
                    it += 1
            elif kind == 'call':
                op[1]()
            elif kind == 'range':
                # destinations of the NEXT pair / generic op (one-shot in the library too)
                self._range = dict((d, (index_value(lo, pa), -1 if hi is None else index_value(hi, pa)))
                                   for d, (lo, hi, pa) in op[1].items())
            elif kind == 'generic':
                self._run_generic(op[1], t, dt)
            elif kind == 'eos':
                ctx.call('b200sph_eos', *op[1:])
            elif kind == 'ferrari':
                ctx.call('b200sph_ferrari_h', *op[1:])
            elif kind == 'pair':
                rng, self._range = self._range, None
                for d, (lo, hi) in (rng or {}).items():
                    ctx.call('b200sph_set_dest_range', d, lo, hi)
                if self.count_pairs:
                    ctx.call('b200sph_pair_pass', C.byref(op[1]), C.byref(cnt))
                    self._pairs += cnt.value
                else:
                    ctx.call('b200sph_pair_pass', C.byref(op[1]), None)
            elif kind == 'tvf':
                op[1].t = float(t)          # body-force damping, wc/edac.py:483-488
                if self.count_pairs:
                    ctx.call('b200sph_tvf_pass', C.byref(op[1]), C.byref(cnt))
                    self._pairs += cnt.value
                else:
                    ctx.call('b200sph_tvf_pass', C.byref(op[1]), None)
            elif kind == 'solid':
                if self.count_pairs:
                    ctx.call('b200sph_solid_pass', C.byref(op[1]), C.byref(cnt))
                    self._pairs += cnt.value
                else:
                    ctx.call('b200sph_solid_pass', C.byref(op[1]), None)
            elif kind == 'update_nnps':
                # mako:139-145: nnps.update_domain(); nnps.update()
                ctx.call('b200sph_update_domain')
                ctx.call('b200sph_nnps_update')

    # -- generic-equation fallback (codegen.py) -------------------------------------
    def _run_generic(self, gg, t, dt):
        """do_group (acceleration_eval_cython.mako:10-155) for a Group of translated equations:
        destination after destination -- initialize over its particles, the neighbour loops,
        post_loop -- each a launch of the Group's run-time compiled kernel."""
        from . import codegen
        ctx = self.ctx
        if getattr(gg, 'module', None) is None:
            image = codegen.compile_cached(gg.source)
            buf = C.create_string_buffer(image, len(image))
            gg.module = ctx.call('b200sph_generic_load', C.cast(buf, C.c_void_p), len(image))
            w = gg.writes
            gg.write_flags = (1 if w & {'x', 'y', 'z', 'h'} else 0) | \
                (2 if w & {'u', 'v', 'w', 'm', 'rho', 'p', 'cs'} else 0)
        rng, self._range = self._range, None
        for name, d, has_init, has_loop, has_post, src_mask in gg.kernels:
            py_inits, reduces = gg.host_calls.get(d, ((), ()))
            for eq in py_inits:          # host side, before anything of the destination (mako:29-40)
                eq.py_initialize(self.particle_arrays[d], t, dt)
            for phase, on in ((0, has_init), (1, has_loop), (2, has_post)):
                if not on:
                    continue
                if rng and d in rng:
                    ctx.call('b200sph_set_dest_range', d, rng[d][0], rng[d][1])
                ctx.call('b200sph_generic_launch', gg.module, name.encode(), d, phase, src_mask,
                         gg.real_only, float(t), float(dt), gg.write_flags)
            for eq in reduces:           # host side, after post_loop (mako:127-130)
                eq.reduce(self.particle_arrays[d], t, dt)


def _writes_h_or_m(ops):
    """Whether an op of the list (nested ones included) stores to h or m on the device."""
    for op in ops:
        kind = op[0]
        if kind == 'ferrari':
            return True
        if kind == 'generic' and set(op[1].writes) & {'h', 'm'}:
            return True
        if kind == 'cond' and _writes_h_or_m(op[2]):
            return True
        if kind == 'iterate' and _writes_h_or_m(op[4]):
            return True
    return False
