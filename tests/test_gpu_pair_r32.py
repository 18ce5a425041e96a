"""The 32-byte-record form of the WCSPH list kernel (k_pair_list<..., R32>): with one h for
every particle, m and the Tait EOS uniform within each of at most two source classes and no
ghosts, a neighbour costs one 256-bit gather instead of a 256-bit and a 128-bit one.  Against
the 48-byte path (B200SPH_PAIR_R32=0): the same pairs, and fields that differ only by the few
ulp of the recomputed sound speed c_s,j inside the artificial viscosity.  Every case outside
those conditions must take the 48-byte path and give its bits exactly."""
import numpy as np
import pytest

from helpers import ACC_FIELDS
from test_gpu_parity import _perturbed_dam_break, make_solver, scheme_params
from test_gpu_periodic import _periodic_case

pytestmark = pytest.mark.gpu

FIELDS = ACC_FIELDS + ['x', 'u', 'rho']


def _run(monkeypatch, r32, make, steps=1):
    monkeypatch.setenv('B200SPH_PAIR_R32', '1' if r32 else '0')
    s, pas = make()
    s.a_eval.count_pairs = True
    s.initialise()
    pairs = s.a_eval.last_pairs
    for _ in range(steps):
        s.step()
    s.pull()
    st = s.a_eval.backend.stats()
    out = {}
    for pa in pas:
        order = np.argsort(pa.gid)
        for k in FIELDS:
            out[(pa.name, k)] = pa.properties[k][order].copy()
    return pairs, st, out


def _dam_break(dx, edit=None):
    def make():
        pas, params = _perturbed_dam_break(dx=dx)
        params = scheme_params(params)
        if edit:
            pas, params = edit(pas, params)
        return make_solver(pas, params, 'CubicSpline'), pas
    return make


def test_r32_matches_the_48_byte_path(gpu_device, monkeypatch, dx=0.05):
    """Perturbed 3-D dam break (fluid + boundary + obstacle: two source classes): the
    R32 kernel runs every pair pass, the pair counts are identical and after one EPEC
    step every field is within 1e-6 of its maximum of the 48-byte path's."""
    p1, st1, o1 = _run(monkeypatch, True, _dam_break(dx))
    p0, st0, o0 = _run(monkeypatch, False, _dam_break(dx))
    assert p1 == p0 and p1 > 0
    assert st1['pair_r32_launches'] == st1['pair_launches'] > 0
    assert st0['pair_r32_launches'] == 0
    for key, v in o0.items():
        scale = max(np.max(np.abs(v)), 1e-30)
        assert np.max(np.abs(o1[key] - v)) <= 1e-6 * scale, key


def _one_h(pas, params):
    pas[0].h[7] *= 1.01
    return pas, params


def _m_in_class(pas, params):
    pas[1].m[3] *= 1.5            # a boundary particle: the class {boundary, obstacle}
    return pas, params


def _three_classes(pas, params):
    # a second fluid: XSPH runs fluid -> fluid only, so fluid, fluid2 and the solids
    # are three different source columns
    import pysph_b200 as pb
    f = pas[0]
    sel = np.arange(f.x.size) % 3 == 0
    props = dict((k, v[sel].copy()) for k, v in f.properties.items())
    f2 = pb.get_particle_array_wcsph(name='fluid2', **props)
    keep = dict((k, v[~sel].copy()) for k, v in f.properties.items())
    f1 = pb.get_particle_array_wcsph(name=f.name, **keep)
    params = dict(params, fluids=list(params['fluids']) + ['fluid2'])
    return [f1, f2] + list(pas[1:]), params


def _update_h(pas, params):
    return pas, dict(params, update_h=True)


@pytest.mark.parametrize('case', ['h', 'm', 'classes', 'update_h'])
def test_r32_fallbacks_are_the_48_byte_path(gpu_device, monkeypatch, case, dx=0.05):
    """Outside its conditions the pair pass keeps the 48-byte kernel, bit for bit:
    one particle with another h, m differing within a source class, three source
    classes, a scheme that updates h."""
    edit = {'h': _one_h, 'm': _m_in_class, 'classes': _three_classes, 'update_h': _update_h}[case]
    p1, st1, o1 = _run(monkeypatch, True, _dam_break(dx, edit))
    p0, st0, o0 = _run(monkeypatch, False, _dam_break(dx, edit))
    assert p1 == p0 and p1 > 0
    assert st1['pair_r32_launches'] == 0 and st1['pair_launches'] > 0
    for key, v in o0.items():
        assert np.array_equal(o1[key], v), key


def test_r32_periodic(gpu_device, monkeypatch, n=10):
    """A periodic box has no ghost particles: it stays on the R32 kernel and agrees with
    the 48-byte path over 3 steps."""
    import pysph_b200 as pb

    def make():
        pa, params = _periodic_case(3, n)
        params['tensile_correction'] = False
        dm = pb.DomainManager(xmin=0, xmax=1, ymin=0, ymax=1, zmin=0, zmax=1,
                              periodic_in_x=True, periodic_in_y=True, periodic_in_z=True)
        return pb.make_wcsph_solver([pa], dict(params), pb.CubicSpline(dim=3), domain=dm), [pa]
    p1, st1, o1 = _run(monkeypatch, True, make, steps=3)
    p0, st0, o0 = _run(monkeypatch, False, make, steps=3)
    assert p1 == p0 and p1 > 0
    assert st1['pair_r32_launches'] == st1['pair_launches'] > 0
    assert st0['pair_r32_launches'] == 0
    for key, v in o0.items():
        scale = max(np.max(np.abs(v)), 1e-30)
        assert np.max(np.abs(o1[key] - v)) <= 1e-6 * scale, key
