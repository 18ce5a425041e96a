"""Compare two `bench.py --dump-outputs` directories field by field, in the parity units of
the dam break (h0, c0, rho0): max |a - b| over the rows of every <array>_<field>.npy,
divided by the field's unit.  Prints one JSON line."""
import glob
import json
import os
import sys

import numpy as np


def units(h0, c0, rho0):
    u = {}
    for k in ('x', 'y', 'z'):
        u[k] = h0
    for k in ('u', 'v', 'w'):
        u[k] = c0
    u['rho'] = rho0
    u['p'] = rho0 * c0 * c0
    u['arho'] = rho0 * c0 / h0
    for k in ('au', 'av', 'aw'):
        u[k] = c0 * c0 / h0
    return u


def main(a, b, h0, c0, rho0):
    un = units(h0, c0, rho0)
    out, worst = {}, 0.0
    for fa in sorted(glob.glob(os.path.join(a, '*.npy'))):
        name = os.path.basename(fa)[:-4]
        arr, field = name.rsplit('_', 1)
        if field == 'gid':
            assert np.array_equal(np.load(fa), np.load(os.path.join(b, name + '.npy'))), name
            continue
        d = float(np.max(np.abs(np.load(fa) - np.load(os.path.join(b, name + '.npy'))), initial=0.0))
        out[name] = d / un[field]
        worst = max(worst, out[name])
    print(json.dumps({'max_parity_units': worst, 'fields': out}))


if __name__ == '__main__':
    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    from pysph_b200 import geometry as geo
    dx = float(sys.argv[3]) if len(sys.argv) > 3 else 0.00877
    p = geo.dam_break_3d_params(dx)
    main(sys.argv[1], sys.argv[2], p['h0'], p['c0'], p['rho0'])
