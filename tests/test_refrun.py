"""oracle/_ref (C emitted by the reference's own code generator) agrees with the oracle port — guards the
argument marshalling of the `kind: "reference"` CPU baseline. What that generated code computes on this
problem is stored in tests/golden/refgen_iso3d_so*.npz (oracle/make_refgen_golden.py): the oracle port is
always compared with it, and the generated code itself as well wherever oracle/_ref was generated."""
import os

import numpy as np
import pytest

from oracle import oracle as O
from oracle import refrun
from helpers import iso_problem, load_golden, rel_linf


def _matches_golden(u, rec, g, tol=1e-5):
    scale = float(g['u_max'])
    assert abs(float(np.abs(u).max()) - scale) <= tol * scale
    xs = int(g['plane_x'])
    assert float(np.abs(u[:, xs].astype(np.float64) - g['u_plane']).max()) / scale < tol
    assert float(np.abs(u.reshape(-1)[g['u_index']].astype(np.float64) - g['u_sample']).max()) / scale < tol
    assert rel_linf(rec, g['rec']) < tol


@pytest.mark.parametrize('so', [8, 12])
def test_reference_generated_code_matches_oracle(so):
    g = load_golden(f'refgen_iso3d_so{so}')
    args = (int(g['n']), int(g['nbl']), so, float(g['tn']))
    p = iso_problem(*args)
    O.iso_forward(p['u'], so, p['w'], p['dt'], 1, p['nt'] - 2, damp=p['damp'], vp=1.5,
                  src=p['src'], rec=p['rec'])
    _matches_golden(p['u'], p['rec']['data'], g)
    ref = refrun.load_forward(so)
    if ref is None:                                 # oracle/_ref is only generated where the reference is
        return
    q = iso_problem(*args)
    refrun.run_forward(ref, q['u'], q['damp'], 1.5, q['dt'], 1, q['nt'] - 2, q['src'], q['rec'], so,
                       threads=min(4, os.cpu_count() or 1))
    assert rel_linf(q['u'], p['u']) < 1e-5
    assert rel_linf(q['rec']['data'], p['rec']['data']) < 1e-5
    _matches_golden(q['u'], q['rec']['data'], g)
