"""CPU-side tests (no GPU): the DSL, the finite-difference machinery, the pattern recogniser,
the NumPy interpreter for set-up operators, the host-side tabulation, and the C-ABI library's
exported symbols. Golden values come from the reference (tests/golden, oracle/make_golden.py)."""
import os

import numpy as np
import pytest

import devito_b200 as dv
from devito_b200 import Grid, Function, TimeFunction, Eq, Operator, solve
from devito_b200.symbolics import fd_weights, fd_offsets
from devito_b200.seismic import (demo_model, setup_geometry, AcousticWaveSolver, AnisotropicWaveSolver)
from helpers import load_golden, rel_linf


def test_library_loads_and_exports_every_declared_symbol():
    from devito_b200 import _lib
    L = _lib.load_library()
    hdr = open(os.path.join(os.path.dirname(_lib.LIB_PATH), '..', 'include', 'b200stencil.h')).read()
    import re
    declared = set(re.findall(r'\b(b2_[a-z0-9_]+)\s*\(', hdr))
    assert declared == set(_lib.SYMBOLS)
    for s in declared:
        assert hasattr(L, s), s
    assert b'sm_100a' in L.b2_version()


def test_hot_path_fails_loudly_without_gpu(monkeypatch):
    """No CPU fallback: a recognised propagator raises when no CUDA device is present (where there is
    one, the library is made to report none)."""
    from devito_b200 import _lib
    if _lib.have_gpu():
        monkeypatch.setattr(_lib, '_gpu_checked', False)
    model = demo_model('constant-isotropic', shape=(12, 12, 12), spacing=(10., 10., 10.), nbl=4, space_order=4)
    solver = AcousticWaveSolver(model, setup_geometry(model, 20.0), space_order=4)
    assert solver.op_fwd().backend == 'cuda-sm100a'
    with pytest.raises(dv.BackendUnavailable):
        solver.forward()


def test_fd_weights_match_reference_literals():
    # literals printed by the reference's generated code for so=8, h=10 (Forward / ForwardTTI)
    w = fd_weights(2, list(range(-4, 5)), 0)
    assert np.allclose(np.float32(np.array(w[4:]) / 100.0),
                       np.float32([-2.84722216e-2, 1.59999996e-2, -1.99999996e-3, 2.53968248e-4, -1.78571425e-5]))
    from fractions import Fraction
    assert fd_offsets(4, Fraction(1, 2)) == [-1, 0, 1, 2]
    assert fd_offsets(4, Fraction(-1, 2)) == [-2, -1, 0, 1]
    assert fd_offsets(8, 0) == list(range(-4, 5))
    assert fd_offsets(1, 0, is_time=True) == [0, 1]          # u.dt: forward difference
    w1 = fd_weights(1, [-1, 0, 1, 2], Fraction(1, 2))
    assert np.allclose(np.float32(np.array(w1) / 10.0),
                       np.float32([4.16666673e-3, -1.12500002e-1, 1.12500002e-1, -4.16666673e-3]))


def test_time_derivative_semantics():
    g = Grid(shape=(8, 8))
    u = TimeFunction(name='u', grid=g, time_order=2, space_order=2)
    dt = g.stepping_dim.spacing
    e = (u.dt2 * dt ** 2).evaluate
    from devito_b200.symbolics import linear_terms
    terms, rest = linear_terms(e, lambda a: a.function is u)
    got = {int(a.index_objs[0].shift): c for a, c in terms.items()}
    from devito_b200.operator import eval_scalar
    vals = {k: eval_scalar(v, lambda n: 0.7) for k, v in got.items()}
    assert np.allclose([vals[-1], vals[0], vals[1]], [1, -2, 1])


def test_model_matches_reference_golden():
    g = load_golden('iso3d_so8')
    model = demo_model('constant-isotropic', spacing=(10., 10., 10.), shape=(20, 20, 20), nbl=8, space_order=8)
    geometry = setup_geometry(model, float(g['tn']))
    AcousticWaveSolver(model, geometry, space_order=8)     # switches damp to the "damp" profile
    assert model.critical_dt == g['dt']
    assert geometry.nt == int(g['nt'])
    assert rel_linf(model.damp.data, g['damp']) < 1e-6     # initdamp ran through the interpreter
    assert rel_linf(geometry.src.data, g['src']) < 1e-6
    np.testing.assert_allclose(geometry.src.coordinates.data, g['src_coords'], rtol=1e-6)
    np.testing.assert_allclose(geometry.rec.coordinates.data, g['rec_coords'], rtol=1e-6)
    c = load_golden('coefficients')
    for so in (4, 8, 12, 16):
        m = demo_model('constant-isotropic', spacing=(10., 10., 10.), shape=(8, 8, 8), nbl=2, space_order=so)
        assert m.critical_dt == c[f'dt_iso_so{so}']
        m = demo_model('constant-tti', spacing=(10., 10., 10.), shape=(8, 8, 8), nbl=2, space_order=so)
        assert m.critical_dt == c[f'dt_tti_so{so}']


def test_tabulation_matches_oracle():
    from oracle import oracle as O
    model = demo_model('constant-isotropic', spacing=(10., 10., 10.), shape=(20, 20, 20), nbl=8, space_order=8)
    for interp in ('linear', 'sinc'):
        geometry = setup_geometry(model, 50.0, interpolation=interp)
        rec = geometry.rec
        gp, ws = rec.tabulate()
        r = 1 if interp == 'linear' else 4
        gp2, ws2 = O.tabulate(rec.coordinates.data, model.grid.origin, model.grid.spacing, r, interp)
        assert np.array_equal(gp, gp2)
        for a, b in zip(ws, ws2):
            assert np.array_equal(a, b)


def test_recogniser_accepts_the_reference_formulations():
    model = demo_model('constant-isotropic', spacing=(10., 10., 10.), shape=(12, 12, 12), nbl=4, space_order=8)
    op = AcousticWaveSolver(model, setup_geometry(model, 20.0), space_order=8).op_fwd()
    assert op.backend == 'cuda-sm100a' and op._plan['kind'] == 'iso'
    assert op._plan['m_role'][0] == 'vp_c' and op._plan['damp'] is model.damp
    assert op._plan['rec_toff'] == 0
    assert op.cfunction.__name__ == 'b2_iso_forward'
    m2 = demo_model('layers-isotropic', spacing=(10., 10., 10.), shape=(12, 12, 12), nbl=4, space_order=4)
    op2 = AcousticWaveSolver(m2, setup_geometry(m2, 20.0), space_order=4).op_fwd()
    assert op2._plan['m_role'][0] == 'vp_f'
    m3 = demo_model('constant-tti', spacing=(10., 10., 10.), shape=(12, 12, 12), nbl=4, space_order=8)
    op3 = AnisotropicWaveSolver(m3, setup_geometry(m3, 20.0), space_order=8).op_fwd()
    assert op3._plan['kind'] == 'tti' and op3.cfunction.__name__ == 'b2_tti_forward'


def test_recogniser_rejects_other_equations():
    g = Grid(shape=(16, 16), extent=(1., 1.))
    u = TimeFunction(name='u', grid=g, time_order=1, space_order=2)
    # a constant-coefficient explicit update is not a wave scheme: it goes to the generic stencil entry
    op = Operator([Eq(u.forward, u + 0.1 * u.laplace)], subs=g.spacing_map)
    assert op.backend == 'cuda-sm100a' and op._plan['kind'] == 'linear'
    # a wave equation with a wrong coefficient is NOT silently mapped to the wave kernels
    v = TimeFunction(name='v', grid=g, time_order=2, space_order=4)
    m = Function(name='m', grid=g, space_order=4)
    m.data[:] = 1.0
    pde = m * v.dt2 - 1.5 * v.laplace
    op2 = Operator([Eq(v.forward, solve(pde, v.forward))], subs=g.spacing_map)
    assert op2.backend == 'numpy-interpreter'


def test_diffusion_config1_is_on_the_generic_stencil_path():
    """BASELINE config 1: 2-D diffusion, Laplace so=2 (examples/cfd/example_diffusion.py:120-133). The
    operator is recognised as a constant-coefficient explicit update and marshalled for
    `b2_linear_forward`; the kernel's point code against the NumPy twin is tests/test_zz_emulation.py,
    the run on the GPU tests/test_zz_linear.py."""
    n, a = 64, 0.5
    g = Grid(shape=(n, n), extent=(2., 2.))
    u = TimeFunction(name='u', grid=g, time_order=1, space_order=2)
    hx, hy = g.spacing
    dt = 0.2 * hx * hy / a
    eq = Eq(u.forward, solve(Eq(u.dt, a * u.laplace), u.forward), subdomain=g.interior)
    op = Operator([eq])
    assert op.backend == 'cuda-sm100a' and op._plan['kind'] == 'linear'
    args = op.arguments(time_M=19, dt=dt)
    taps = {(t, o): c for t, o, c in args['taps']}
    dtf = float(np.float32(dt))
    want = {(0, (0, 0)): 1 - 2 * a * dtf / hx ** 2 - 2 * a * dtf / hy ** 2,
            (0, (1, 0)): a * dtf / hx ** 2, (0, (-1, 0)): a * dtf / hx ** 2,
            (0, (0, 1)): a * dtf / hy ** 2, (0, (0, -1)): a * dtf / hy ** 2}
    assert set(taps) == set(want)
    for k in want:
        assert abs(taps[k] - want[k]) < 1e-6 * max(1.0, abs(want[k]))
    assert (args['lo'], args['hi'], args['time_m'], args['time_M']) == ([1, 1], [n - 2, n - 2], 0, 19)
    # the reference's own call: `op.apply(u=u, t=timesteps, dt=dt)` on the whole grid
    op2 = Operator(Eq(u.forward, solve(Eq(u.dt, a * (u.dx2 + u.dy2)), u.forward)))
    a2 = op2.arguments(u=u, t=500, dt=dt)
    assert (a2['lo'], a2['hi'], a2['time_M']) == ([0, 0], [n - 1, n - 1], 500)
    # it fails loudly without a GPU — no interpreter fallback for a recognised operator
    from devito_b200.exceptions import BackendUnavailable
    from devito_b200 import _lib
    if not _lib.have_gpu():
        with pytest.raises(BackendUnavailable):
            op(time_M=3, dt=dt)


def test_interpolation_and_injection_interpreter():
    """Linear interpolation reproduces a linear field exactly; injection is its transpose
    (tests/test_interpolation.py:127-260 of the reference)."""
    from devito_b200 import SparseFunction
    g = Grid(shape=(11, 11), extent=(10., 10.))
    f = Function(name='f', grid=g, space_order=2)
    x = np.linspace(0, 10, 11)
    f.data[:] = x[:, None] + 2 * x[None, :]
    sf = SparseFunction(name='s', grid=g, npoint=3, coordinates=np.array([[1.5, 2.25], [7.1, 3.9], [0.0, 9.99]]))
    Operator(sf.interpolate(f))()
    c = sf.coordinates.data
    assert np.allclose(sf.data, c[:, 0] + 2 * c[:, 1], rtol=1e-6)
    h = Function(name='h', grid=g, space_order=2)
    sf.data[:] = [1.0, 2.0, 3.0]
    Operator(sf.inject(h, sf))()
    assert np.isclose(h.data.sum(), 6.0)


def test_apply_argument_checks():
    model = demo_model('constant-isotropic', spacing=(10., 10., 10.), shape=(12, 12, 12), nbl=4, space_order=8)
    geometry = setup_geometry(model, 20.0)
    op = AcousticWaveSolver(model, geometry, space_order=8).op_fwd()
    with pytest.raises(dv.InvalidArgument):
        op.arguments(dt=1.0, bogus=3)
    with pytest.raises(dv.InvalidArgument):
        op.arguments()                                    # no dt
    args = op.arguments(dt=model.critical_dt)
    assert args['time_m'] == 1 and args['time_M'] == geometry.nt - 2    # devito/types/dimension.py:279-331
    with pytest.raises(dv.InvalidArgument):
        op.arguments(dt=1.0, time_M=geometry.nt)          # OOB in the sparse time axis
    with pytest.raises(dv.InvalidArgument):
        op.arguments(dt=1.0, x_M=1000)


def test_reference_examples_run_unchanged_up_to_the_ffi():
    """The reference's own examples/seismic, imported unmodified against this package aliased as
    `devito`, build operators that the recogniser maps to the CUDA entry points."""
    ref = '/root/reference'
    if not os.path.isdir(os.path.join(ref, 'examples', 'seismic')):
        pytest.skip("reference tree not present")
    import subprocess, sys, textwrap
    code = textwrap.dedent('''
        import sys
        sys.path.insert(0, %r)
        import devito_b200
        devito_b200.install_as_devito()
        sys.path.insert(0, %r)
        import numpy as np
        from examples.seismic import demo_model, setup_geometry
        from examples.seismic.acoustic import AcousticWaveSolver
        from examples.seismic.tti import AnisotropicWaveSolver
        m = demo_model('constant-isotropic', spacing=(10., 10., 10.), shape=(12, 12, 12), nbl=4, space_order=8)
        op = AcousticWaveSolver(m, setup_geometry(m, 20.0), space_order=8).op_fwd()
        assert op.backend == 'cuda-sm100a', op._why_not
        m = demo_model('constant-tti', spacing=(10., 10., 10.), shape=(12, 12, 12), nbl=4, space_order=8)
        op = AnisotropicWaveSolver(m, setup_geometry(m, 20.0), space_order=8).op_fwd()
        assert op.backend == 'cuda-sm100a', op._why_not
        print('OK')
    ''') % (os.path.dirname(os.path.dirname(os.path.abspath(__file__))), ref)
    r = subprocess.run([sys.executable, '-c', code], capture_output=True, text=True, timeout=300)
    assert 'OK' in r.stdout, r.stdout + r.stderr


@pytest.mark.parametrize('so', [2, 4, 8, 12])
@pytest.mark.parametrize('deriv,attr', [(1, 'dx'), (2, 'dx2'), (1, 'dy'), (2, 'dy2')])
def test_derivatives_are_exact_on_polynomials(so, deriv, attr):
    """Like the reference's tests/test_derivatives.py: an FD derivative of space order `so` is exact
    (to rounding) for polynomials of degree <= so, through Derivative.evaluate and the interpreter."""
    from devito_b200 import Function
    n, h = 24, 0.5
    grid = Grid(shape=(n, n), extent=((n - 1) * h, (n - 1) * h), dtype=np.float64)
    f = Function(name='f', grid=grid, space_order=so, dtype=np.float64)
    g = Function(name='g', grid=grid, space_order=so, dtype=np.float64)
    x = (np.arange(n + 2 * so) - so) * h
    X, Y = np.meshgrid(x, x, indexing='ij')
    axis = X if attr.startswith('dx') else Y
    other = Y if attr.startswith('dx') else X
    # the reference's first derivative at space_order 2 is the two-point forward difference
    # (`-f(x)/h + f(x+h)/h`), exact for degree 1 only
    deg = 1 if (so == 2 and deriv == 1) else min(so, 6)
    coef = np.linspace(1.0, 2.0, deg + 1)
    f.data_with_halo[:] = sum(c * axis ** k for k, c in enumerate(coef)) * (1.0 + 0.1 * other)
    exact = sum(c * np.prod(np.arange(k, k - deriv, -1)) * axis ** (k - deriv)
                for k, c in enumerate(coef) if k >= deriv) * (1.0 + 0.1 * other)
    Operator([Eq(g, getattr(f, attr))])()
    got = np.asarray(g.data)
    want = exact[so:-so, so:-so]
    assert np.max(np.abs(got - want)) <= 1e-7 * np.max(np.abs(want))


def test_interpreter_runs_backward_updates_backward_in_time():
    """`f.backward = ...` is stepped from time_M down to time_m like the reference's backward loop
    (ADVICE r1: the interpreter iterated forward and read levels nobody had produced)."""
    g = Grid(shape=(8, 8))
    nt = 6
    f = TimeFunction(name='f', grid=g, time_order=1, space_order=2, save=nt)
    c = Function(name='c', grid=g, space_order=2)           # position-dependent factor: not the linear path
    c.data[:] = 2.0
    f.data[nt - 1] = 1.0
    op = Operator([Eq(f.backward, c * f)])
    assert op.backend == 'numpy-interpreter'
    op(time_m=1, time_M=nt - 1)
    for k in range(nt):
        assert np.allclose(f.data[k], 2.0 ** (nt - 1 - k))


def test_sparse_radius_must_fit_the_halo():
    """devito/operations/interpolators.py:28-37 `check_radius`."""
    from devito_b200 import SparseTimeFunction
    g = Grid(shape=(12, 12, 12))
    u2 = TimeFunction(name='u2', grid=g, time_order=2, space_order=2)
    s = SparseTimeFunction(name='s', grid=g, npoint=1, nt=4, interpolation='sinc', r=4)
    with pytest.raises(ValueError):
        s.inject(field=u2.forward, expr=s)
    with pytest.raises(ValueError):
        s.interpolate(expr=u2)


def test_critical_dt_is_cached_until_a_parameter_is_written():
    """`SeismicModel.critical_dt` (examples/seismic/model.py:370-382) reduces vp and epsilon over the whole grid; the
    mirror caches the result on the parameter storages' write versions (86 ms per apply at 512^3 otherwise)."""
    from devito_b200.seismic import SeismicModel
    from devito_b200.seismic import model as M
    shape = (24, 20, 22)
    v = np.full(shape, 1.5, dtype=np.float32)
    v[..., 11:] = 2.5
    m = SeismicModel(origin=(0., 0., 0.), spacing=(10., 10., 10.), shape=shape, space_order=4, vp=v, nbl=4,
                     bcs='damp', epsilon=0.1 * (v - 1.5), delta=0.05 * (v - 1.5), theta=0.3 * (v - 1.5),
                     phi=0.1 * (v - 1.5))
    calls = []
    real = M.mmax
    M.mmax = lambda f: (calls.append(1), real(f))[1]
    try:
        dt0 = m.critical_dt
        n0 = len(calls)
        assert n0 >= 1
        assert m.critical_dt == dt0 and len(calls) == n0           # cached
        m.vp.data[:] = 3.0                                         # write access -> recomputed
        dt1 = m.critical_dt
        assert len(calls) > n0 and dt1 < dt0
        m.dt_scale = 0.5
        assert abs(float(m.critical_dt) - 0.5 * float(dt1)) < 1e-3 * float(dt1)
    finally:
        M.mmax = real
