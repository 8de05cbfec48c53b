"""ctypes wrapper around oracle/oracle.c + NumPy restatements of the host-side pieces.

TEST INFRASTRUCTURE ONLY: may be imported by tests/, __graft_entry__.smoke() and bench.py's
cpu_baseline / --impl reference legs. Parity is pinned against golden vectors generated from
the reference itself (oracle/make_golden.py -> tests/golden/).
"""
import ctypes
import os
import subprocess
from ctypes import POINTER, Structure, c_float, c_int

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))


class OSparse(Structure):
    _fields_ = [('data', POINTER(c_float)), ('gp', POINTER(c_int)), ('w', POINTER(c_float) * 3),
                ('nt', c_int), ('npoint', c_int), ('p_m', c_int), ('p_M', c_int), ('r', c_int)]


_libs = {}


def build(fast=False):
    src = os.path.join(HERE, 'oracle.c')
    env = dict(os.environ)
    env.pop('CC', None)
    if fast:
        # -march=native: built at run time for the host it runs on, outside the source tree
        from .refrun import host_build_path
        path = host_build_path('liboracle_fast', [src, os.path.join(HERE, 'Makefile')])
        if not os.path.exists(path):
            tmp = f'{path}.{os.getpid()}'
            subprocess.run(['make', '-B', '-C', HERE, 'liboracle_fast.so', f'FAST_SO={tmp}'], check=True,
                           capture_output=True, env=env)
            os.replace(tmp, path)
        return path
    path = os.path.join(HERE, 'liboracle.so')
    if not os.path.exists(path) or os.path.getmtime(path) < os.path.getmtime(src):
        subprocess.run(['make', '-B', '-C', HERE, 'liboracle.so'], check=True, capture_output=True, env=env)
    return path


def load(fast=False):
    if fast in _libs:
        return _libs[fast]
    L = ctypes.CDLL(build(fast))
    fp, ip = POINTER(c_float), POINTER(c_int)
    L.oracle_iso_forward.argtypes = [c_int, fp, c_int, ip, c_int, c_int, fp, fp, fp, fp, c_int, fp,
                                     c_float, c_float, ip, ip, c_int, c_int, POINTER(OSparse),
                                     POINTER(OSparse), c_int, c_int, fp, ip, c_int, fp, c_int, c_int]
    L.oracle_iso_forward.restype = c_int
    L.oracle_born_forward.argtypes = [fp, fp, c_int, ip, c_int, c_int, fp, fp, fp, fp, c_int, fp, c_float,
                                      c_float, ip, ip, c_int, c_int, POINTER(OSparse), POINTER(OSparse),
                                      fp, ip, c_int]
    L.oracle_born_forward.restype = c_int
    L.oracle_tti_forward.argtypes = [fp, fp, c_int, ip, c_int, c_int, fp, fp, fp, fp, fp, fp, fp,
                                     c_float, c_float, c_float, c_float, c_float, c_float, ip, ip,
                                     c_int, c_int, POINTER(OSparse), POINTER(OSparse), c_int,
                                     fp, fp, fp, fp, fp]
    L.oracle_tti_forward.restype = c_int
    _libs[fast] = L
    return L


def _fp(a):
    return a.ctypes.data_as(POINTER(c_float)) if a is not None else None


def _ip(a):
    return a.ctypes.data_as(POINTER(c_int))


def _sparse(data, gp, ws, r, keep):
    if data is None:
        return None
    s = OSparse()
    gp = np.ascontiguousarray(gp, dtype=np.int32)
    ws = [np.ascontiguousarray(w, dtype=np.float32) for w in ws]
    keep.extend([gp, ws])
    s.data = _fp(data)
    s.gp = _ip(gp)
    for i, w in enumerate(ws):
        s.w[i] = _fp(w)
    s.nt, s.npoint = data.shape
    s.p_m, s.p_M = 0, data.shape[1] - 1
    s.r = r
    return s


def iso_forward(u, so, w, dt, time_m, time_M, damp=None, vp=1.5, param=None, param_kind=0,
                src=None, rec=None, rec_toff=0, lo=None, hi=None, fast=False, adjoint=False,
                grad=None, ghalo=0, usave=None, free_surface=False, ot4=False):
    """grad (3-D, halo `ghalo`) / usave (nt, ...) enable the Gradient operator's imaging condition.
    u: (T, [nx+2so,] ny+2so, nz+2so) float32 C-contiguous, updated in place.
    w: list (per dim) of weights [0..R] incl. 1/h^2. src/rec: dict(data, gp, w, r)."""
    L = load(fast)
    nd = u.ndim - 1
    R = len(w[0]) - 1
    alloc = np.array(u.shape[1:], dtype=np.int32)
    lo = np.array(lo if lo is not None else [0] * nd, dtype=np.int32)
    hi = np.array(hi if hi is not None else [s - 2 * so - 1 for s in u.shape[1:]], dtype=np.int32)
    wa = [np.ascontiguousarray(x, dtype=np.float32) for x in w] + [None] * (3 - nd)
    keep = []
    s = _sparse(src['data'], src['gp'], src['w'], src['r'], keep) if src else None
    r = _sparse(rec['data'], rec['gp'], rec['w'], rec['r'], keep) if rec else None
    galloc = np.array(grad.shape, dtype=np.int32) if grad is not None else None
    rc = L.oracle_iso_forward(nd, _fp(u), u.shape[0], _ip(alloc), so, R, _fp(wa[0]), _fp(wa[1]),
                              _fp(wa[2]) if wa[2] is not None else None, _fp(damp), param_kind,
                              _fp(param), vp, dt, _ip(lo), _ip(hi), time_m, time_M,
                              ctypes.byref(s) if s else None, ctypes.byref(r) if r else None, rec_toff,
                              1 if adjoint else 0, _fp(grad),
                              _ip(galloc) if galloc is not None else None,
                              ghalo, _fp(usave), 1 if free_surface else 0, 1 if ot4 else 0)
    assert rc == 0
    return u


def born_forward(u, U, dm, so, w, dt, time_m, time_M, damp=None, vp=1.5, param=None, param_kind=0,
                 src=None, rec=None, dmhalo=0, fast=False):
    """The reference's `Born` operator (examples/seismic/acoustic/operators.py:235-277): u driven by
    `src`, the linearised field U driven by -dm * u.dt2, `rec` sampled from U. 3-D."""
    L = load(fast)
    R = len(w[0]) - 1
    alloc = np.array(u.shape[1:], dtype=np.int32)
    lo = np.array([0] * 3, dtype=np.int32)
    hi = np.array([s - 2 * so - 1 for s in u.shape[1:]], dtype=np.int32)
    wa = [np.ascontiguousarray(x, dtype=np.float32) for x in w]
    keep = []
    s = _sparse(src['data'], src['gp'], src['w'], src['r'], keep) if src else None
    r = _sparse(rec['data'], rec['gp'], rec['w'], rec['r'], keep) if rec else None
    dm = np.ascontiguousarray(dm, dtype=np.float32)
    dmalloc = np.array(dm.shape, dtype=np.int32)
    rc = L.oracle_born_forward(_fp(u), _fp(U), u.shape[0], _ip(alloc), so, R, _fp(wa[0]), _fp(wa[1]), _fp(wa[2]),
                               _fp(damp), param_kind, _fp(param), vp, dt, _ip(lo), _ip(hi), time_m, time_M,
                               ctypes.byref(s) if s else None, ctypes.byref(r) if r else None, _fp(dm),
                               _ip(dmalloc), dmhalo)
    assert rc == 0
    return u, U


def tti_forward(u, v, so, w2, w1, dt, time_m, time_M, damp, vp, epsilon, delta, theta, phi,
                src=None, rec=None, rec_toff=0, lo=None, hi=None, fast=False, arrays=None):
    """arrays: optional dict name -> (allocated-layout f32 array) for vp/epsilon/delta/theta/phi."""
    L = load(fast)
    arrays = arrays or {}
    R = len(w2[0]) - 1
    alloc = np.array(u.shape[1:], dtype=np.int32)
    lo = np.array(lo if lo is not None else [0] * 3, dtype=np.int32)
    hi = np.array(hi if hi is not None else [s - 2 * so - 1 for s in u.shape[1:]], dtype=np.int32)
    w2a = [np.ascontiguousarray(x, dtype=np.float32) for x in w2]
    w1a = [np.ascontiguousarray(x, dtype=np.float32) for x in w1]
    keep = []
    s = _sparse(src['data'], src['gp'], src['w'], src['r'], keep) if src else None
    r = _sparse(rec['data'], rec['gp'], rec['w'], rec['r'], keep) if rec else None
    rc = L.oracle_tti_forward(_fp(u), _fp(v), u.shape[0], _ip(alloc), so, R, _fp(w2a[0]), _fp(w2a[1]),
                              _fp(w2a[2]), _fp(w1a[0]), _fp(w1a[1]), _fp(w1a[2]), _fp(damp), vp,
                              epsilon, delta, theta, phi, dt, _ip(lo), _ip(hi), time_m, time_M,
                              ctypes.byref(s) if s else None, ctypes.byref(r) if r else None, rec_toff,
                              _fp(arrays.get('vp')), _fp(arrays.get('epsilon')), _fp(arrays.get('delta')),
                              _fp(arrays.get('theta')), _fp(arrays.get('phi')))
    assert rc == 0
    return u, v


# ---------------------------------------------------------------------------------------------
# host-side restatements (NumPy / SymPy)
# ---------------------------------------------------------------------------------------------
def fd2_weights(space_order, h):
    """Second-derivative weights/h^2: finite_diff_weights(2, range(-so/2, so/2+1), 0), evalf(9)
    (devito/finite_differences/tools.py:231-236; finite_difference.py:185-187)."""
    from sympy import finite_diff_weights
    R = space_order // 2
    w = finite_diff_weights(2, list(range(-R, R + 1)), 0)[-1][-1]
    w = [float(c.evalf(9)) for c in w]
    return np.array([w[R + k] / float(h) ** 2 for k in range(R + 1)], dtype=np.float32)


def fd1_half_weights(space_order, h):
    """Half-node first-derivative weights/h for offsets (-R/2+1..R/2) about x+h/2
    (tools.py:289-297 with fd_order=so/2, x0=x+h/2)."""
    from sympy import finite_diff_weights, Rational
    R = space_order // 2
    offs = list(range(-R // 2 + 1, R // 2 + 1))
    w = finite_diff_weights(1, offs, Rational(1, 2))[-1][-1]
    return np.array([float(c.evalf(9)) / float(h) for c in w], dtype=np.float32)


def critical_dt(space_order, ndim, h_min, vp_max, eps_max=None, dtype=np.float32):
    """examples/seismic/model.py:353-382"""
    from sympy import finite_diff_weights
    c = finite_diff_weights(2, range(-space_order, space_order + 1), 0)[-1][-1]
    coeff = np.sqrt(4.0 / float(ndim * sum(abs(float(x)) for x in c)))
    scale = np.sqrt(1 + 2 * eps_max) if eps_max is not None else 1
    return dtype("%.3e" % (coeff * h_min / (scale * vp_max)))


def damp_field(shape, nbl, spacing, so, fs=False):
    """Absorbing profile with halo `so` (zeros in the halo) — examples/seismic/model.py:25-63.
    fs: free surface, no layer on the low side of the last axis (model.py:45, :166-172)."""
    out = np.zeros(shape, dtype=np.float64)
    coeff = 1.5 * np.log(1.0 / 0.001) / nbl
    for ax, h in enumerate(spacing):
        n = shape[ax]
        prof = np.zeros(n)
        for i in range(nbl):
            pos = abs((nbl - i + 1) / float(nbl))
            val = coeff * (pos - np.sin(2 * np.pi * pos) / (2 * np.pi))
            if not (fs and ax == len(shape) - 1):
                prof[i] += val / float(h)
            prof[n - 1 - i] += val / float(h)
        sh = [1] * len(shape)
        sh[ax] = n
        out += prof.reshape(sh)
    return np.pad(out.astype(np.float32), so)


def ricker(f0, time_values, t0=None, a=1.0):
    """examples/seismic/source.py:284-289"""
    t0 = t0 or 1.0 / f0
    r = np.pi * f0 * (time_values - t0)
    return a * (1 - 2. * r ** 2) * np.exp(-r ** 2)


def time_axis(t0, tn, dt):
    """examples/seismic/source.py:52-63: num = ceil((tn - t0 + dt)/dt); values = linspace."""
    num = int(np.ceil((tn - t0 + dt) / dt))
    stop = dt * (num - 1) + t0
    return num, np.linspace(t0, stop, num)


def tabulate(coords, origin, spacing, r=1, interpolation='linear', dtype=np.float32):
    """Base cell + per-dim weights, fp64 on the host (devito/operations/interpolators.py:674-718)."""
    f64 = lambda v: np.float64(np.format_float_positional(v, unique=True, trim='0'))
    sp = np.array([f64(h) for h in spacing])
    og = np.array([f64(o) for o in origin])
    pos = (np.asarray(coords, dtype=np.float64) - og) / sp
    gp = np.floor(pos).astype(np.int32)
    frac = pos - np.floor(pos)
    ws = []
    for j in range(pos.shape[1]):
        if interpolation == 'linear':
            w = np.empty((pos.shape[0], 2), dtype=dtype)
            w[:, 0] = 1.0 - frac[:, j]
            w[:, 1] = frac[:, j]
        else:
            from scipy.special import i0
            b = {2: 2.94, 3: 4.53, 4: 4.14, 5: 5.26, 6: 6.40, 7: 7.51, 8: 8.56, 9: 9.56, 10: 10.64}[r]
            w = np.zeros((pos.shape[0], 2 * r), dtype=dtype)
            for ri in range(2 * r):
                rpos = ri - r + 1 - frac[:, j]
                w[:, ri] = i0(b * np.sqrt(1 - (rpos / r) ** 2)) / i0(b) * np.sinc(rpos)
        ws.append(w)
    return gp, ws


def layered_vp(shape, nlayers, vp_top=1.5, vp_bottom=3.5, dtype=np.float32):
    """Preset `layers-isotropic` (examples/seismic/preset_models.py:120-133)."""
    v = np.empty(shape, dtype=dtype)
    v[:] = vp_top
    vals = np.linspace(vp_top, vp_bottom, nlayers)
    for i in range(1, nlayers):
        v[..., i * int(shape[-1] / nlayers):] = vals[i]
    return v
