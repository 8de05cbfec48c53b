"""Compile and call the reference-generated C in oracle/_ref/ (see oracle/make_ref.py).
TEST/BENCH INFRASTRUCTURE ONLY — CPU baseline `kind: "reference"`."""
import ctypes
import json
import os
import subprocess
from ctypes import POINTER, Structure, c_double, c_float, c_int, c_ulong, c_void_p

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
REF = os.path.join(HERE, '_ref')

# the reference's CPU flags (devito/arch/compiler.py:216, 482-517)
CFLAGS = ['-O3', '-g', '-fPIC', '-Wall', '-std=c99', '-march=native', '-Wno-unused-result',
          '-Wno-unused-variable', '-Wno-unused-but-set-variable', '-ffast-math', '-fopenmp', '-shared']


class Dataobj(Structure):
    _fields_ = [('data', c_void_p), ('size', POINTER(c_int)), ('nbytes', c_ulong),
                ('npsize', POINTER(c_ulong)), ('dsize', POINTER(c_ulong)), ('hsize', POINTER(c_int)),
                ('hofs', POINTER(c_int)), ('oofs', POINTER(c_int)), ('dmap', c_void_p)]


class Profiler(Structure):
    _fields_ = [('section0', c_double), ('section1', c_double), ('section2', c_double)]


def cpu_signature():
    """Identifies the instruction set `-march=native` compiled for: the binaries travel from the build
    container to the GPU box, whose CPU may differ (an unsupported instruction is a SIGILL, not an error
    code) — a library is rebuilt whenever its recorded signature is not this host's."""
    import hashlib
    try:
        with open('/proc/cpuinfo') as f:
            for line in f:
                if line.startswith('flags'):
                    return hashlib.sha1(' '.join(sorted(line.split(':', 1)[1].split())).encode()).hexdigest()
    except OSError:
        pass
    return 'unknown'


def host_build_path(name, sources, flags=()):
    """Where a library compiled at run time for this host (-march=native) goes: a per-user temporary
    directory, never the source tree, under a name keyed by the sources, the flags and the host's CPU
    (a binary made on another CPU is never loaded)."""
    import hashlib
    import tempfile
    h = hashlib.sha1()
    for path in sources:
        with open(path, 'rb') as f:
            h.update(f.read())
    h.update(' '.join(flags).encode())
    h.update(cpu_signature().encode())
    d = os.path.join(tempfile.gettempdir(), f'devito-b200-oracle-uid{os.getuid()}')
    os.makedirs(d, exist_ok=True)
    return os.path.join(d, f'{name}-{h.hexdigest()[:16]}.so')


def _compile(name):
    src = os.path.join(REF, name + '.c')
    if not os.path.exists(src):
        return None
    so = host_build_path(name, [src], CFLAGS)
    if not os.path.exists(so):
        tmp = f'{so}.{os.getpid()}'
        r = subprocess.run(['gcc'] + CFLAGS + [src, '-lm', '-o', tmp], capture_output=True, text=True)
        if r.returncode != 0:
            return None
        os.replace(tmp, so)
    try:
        return ctypes.CDLL(so)
    except OSError:
        return None


def load_forward(so, kind='iso'):
    name = f'forward_{kind}_so{so}'
    lib = _compile(name)
    if lib is None:
        return None
    with open(os.path.join(REF, name + '.json')) as f:
        meta = json.load(f)
    return lib, meta


def _obj(arr, keep):
    arr = np.ascontiguousarray(arr)
    size = (c_int * arr.ndim)(*arr.shape)
    o = Dataobj()
    o.data = arr.ctypes.data
    o.size = ctypes.cast(size, POINTER(c_int))
    o.nbytes = arr.nbytes
    keep.extend([arr, size, o])
    return o


def run_forward(ref, u, damp, vp, dt, time_m, time_M, src, rec, so, threads, v=None, extra=None):
    """Marshal arguments in the order the reference reports (op.parameters) and call."""
    lib, meta = ref
    fn = getattr(lib, meta['name'])
    keep = []
    n = [s - 2 * so for s in u.shape[1:]]
    arrays = {'u': u, 'v': v, 'damp': damp, 'src': src['data'], 'rec': rec['data'],
              'src_gp': src['gp'], 'rec_gp': rec['gp']}
    for d, nm in enumerate('xyz'):
        arrays[f'src_w{nm}'] = src['w'][d]
        arrays[f'rec_w{nm}'] = rec['w'][d]
    scal = {'vp': c_float(vp), 'dt': c_float(dt), 'time_m': c_int(time_m), 'time_M': c_int(time_M),
            'x_m': c_int(0), 'x_M': c_int(n[0] - 1), 'y_m': c_int(0), 'y_M': c_int(n[1] - 1),
            'z_m': c_int(0), 'z_M': c_int(n[2] - 1), 'z_size': c_int(n[2]),
            'p_src_m': c_int(0), 'p_src_M': c_int(src['data'].shape[1] - 1),
            'p_rec_m': c_int(0), 'p_rec_M': c_int(rec['data'].shape[1] - 1),
            'x0_blk0_size': c_int(16), 'y0_blk0_size': c_int(16),
            'nthreads': c_int(threads), 'nthreads_nonaffine': c_int(threads)}
    for k, val in (extra or {}).items():
        scal[k] = c_float(val)
    timers = Profiler()
    args = []
    for p in meta['parameters']:
        nm = p['name']
        if nm == 'timers':
            args.append(ctypes.byref(timers))
        elif nm in arrays and arrays[nm] is not None and p['is_fn']:
            args.append(ctypes.byref(_obj(arrays[nm], keep)))
        elif nm in scal:
            args.append(scal[nm])
        else:
            raise KeyError(f"refrun: no value for reference parameter {nm!r}")
    rc = fn(*args)
    if rc != 0:
        raise RuntimeError(f"reference kernel returned {rc}")
    return timers
