#!/usr/bin/env python
"""bench.py — headline benchmark of the hot path (driver contract, see DESIGN.md §Measurement).

Metric (BASELINE.json): GPts/s of the 3-D isotropic acoustic forward operator, space_order=8,
on a 1024^3 grid (absorbing layers included: GPts/s counts every grid point the stencil
updates, devito/operator/profiling.py:355-366), fp32, synthetic constant-velocity model,
one Ricker source, 512 receivers sampled every step.

A "step" = one `Operator.apply` of the Forward operator over NT time steps.
  value : whole-job GPts/s with fields resident in HBM when the timed region starts
  e2e   : the same call made with HOST buffers through the C ABI (H2D of u/damp/src and D2H of
          u/rec inside the timed region — the reference's per-apply copy semantics)
  roofline : the stencil kernel's algorithmic bytes (16 B/point) / its mean launch duration
             (CUDA events on the library stream), against MEASURED_PEAKS.json hbm_gbs
  cpu_baseline : the reference's CPU implementation timed on this box's host cores, same grid
  parity_check : outside the timed region, a short propagation on a small grid (decomposed over the
             same N ranks, sources on the slab boundaries) compared with the CPU oracle on the
             undecomposed grid: every halo data path; a failure makes the run exit non-zero
  configs  : short runs of the other BASELINE configs — C3 (so=12, 1024^3), C4 (TTI so=8, 768^3), C4b (TTI so=8
             with array-valued vp/eps/delta/theta/phi, 512^3) at N=1, C5 (so=8, 2048x1024x1024 FIXED, x-slabs =
             strong scaling) at every N

`--dump-outputs DIR` writes what the last timed apply returned (Bench.dump_outputs). The inputs are synthetic
and fixed by the arguments, so two builds run with the same arguments can be compared output for output.

`--impl reference` times the reference's own CPU code path (oracle/_ref = C code emitted by the
reference's code generator for this operator, compiled here with its flags; else the oracle
port) on the SAME grid, a bounded number of time steps per "step".

Multi-GPU (torchrun, one rank per GPU): x-slab decomposition, weak scaling — every rank owns a
1024-plane slab of a (N*1024) x 1024 x 1024 grid. The halo step is fused into the sweep kernel:
boundary planes are stored into the neighbour GPU's halo over NVLink by the CTAs that produce them
(CUDA-IPC peer memory) and ordered by release/acquire flags; `B2_HALO_FUSED=0` selects the
copy-based peer path, `B2_HALO=nccl` NCCL send/recv overlapped with the interior update.
"""
import argparse
import ctypes
import gc
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

B_ALG = {'iso': 16.0, 'tti': 28.0,    # algorithmic bytes / point / step (SURVEY §8d)
         'tti-arrays': 52.0}           # + cx, cy, cz, 1+2eps, sqrt(1+2delta), m/dt^2 tables (DESIGN §3.3a2)
DUMP_SAMPLE = 1 << 20                  # grid points per wavefield in the seeded sample of --dump-outputs


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=4)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--grid', type=int, default=int(os.environ.get('B2_BENCH_GRID', 1024)),
                    help='grid points per dimension incl. absorbing layers')
    ap.add_argument('--nt', type=int, default=int(os.environ.get('B2_BENCH_NT', 256)),
                    help='time steps per Operator.apply')
    ap.add_argument('--space-order', type=int, default=8)
    ap.add_argument('--workload', default='iso', choices=['iso', 'tti', 'tti-arrays'],
                    help="iso: the headline metric; tti: BASELINE config 4 (not the driver's line)")
    ap.add_argument('--scaling', default='weak', choices=['weak', 'strong'],
                    help="strong: BASELINE config 5 as the headline (2048x1024x1024 fixed)")
    ap.add_argument('--no-e2e', action='store_true')
    ap.add_argument('--no-cpu', action='store_true')
    ap.add_argument('--no-extra', action='store_true', help='skip the C3/C4/C5 side runs')
    ap.add_argument('--no-parity', action='store_true')
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help='after the timed steps, write what the last one returned as DIR/<name>.npy (see dump_outputs)')
    a = ap.parse_args()
    if a.steps < 1 or a.warmup < 0:
        ap.error('--steps must be at least 1 and --warmup at least 0')
    return a


def peaks():
    path = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(path):
        with open(path) as f:
            return float(json.load(f)['hbm_gbs']), 'measured'
    return 6650.0, 'fallback'


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region."""
    Q = ('clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,'
         'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,'
         'clocks_event_reasons.sw_power_cap')

    def __init__(self, index=0):
        self.index = index
        self.samples = []
        self._stop = False
        self._t = None

    def _run(self):
        while not self._stop:
            try:
                out = subprocess.run(['nvidia-smi', f'--query-gpu={self.Q}', '--format=csv,noheader,nounits',
                                      '-i', str(self.index)], capture_output=True, text=True, timeout=5).stdout
                parts = [p.strip() for p in out.strip().split(',')]
                if len(parts) >= 6:
                    self.samples.append(parts)
            except Exception:
                pass
            time.sleep(0.2)

    def __enter__(self):
        self._t = threading.Thread(target=self._run, daemon=True)
        self._t.start()
        return self

    def __exit__(self, *a):
        self._stop = True
        self._t.join(timeout=6)

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        sm = sorted(float(s[0]) for s in self.samples)
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        reasons = [n for i, n in enumerate(names) if any(s[2 + i].lower().startswith('active') for s in self.samples)]
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": float(self.samples[0][1]), "reasons": reasons}


# ---------------------------------------------------------------------------------------------
# CPU arm: the reference's implementation of the path on the host cores
# ---------------------------------------------------------------------------------------------
def usable_cores():
    """Host threads this process may actually use: affinity mask capped by the cgroup CPU quota."""
    try:
        n = len(os.sched_getaffinity(0))
    except AttributeError:
        n = os.cpu_count() or 1
    try:
        with open('/sys/fs/cgroup/cpu.max') as f:
            q, per = f.read().split()
        if q != 'max':
            n = max(1, min(n, int(float(q) / float(per) + 0.5)))
    except Exception:
        pass
    return n


_cpu_problem_cache = {}


def _cpu_problem(so, grid_n, nts):
    """Inputs of the CPU arm on a grid_n^3 grid (absorbing layers included), built with the oracle's
    host-side restatements; 1 Ricker source, 512 receivers, like the GPU arm."""
    key = (so, grid_n, nts)
    if key in _cpu_problem_cache:
        return _cpu_problem_cache[key]
    from oracle import oracle as O
    nbl = 40 if grid_n >= 160 else 8
    n = grid_n - 2 * nbl
    h = 10.0
    spacing = (np.float32(h),) * 3
    origin = tuple(np.float32(-nbl * h) for _ in range(3))
    dt = float(O.critical_dt(so, 3, h, 1.5))
    damp = O.damp_field((grid_n,) * 3, nbl, spacing, so)
    dom = (n - 1) * h
    src_c = np.array([[dom * .5, dom * .5, h]])
    rec_c = np.array([[x, y, 2 * h] for x in np.linspace(0, dom, 32) for y in np.linspace(0, dom, 16)])
    sgp, sw = O.tabulate(src_c.astype(np.float32), origin, spacing, 1, 'linear')
    rgp, rw = O.tabulate(rec_c.astype(np.float32), origin, spacing, 1, 'linear')
    tvals = np.arange(nts, dtype=np.float64) * dt
    src = dict(data=np.ascontiguousarray(O.ricker(0.010, tvals).astype(np.float32).reshape(nts, 1)), gp=sgp, w=sw, r=1)
    rec = dict(data=np.zeros((nts, len(rec_c)), dtype=np.float32), gp=rgp, w=rw, r=1)
    u = np.zeros((3,) + (grid_n + 2 * so,) * 3, dtype=np.float32)
    p = dict(u=u, damp=damp, dt=dt, w=[O.fd2_weights(so, h)] * 3)
    _cpu_problem_cache.clear()                      # one resident CPU problem at a time (18 GB at 1024^3)
    _cpu_problem_cache[key] = (p, src, rec)
    return _cpu_problem_cache[key]


def _cpu_run_once(so, grid_n, nt, threads):
    from oracle import oracle as O
    from oracle import refrun
    p, src, rec = _cpu_problem(so, grid_n, 512)
    ref = refrun.load_forward(so)
    t0 = time.perf_counter()
    if ref is not None:
        kind = 'reference'
        refrun.run_forward(ref, p['u'], p['damp'], 1.5, p['dt'], 1, nt, src, rec, so, threads)
    else:
        kind = 'port'
        os.environ['OMP_NUM_THREADS'] = str(threads)
        O.iso_forward(p['u'], so, p['w'], p['dt'], 1, nt, damp=p['damp'], vp=1.5, src=src, rec=rec, fast=True)
    return time.perf_counter() - t0, kind


_cpu_threads_choice = {}


def cpu_reference_run(so, grid_n, budget_s=12.0):
    """Time the reference's CPU code path on a bounded sample of the workload: the same operator
    (iso acoustic, same space order, source + 512 receivers) on the SAME grid_n^3 grid, fewer time
    steps. The thread count is the best of a short probe over {all usable cores, 1/2, 1/4, ...}
    (the reference's own advice is one thread per physical core, benchmarks/user/README.md:22-64);
    the number of time steps is then sized to ~budget_s seconds.
    Returns (GPts/s, kind, sample, cores, seconds)."""
    cores = usable_cores()
    key = (so, grid_n)
    if key not in _cpu_threads_choice:
        cands = sorted({max(1, cores), max(1, cores // 2), max(1, cores // 4), min(cores, 16), min(cores, 8)},
                       reverse=True)
        best = None
        _cpu_run_once(so, grid_n, 1, cands[0])                          # build / first touch
        for c in cands:
            el, _ = _cpu_run_once(so, grid_n, 2, c)
            if best is None or el < best[0]:
                best = (el, c)
        _cpu_threads_choice[key] = best[1], best[0] / 2
    threads, per_step = _cpu_threads_choice[key]
    nt = int(max(2, min(500, budget_s / max(per_step, 1e-4))))
    el, kind = _cpu_run_once(so, grid_n, nt, threads)
    pts = float(grid_n) ** 3 * nt
    sample = (f"iso so={so} {grid_n}^3 x {nt} time steps (same operator, same grid, fewer steps), {threads} of "
              f"{cores} usable host threads")
    return pts / el / 1e9, kind, sample, threads, el


def host_fits(grid_n, so):
    """The CPU arm needs u (3 slots) + damp on the host: ~18 GB at 1024^3."""
    need = 4.0 * (grid_n + 2 * so) ** 3 * 4 * 1.15
    try:
        with open('/proc/meminfo') as f:
            for line in f:
                if line.startswith('MemAvailable'):
                    return float(line.split()[1]) * 1024 > need + (8 << 30)
    except OSError:
        pass
    return True


def run_reference_arm(a):
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    G = a.grid if host_fits(a.grid, a.space_order) else 384
    vals = []
    budget = max(3.0, min(15.0, 150.0 / max(1, a.warmup + a.steps)))   # whole arm within minutes
    for i in range(a.warmup + a.steps):
        gp, kind, sample, cores, el = cpu_reference_run(a.space_order, G, budget_s=budget)
        if i >= a.warmup:
            vals.append((gp, el))
    value = float(np.mean([v for v, _ in vals]))
    ms = float(np.mean([e for _, e in vals])) * 1e3
    line = {"impl": "reference", "metric": "GPts/s (3D isotropic acoustic forward, so=%d, %d^3 per GPU)" % (a.space_order, a.grid),
            "value": value, "unit": "GPts/s", "n_gpus": a.gpus, "steps": a.steps, "warmup": a.warmup,
            "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"3D isotropic acoustic so={a.space_order}, grid {G}x{G}x{G} (nbl=40 included), "
                                   f"1 Ricker source, 512 receivers, constant vp=1.5; the reference's CPU (OpenMP) "
                                   f"path on a bounded sample: {sample}",
                       "l2": "inputs larger than the CPU caches"},
            "cpu_baseline": {"value": value, "unit": "GPts/s", "cores": cores, "kind": kind, "sample": sample},
            "e2e": {"value": value, "unit": "GPts/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------
# B200 arm
# ---------------------------------------------------------------------------------------------
class Bench:
    def __init__(self, a):
        import torch
        import torch.distributed as dist
        import devito_b200 as dv
        from devito_b200 import _lib
        self.a, self.torch, self.dist, self.dv = a, torch, dist, dv
        world = dv.init_distributed()
        self.rank, self.nranks = world.rank, world.size
        self.local = int(os.environ.get('LOCAL_RANK', '0'))
        torch.cuda.set_device(self.local)
        dv.configuration['deviceid'] = self.local
        self.dev = torch.device('cuda', self.local)
        self.L = _lib.lib()
        from devito_b200.numa import bind_to_gpu
        self.numa = bind_to_gpu(self.local)          # pinned host buffers on the GPU's own socket
        # The library enqueues on torch's current stream so that CUDA events recorded on that stream
        # bracket exactly its work (torch.cuda.Event only sees torch's current stream).
        self.stream = torch.cuda.Stream(device=self.dev)
        torch.cuda.set_stream(self.stream)
        self.L.b2_set_stream(ctypes.c_void_p(self.stream.cuda_stream))

    def barrier(self):
        self.torch.cuda.synchronize()
        if self.nranks > 1:
            self.dist.barrier()
            self.torch.cuda.synchronize()

    def timed(self, fn, reps):
        torch = self.torch
        self.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        dev = e0.elapsed_time(e1) * 1e-3
        self.barrier()
        # device time between the two events (includes host gaps between applies); max over ranks
        t = torch.tensor([dev], dtype=torch.float64, device=self.dev)
        if self.nranks > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t[0].item())

    def workload(self, kind, so, shape_total, NT):
        """Model + solver + fields for a `shape_total` grid (absorbing layers included), x-slabs over
        the ranks."""
        dv = self.dv
        from devito_b200.seismic import (SeismicModel, AcquisitionGeometry, AcousticWaveSolver,
                                         AnisotropicWaveSolver)
        nbl = 40
        shape = tuple(s - 2 * nbl for s in shape_total)
        tti = kind.startswith('tti')
        extra = dict(epsilon=.3, delta=.2, theta=.7, phi=.35) if tti else {}
        vp = 1.5
        if kind == 'tti-arrays':
            # array-valued vp / epsilon / delta / theta / phi (the reference's `layers-tti` shape of problem, here
            # with lateral variation as well): per-point tables instead of scalars in the kernel
            ax = [np.linspace(0., 1., n, dtype=np.float32) for n in shape]
            gx, gy, gz = ax[0][:, None, None], ax[1][None, :, None], ax[2][None, None, :]
            vp = (1.5 + 0.3 * gx + 0.2 * gy + 1.5 * gz).astype(np.float32)
            extra = dict(epsilon=(0.05 + 0.25 * gz + 0.0 * gx + 0.0 * gy).astype(np.float32),
                         delta=(0.02 + 0.1 * gz + 0.05 * gx + 0.0 * gy).astype(np.float32),
                         theta=(0.2 + 0.5 * gz + 0.2 * gx * gy).astype(np.float32),
                         phi=(0.1 + 0.3 * gy + 0.2 * gz + 0.0 * gx).astype(np.float32))
        model = SeismicModel(origin=(0., 0., 0.), spacing=(10., 10., 10.), shape=shape, space_order=so,
                             vp=vp, nbl=nbl, bcs="damp", topology=('*', 1, 1) if self.nranks > 1 else None,
                             **extra)
        dt = model.critical_dt
        tn = float(dt) * (NT + 0.5)                    # geometry.nt = NT + 2, NT time steps per apply
        src_c = np.array([[model.domain_size[0] * .5, model.domain_size[1] * .5, 10.0]])
        rx = np.linspace(0, model.domain_size[0], 32)
        ry = np.linspace(0, model.domain_size[1], 16)
        rec_c = np.array([[x, y, 20.0] for x in rx for y in ry])           # 512 receivers
        geometry = AcquisitionGeometry(model, rec_c, src_c, t0=0.0, tn=tn, src_type='Ricker', f0=0.010)
        solver = (AnisotropicWaveSolver if tti else AcousticWaveSolver)(model, geometry, space_order=so)
        u = dv.TimeFunction(name='u', grid=model.grid, time_order=2, space_order=so)
        v = dv.TimeFunction(name='v', grid=model.grid, time_order=2, space_order=so) if tti else None
        w = dict(kind=kind, so=so, model=model, geometry=geometry, solver=solver, u=u, v=v,
                 src=geometry.src, rec=geometry.rec, src_x=nbl + (shape[0] - 1) // 2,
                 nt_steps=geometry.nt - 2, dt=float(dt),
                 shape_total=tuple(shape_total), pts_step=float(np.prod(shape_total)) * (geometry.nt - 2),
                 fkw=dict(v=v) if tti else {})
        return w

    def run_resident(self, w, steps, warmup, clocks=True, dump=None):
        L = self.L
        fn = lambda: w['solver'].forward(src=w['src'], rec=w['rec'], u=w['u'], **w['fkw'])
        for _ in range(warmup):
            fn()
        launches0 = L.b2_launch_count()
        # timed region: K applies, nothing else on the stream (per-launch CUDA events would sit between the
        # kernels of every time step and stretch the step by ~1 %: they are recorded in a second pass below)
        if clocks:
            with ClockSampler(self.local) as clk:
                t = self.timed(fn, steps)
            clocks = clk.summary()
        else:
            t = self.timed(fn, steps)
            clocks = None
        if dump:
            self.dump_outputs(w, dump)
        launches = int(L.b2_launch_count() - launches0)
        # second pass, same applies: CUDA events around every stencil launch -> mean launch duration
        L.b2_kernel_timing_enable(1)
        L.b2_kernel_timing_reset()
        t_k = self.timed(fn, min(steps, 2))
        nl = ctypes.c_int(0)
        k_ms = L.b2_kernel_timing_ms(ctypes.byref(nl))
        L.b2_kernel_timing_enable(0)
        launches = int(L.b2_launch_count() - launches0)
        out = {"value": w['pts_step'] * steps / t / 1e9, "ms_per_step": t / steps * 1e3, "launches": launches,
               "clocks": clocks}
        # roofline of the dominant kernel: this rank's launch (the whole local slab in one launch on the
        # fused / single-GPU paths); the slowest rank's launch time bounds the job
        peak, peak_kind = peaks()
        pts_launch = float(np.prod(w['model'].grid.shape))
        torch = self.torch
        kt = torch.tensor([k_ms if nl.value else 0.0, float(pts_launch)], dtype=torch.float64, device=self.dev)
        if self.nranks > 1:
            self.dist.all_reduce(kt, op=self.dist.ReduceOp.MAX)
        k_ms_max, pts_launch = float(kt[0].item()), float(kt[1].item())
        if nl.value and k_ms_max > 0:
            ach = B_ALG[w['kind']] * pts_launch / (k_ms_max * 1e-3) / 1e9
            out['roofline'] = {"bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                               "traffic": None, "peak_source": f"MEASURED_PEAKS.json hbm_gbs ({peak_kind})",
                               "kernel": "k_tti_*" if w['kind'].startswith('tti') else "k_iso_tma",
                               "launch_ms": k_ms_max, "launches_timed": int(nl.value),
                               "timed_in": "a second pass of %d applies with CUDA events around every stencil launch "
                                           "(%.1f ms per apply with the events, %.1f ms without)"
                                           % (min(steps, 2), t_k / min(steps, 2) * 1e3, t / steps * 1e3),
                               "scope": "per GPU (slowest rank's mean launch)" if self.nranks > 1 else "single GPU",
                               "points_per_launch": pts_launch, "bytes_per_point": B_ALG[w['kind']]}
        else:
            out['roofline'] = None
        return out

    def dump_outputs(self, w, d):
        """What the last timed apply returned to its caller, as float32 `DIR/<name>.npy`: the receiver traces
        `rec` in full and, of each wavefield (`u`, and `v` for TTI; all three time slots), the x-plane through the
        source `<f>_plane_x` and the grid points of a fixed seeded sample `<f>_sample` (a whole field is
        gigabytes). Under decomposition the sample is of each rank's slab (`<f>_sample_rank<r>`) and the plane
        comes from the rank that owns it."""
        os.makedirs(d, exist_ok=True)
        out = {'rec': w['rec'].data_ro_domain} if self.rank == 0 else {}
        lo, hi = w['model'].grid.distributor.x_range if self.nranks > 1 else (0, w['u'].shape[1])
        sfx = f'_rank{self.rank}' if self.nranks > 1 else ''
        for name in ('u', 'v'):
            if w[name] is None:
                continue
            a = w[name].data_ro_domain                         # (3, x, y, z): read-only, the device copy stays valid
            if lo <= w['src_x'] < hi:
                out[f'{name}_plane_x'] = a[:, w['src_x'] - lo]
            pts = np.unique(np.random.default_rng(2024 + self.rank).integers(0, np.prod(a.shape[1:]), DUMP_SAMPLE))
            out[f'{name}_sample{sfx}'] = a[(slice(None),) + np.unravel_index(pts, a.shape[1:])]
        for name, arr in out.items():
            np.save(os.path.join(d, name + '.npy'), np.ascontiguousarray(arr, dtype=np.float32))

    def run_e2e(self, w, steps, warmup):
        u, model, src, rec = w['u'], w['model'], w['src'], w['rec']
        hostcall = lambda: w['solver'].forward(src=src, rec=rec, u=u, resident=False, **w['fkw'])
        _ = u.data_with_halo          # materialise (pinned) host copies outside the timed region
        _ = model.damp.data_with_halo
        for _ in range(min(warmup, 1) or 1):
            hostcall()
        t = self.timed(hostcall, steps)
        prof = (ctypes.c_double * 5)()
        self.L.b2_last_call_profile(prof)
        h2d = u.storage.host_ro.nbytes + model.damp.storage.host_ro.nbytes + src.data.nbytes
        d2h = u.storage.host_ro.nbytes + rec.data.nbytes
        streamed = prof[4] == 1.0
        return {"value": w['pts_step'] * steps / t / 1e9, "unit": "GPts/s",
                "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                "ms_per_step": t / steps * 1e3,
                "mode": (("streamed: chunks (x planes on one GPU, y rows under x-slab decomposition) uploaded / downloaded on "
                          "copy streams while a skewed sweep time-steps the chunks already on the device"
                          + ("; every sub-launch is a fused halo step" if self.nranks > 1 else "")) if streamed else
                         "serial: host->device, time loop, device->host on one stream"),
                "last_call_ms": {"before_loop": prof[0], "time_loop": prof[1], "after_loop": prof[2], "call": prof[3]},
                "pinned_host": bool(getattr(u.storage, '_pinned', None) is not None),
                "numa": self.numa}

    def release(self, w):
        w.clear()
        gc.collect()
        self.L.b2_staging_cache_release()
        self.torch.cuda.empty_cache()


# ---------------------------------------------------------------------------------------------
# parity check on the launch configuration the bench runs (every rank, every halo data path)
# ---------------------------------------------------------------------------------------------
def parity_check(b, so=8, tol=1e-5):
    """A short propagation on a small grid, decomposed over the bench's own ranks with sources sitting ON
    the slab boundaries, against the CPU oracle run on the undecomposed grid: every rank compares the
    three time slots of its slab (L-inf relative to the global maximum), rank 0 the receiver traces.
    Reference for the decomposed semantics: tests/test_mpi.py:3373-3457 (decomposed == serial)."""
    from oracle import oracle as O
    from devito_b200.seismic import SeismicModel, AcquisitionGeometry, AcousticWaveSolver
    dv, torch, dist = b.dv, b.torch, b.dist
    N, rank = b.nranks, b.rank
    nbl, h, slab = 8, 10.0, 48
    total = (N * slab, 72, 72)
    shape = tuple(s - 2 * nbl for s in total)
    dom = [(s - 1) * h for s in shape]
    # sources: one per internal slab boundary (half a cell off the boundary plane), plus the grid centre
    xs = [((r + 1) * slab - nbl - 0.5) * h for r in range(N - 1)] + [dom[0] * .5 + 3.3]
    src_c = np.array([[x, dom[1] * (0.35 + 0.3 * (i % 2)), dom[2] * .45] for i, x in enumerate(xs)])
    rec_c = np.array([[x, dom[1] * .5, 2 * h] for x in np.linspace(0, dom[0], 16 * N + 1)])
    NT = 90
    results = {}
    paths = [('single', {})] if N == 1 else [('fused-p2p', {}), ('copy-p2p', {'B2_HALO_FUSED': '0'}),
                                            ('nccl', {'B2_HALO': 'nccl'})]
    # oracle on the undecomposed grid (identical on every rank; ~1 s)
    spacing = (np.float32(h),) * 3
    origin = tuple(np.float32(-nbl * h) for _ in range(3))
    dt = float(O.critical_dt(so, 3, h, 1.5))
    nt, tvals = O.time_axis(0.0, dt * (NT + 0.5), dt)
    damp = O.damp_field(total, nbl, spacing, so)
    sgp, sw = O.tabulate(src_c.astype(np.float32), origin, spacing, 1, 'linear')
    rgp, rw = O.tabulate(rec_c.astype(np.float32), origin, spacing, 1, 'linear')
    amp = O.ricker(0.010, tvals).astype(np.float32)
    sdata = np.stack([amp * (1.0 + 0.25 * i) for i in range(len(src_c))], axis=1).astype(np.float32)
    ou = np.zeros((3,) + tuple(s + 2 * so for s in total), dtype=np.float32)
    orec = dict(data=np.zeros((nt, len(rec_c)), dtype=np.float32), gp=rgp, w=rw, r=1)
    O.iso_forward(ou, so, [O.fd2_weights(so, h)] * 3, dt, 1, nt - 2, damp=damp, vp=1.5,
                  src=dict(data=np.ascontiguousarray(sdata), gp=sgp, w=sw, r=1), rec=orec)
    umax = float(np.abs(ou).max())
    rmax = float(np.abs(orec['data']).max())
    ok = True
    for name, env in paths:
        old = {k: os.environ.get(k) for k in env}
        os.environ.update(env)
        try:
            model = SeismicModel(origin=(0., 0., 0.), spacing=(h, h, h), shape=shape, space_order=so, vp=1.5,
                                 nbl=nbl, bcs="damp", topology=('*', 1, 1) if N > 1 else None)
            assert abs(float(model.critical_dt) - dt) < 1e-6 * dt
            geometry = AcquisitionGeometry(model, rec_c, src_c, t0=0.0, tn=dt * (NT + 0.5), src_type='Ricker', f0=0.010)
            assert geometry.nt == nt
            src = geometry.src
            src.data[:] = sdata
            solver = AcousticWaveSolver(model, geometry, space_order=so)
            rec, u, _ = solver.forward(src=src)
            lo, hi = model.grid.distributor.x_range if N > 1 else (0, total[0])
            mine = np.asarray(u.data)
            want = ou[:, so + lo:so + hi, so:-so, so:-so]
            eu = float(np.abs(mine.astype(np.float64) - want).max()) / umax
            er = float(np.abs(np.asarray(rec.data, dtype=np.float64) - orec['data']).max()) / rmax
            t = torch.tensor([eu, er], dtype=torch.float64, device=b.dev)
            if N > 1:
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
            eu, er = float(t[0].item()), float(t[1].item())
            halo = getattr(u.storage, 'p2p_registered', False)
            results[name] = {"u_linf": eu, "rec_linf": er, "ok": bool(eu < tol and er < tol),
                             "peer_memory": bool(halo)}
            ok = ok and results[name]["ok"]
            del solver, model, geometry, u, rec, src
        finally:
            for k, v in old.items():
                if v is None:
                    os.environ.pop(k, None)
                else:
                    os.environ[k] = v
    gc.collect()
    return {"ok": ok, "ranks": N, "tol": tol, "grid": list(total), "time_steps": nt - 2,
            "sources": len(src_c), "receivers": len(rec_c),
            "against": "CPU oracle (oracle/oracle.c) on the undecomposed grid; every rank checks the 3 time "
                       "slots of its slab, receivers after the merge",
            "u_linf": max(r["u_linf"] for r in results.values()),
            "rec_linf": max(r["rec_linf"] for r in results.values()),
            "path": list(results), "paths": results}


def main():
    a = parse()
    if a.impl == 'reference':
        run_reference_arm(a)
        return
    b = Bench(a)
    rank, nranks = b.rank, b.nranks
    so, G, NT = a.space_order, a.grid, a.nt

    parity = None
    if not a.no_parity:
        parity = parity_check(b)

    strong = a.scaling == 'strong'
    if strong:
        total = (2 * G, G, G)                                # BASELINE config 5: 2048 x 1024 x 1024, fixed
    else:
        total = (nranks * G, G, G)                           # every rank owns a G-plane slab
    w = b.workload(a.workload, so, total, NT)
    res = b.run_resident(w, a.steps, a.warmup, dump=a.dump_outputs)
    halo_path = None
    if nranks > 1:
        halo_path = ("NCCL send/recv" if not getattr(w['u'].storage, 'p2p_registered', False) else
                     "peer-memory copies over NVLink (CUDA IPC + device flags)"
                     if os.environ.get('B2_HALO_FUSED') == '0' or a.workload.startswith('tti') else
                     "fused into the sweep kernel: boundary planes stored into the neighbour's halo over NVLink "
                     "(CUDA IPC) by the CTAs that produce them, release/acquire flags")
    nvlink = None
    if nranks > 1:
        R = so // 2
        per_plane = (G + 2 * so) ** 2 * 4 if a.workload == 'iso' else 2 * (G + 2 * so) ** 2 * 4
        nvlink = {"bytes_per_step_per_interior_rank": 2 * R * per_plane,
                  "planes_per_side": R}
    roof = res['roofline']
    if roof is not None:
        try:   # dram__bytes_read+write per launch from the committed `ncu --set full` capture
            with open(os.path.join(ROOT, 'profiles', 'traffic.json')) as f:
                tj = json.load(f)
            roof['traffic'] = tj.get(f"{a.workload}_so{so}_{G}")
            roof['traffic_source'] = tj.get('source', 'profiles/traffic.json (ncu --set full capture of this kernel, not this run)')
        except Exception:
            roof['traffic'] = None

    e2e = None
    if not a.no_e2e:
        e2e = b.run_e2e(w, a.steps, a.warmup)
    nt_steps, dt = w['nt_steps'], w['dt']
    b.release(w)

    # ---- the other BASELINE configs, short runs (same timing rules, fewer time steps) ----
    extra = {}
    if not a.no_extra and a.workload == 'iso' and not strong:
        def side(kind, so_, total_, nt_, reps=3):
            ww = b.workload(kind, so_, total_, nt_)
            r = b.run_resident(ww, reps, 3)
            r['config'] = (f"{ {'tti': 'TTI', 'tti-arrays': 'TTI, array-valued vp/eps/delta/theta/phi'}.get(kind, 'iso acoustic')} so={so_}, grid {'x'.join(map(str, total_))}, "
                           f"{ww['nt_steps']} time steps per apply, {reps} applies after 3 warm-up")
            r['unit'] = 'GPts/s'
            b.release(ww)
            return r
        if nranks == 1:
            extra['C3_iso_so12_1024'] = side('iso', 12, (G, G, G), 64)
            extra['C4_tti_so8_768'] = side('tti', 8, (768, 768, 768), 64)
            extra['C4b_tti_arrays_so8_512'] = side('tti-arrays', 8, (512, 512, 512), 32, reps=2)
        c5 = side('iso', 8, (2 * G, G, G), 96)
        c5['scaling'] = 'strong'
        extra['C5_iso_so8_2048x1024x1024_strong'] = c5

    cpu = None
    if rank == 0 and nranks == 1 and not a.no_cpu:
        try:
            Gc = G if host_fits(G, so) else 384
            gp, kind, sample, cores, el = cpu_reference_run(so, Gc, budget_s=10.0)
            cpu = {"value": gp, "unit": "GPts/s", "cores": cores, "kind": kind, "sample": sample}
        except Exception as e:                                           # never hide the GPU number
            cpu = {"value": None, "unit": "GPts/s", "cores": None, "kind": "port", "sample": f"failed: {e}"}

    if rank == 0:
        tti = a.workload.startswith('tti')
        gx = total[0]
        line = {"metric": "GPts/s (3D %s forward, so=%d, %d^3 per GPU)" % ("TTI" if tti else "isotropic acoustic", so, G),
                "value": res['value'], "unit": "GPts/s", "n_gpus": nranks, "steps": a.steps, "warmup": a.warmup,
                "ms_per_step": res['ms_per_step'], "higher_is_better": True, "scaling": a.scaling,
                "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": {"workload": f"3D {'TTI centred' if tti else 'isotropic acoustic'} so={so}, grid {gx}x{G}x{G} "
                                       f"(nbl=40 included), {nt_steps} time steps per apply, 1 Ricker source, "
                                       f"512 receivers, constant vp=1.5",
                           "decomposition": f"x-slabs over {nranks} GPU(s)" if nranks > 1 else "single GPU",
                           "halo": halo_path, "nvlink": nvlink,
                           "l2": "inputs (18 GB/GPU) larger than L2; no flush needed",
                           "time_steps_per_apply": nt_steps, "dt": dt},
                "clocks": res['clocks'], "gpu_launches": res['launches'],
                "roofline": roof, "cpu_baseline": cpu, "e2e": e2e,
                "parity_check": parity, "configs": extra or None}
        print(json.dumps(line), flush=True)
    ok = parity is None or parity['ok']
    if nranks > 1:
        from devito_b200.distributed import finalize_distributed
        finalize_distributed()
    if not ok:
        sys.stderr.write(f"bench.py: parity_check FAILED: {json.dumps(parity)}\n")
        sys.exit(3)


if __name__ == '__main__':
    main()
