"""world_size-2 tests. `test_decomposition_host_side` runs on CPU (gloo). The GPU test needs two
devices; it compares the slab-decomposed NCCL run with the single-GPU run on the same inputs."""
import os
import socket
import subprocess
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))


def _free_port():
    s = socket.socket()
    s.bind(('127.0.0.1', 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _launch(args, timeout=600, extra_env=None, nproc=2):
    cmd = [sys.executable, '-m', 'torch.distributed.run', '--nnodes=1', '--nproc-per-node', str(nproc),
           '--master-addr', '127.0.0.1', '--master-port', str(_free_port()),
           os.path.join(HERE, 'dist_worker.py')] + args
    env = dict(os.environ)
    env['OMP_NUM_THREADS'] = '1'
    env.update(extra_env or {})
    return subprocess.run(cmd, capture_output=True, text=True, timeout=timeout, env=env)


def test_decomposition_host_side():
    # both ranks stay on the host: with a device visible, a rank would bind to GPU <LOCAL_RANK>, which a
    # machine with fewer GPUs than ranks does not have
    r = _launch(['host'], extra_env={'CUDA_VISIBLE_DEVICES': ''})
    assert 'DIST-HOST-OK' in r.stdout, r.stdout[-2000:] + r.stderr[-4000:]


# halo data paths: the halo step fused into the sweep kernel (default for the isotropic TMA kernel), the
# copy-based peer-memory path (TTI, generic kernels, B2_HALO_FUSED=0) and the complete NCCL path
_PATHS = [('p2p-fused', {}), ('p2p-copy', {'B2_HALO_FUSED': '0'}), ('nccl', {'B2_HALO': 'nccl'})]
if os.environ.get('B2_TEST_EXPERIMENTAL') == '1':
    _PATHS.append(('p2p-copy-async', {'B2_HALO_FUSED': '0', 'B2_P2P_ASYNC': '1'}))


def _decomposed_vs_single(kind, tol, env, nproc):
    r = _launch(['gpu', kind], extra_env=env, nproc=nproc)
    assert 'DIST-GPU-DONE' in r.stdout, r.stdout[-2000:] + r.stderr[-4000:]
    sys.path.insert(0, HERE)
    from helpers import rel_linf
    from dist_cases import run_case, AXIS
    res, _ = run_case(kind, nproc)
    for name, want in res.items():
        want = np.asarray(want)
        if AXIS[name] is None:
            got = np.load(f'/tmp/b2_dist_{kind}_rec.npy')
        else:
            got = np.concatenate([np.load(f'/tmp/b2_dist_{kind}_{name}_{r}.npy') for r in range(nproc)], axis=AXIS[name])
        assert got.shape == want.shape, (name, got.shape, want.shape)
        assert rel_linf(got, want) < tol, (kind, name, rel_linf(got, want))


@pytest.mark.gpu
@pytest.mark.parametrize('path,env', _PATHS, ids=[p for p, _ in _PATHS])
@pytest.mark.parametrize('kind,tol', [('iso', 1e-5), ('tti', 1e-4)])
def test_two_gpu_halo_exchange_matches_single_gpu(kind, tol, path, env):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    _decomposed_vs_single(kind, tol, env, 2)


@pytest.mark.gpu
@pytest.mark.parametrize('path,env', _PATHS, ids=[p for p, _ in _PATHS])
@pytest.mark.parametrize('kind,tol', [('iso', 1e-5), ('tti', 1e-4)])
def test_four_gpu_halo_exchange_matches_single_gpu(kind, tol, path, env):
    """Ranks 1 and 2 have neighbours on both sides (tests/test_mpi.py of the reference runs its halo tests at
    4 ranks for the same reason)."""
    import torch
    if torch.cuda.device_count() < 4:
        pytest.skip("needs 4 GPUs")
    _decomposed_vs_single(kind, tol, env, 4)


# the schemes that ride on the isotropic update: free surface (copy path: the surface rows are redone after the
# sweep), OT4 (halo of 2*radius planes), Born (two wavefields), gradient (adjoint + imaging), snapshots; and the
# array-parameter TTI kernel (per-point factor tables whose halo planes come with each rank's slab of the model)
_SCHEMES = [('ttiarr', {}), ('ttiarr', {'B2_HALO': 'nccl'}), ('iso12', {}), ('stream', {}), ('fs', {}), ('ot4', {}), ('born', {}), ('grad', {}), ('snap', {}), ('ot4', {'B2_HALO': 'nccl'}),
            ('born', {'B2_HALO': 'nccl'}), ('fs', {'B2_HALO': 'nccl'})]


@pytest.mark.gpu
@pytest.mark.parametrize('kind,env', _SCHEMES, ids=[k + ('-nccl' if e else '') for k, e in _SCHEMES])
def test_two_gpu_schemes_match_single_gpu(kind, env):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    from dist_cases import TOL
    _decomposed_vs_single(kind, TOL[kind], env, 2)
