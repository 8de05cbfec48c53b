"""Golden vectors for tests/test_refrun.py: the reference's own generated C (oracle/_ref, emitted by
oracle/make_ref.py and compiled by oracle/refrun.py) run on that test's small isotropic problem.

    python oracle/make_ref.py && python oracle/make_refgen_golden.py

The whole wavefield would not fit a small fixture, so each file keeps the receiver traces in full, the
x-plane of u through the source, u at a fixed seeded sample of points (halo included) and max|u|.
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, os.path.join(HERE, '..', 'tests'))

from oracle import refrun                                   # noqa: E402
from helpers import iso_problem                              # noqa: E402

OUT = os.path.join(HERE, '..', 'tests', 'golden')
N_SAMPLE = 2048


def main():
    n, nbl, tn = 24, 8, 100.0
    for so in (8, 12):
        ref = refrun.load_forward(so)
        if ref is None:
            raise SystemExit(f"oracle/_ref/forward_iso_so{so}.c is missing: run oracle/make_ref.py first")
        q = iso_problem(n, nbl, so, tn)
        refrun.run_forward(ref, q['u'], q['damp'], 1.5, q['dt'], 1, q['nt'] - 2, q['src'], q['rec'], so, threads=4)
        u = q['u']
        xs = so + nbl + (n - 1) // 2                        # the source sits at x = (n - 1) h / 2
        idx = np.sort(np.random.default_rng(so).choice(u.size, N_SAMPLE, replace=False)).astype(np.int64)
        path = os.path.join(OUT, f'refgen_iso3d_so{so}.npz')
        np.savez_compressed(path, so=so, n=n, nbl=nbl, tn=tn, rec=q['rec']['data'], plane_x=xs,
                            u_plane=np.ascontiguousarray(u[:, xs]), u_index=idx, u_sample=u.reshape(-1)[idx],
                            u_max=np.float32(np.abs(u).max()))
        print(f"{os.path.basename(path)}: {os.path.getsize(path) / 1024:.0f} KiB")


if __name__ == '__main__':
    main()
