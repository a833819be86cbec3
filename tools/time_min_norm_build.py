"""Times the minimum-norm basis build (temd_basis_build_min_norm: Jacobi SVD, truncated whitening, one Cholesky pass)
against the default CholeskyQR2 build, with CUDA events, on one GPU.  Prints the card and its power limit first.

    python tools/time_min_norm_build.py [--reps R]

Cases: the 0.25-degree lat-lon grid (1,038,240 columns, 721 distinct latitudes) at L = 1000, dense and de-duplicated
(the default build refuses there: rank 721 < 1001), and ne120pg2 (345,600 columns, 47,562 distinct latitudes) at
L = 100, where both builds run and the SVD is the tall kind."""
import argparse
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

from pytemdiags_b200 import synthetic as syn
from pytemdiags_b200.engine import DedupEngine, Engine


def card():
    try:
        q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader'], capture_output=True,
                           text=True, check=True).stdout.strip().splitlines()[0]
    except (OSError, subprocess.CalledProcessError, IndexError):
        q = torch.cuda.get_device_name(0) + ', power limit unknown'
    return q


def time_build(eng, reps):
    eng.build_basis()                      # warm-up: module load, workspaces
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    best = None
    for _ in range(reps):
        torch.cuda.synchronize()
        a.record()
        eng.build_basis()
        b.record()
        torch.cuda.synchronize()
        ms = a.elapsed_time(b)
        best = ms if best is None else min(best, ms)
    return best


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--reps', type=int, default=3)
    args = ap.parse_args()
    print('card: %s' % card())
    lat_out = np.arange(-89.5, 90, 1.0)
    cases = (('latlon 721x1440', syn.latlon_grid(721, 1440)[0], 1000, (True,)),
             ('ne120pg2', syn.pg2_grid(120)[0], 100, (True, False)))
    for name, lat, L, modes in cases:
        for dedup in (False, True):
            for min_norm in modes:
                eng = (DedupEngine if dedup else Engine)(lat, lat_out, L, device='cuda:0', min_norm=min_norm)
                ms = time_build(eng, args.reps)
                print('%-16s N=%-8d L=%-5d %-6s %-9s build %9.1f ms  rank %d' % (
                    name, lat.shape[0], L, 'dedup' if dedup else 'dense', 'min_norm' if min_norm else 'default', ms,
                    eng.rank))
                del eng
                torch.cuda.empty_cache()


if __name__ == '__main__':
    main()
