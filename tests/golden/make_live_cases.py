#!/usr/bin/env python
"""Records tests/golden/live_cases.npz: for every case that tests/test_oracle_vs_golden.py compares with the live
reference (same-seed shapes, custom wall maps, stepping a finished env, the 24-shape fuzz of both env ids and
observers), the trajectory under that comparison's protocol, as 8-byte digests of every step's observation,
rewards, dones, info and grid, plus the rewards and dones themselves.

    python tests/golden/make_live_cases.py

The trajectories are the oracle's (oracle/snake_oracle.py), recorded where the original project was not available;
the live tests, which run wherever it is there (oracle.cpu_runner.reference_search_path), hold the oracle to the
original on exactly these cases, and test_live_reference_cases_against_stored_trajectories holds the oracle to this
file on every run.
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path[:0] = [ROOT, os.path.join(ROOT, 'tests')]

from test_oracle_vs_golden import LIVE_GOLDEN, live_cases, oracle_record  # noqa: E402


def main():
    out = {}
    for name in sorted(live_cases()):
        for key, arr in oracle_record(name).items():
            out[f'{name}_{key}'] = arr
    np.savez_compressed(LIVE_GOLDEN, **out)
    print(f'{LIVE_GOLDEN}: {len(live_cases())} cases, {os.path.getsize(LIVE_GOLDEN)} bytes')


if __name__ == '__main__':
    main()
