#!/usr/bin/env python
"""A/B of the launch-shape switches at cfg5 with the observation block in compressible memory, alternating in one
process (the SNK_* variables are read when a batch is created).

    python tools/ab_obs_retune.py [--rounds 3] [--steps 400] [--configs cfg5_full,cfg5_shard] VARIANT ...

A VARIANT is a comma-separated list of SNK_* assignments, or 'default'.  Every round creates one batch per variant and
config (same seed, same actions), burns in 300 steps and times --steps eager steps with CUDA events.  Prints one
line per measurement and a min / median / max summary per variant.
"""
import argparse
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tools'))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('variants', nargs='+')
    ap.add_argument('--rounds', type=int, default=3)
    ap.add_argument('--steps', type=int, default=400)
    ap.add_argument('--configs', default='cfg5_full,cfg5_shard')
    args = ap.parse_args()
    import numpy as np
    import torch
    from bench_configs import CONFIGS
    from marl_snake_b200 import SnakeBatch

    print(f'lib {os.environ.get("SNK_LIB_PATH", "default")}', flush=True)
    res = {}
    for rnd in range(args.rounds):
        for cfg in args.configs.split(','):
            for var in args.variants:
                sets = {} if var == 'default' else dict(kv.split('=') for kv in var.split(','))
                old = {k: os.environ.get(k) for k in sets}
                os.environ.update(sets)
                kw = dict(CONFIGS[cfg])
                N = kw.pop('num_envs')
                b = SnakeBatch(N, seed=0, device=0, **kw)
                for k, v in old.items():
                    if v is None:
                        del os.environ[k]
                    else:
                        os.environ[k] = v
                g = torch.Generator(device='cuda').manual_seed(1)
                pool = torch.randint(0, 3, (251, N, kw['num_snakes']), dtype=torch.uint8, device='cuda', generator=g)
                b.reset()
                for t in range(300):
                    b.step(pool[t % 251], want_info=False)
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                torch.cuda.synchronize()
                e0.record()
                for t in range(args.steps):
                    b.step(pool[(300 + t) % 251], want_info=False)
                e1.record()
                torch.cuda.synchronize()
                ms = e0.elapsed_time(e1) / args.steps
                assert b.device_errors() == 0
                res.setdefault((cfg, var), []).append(ms)
                print(f'round {rnd} {cfg:11s} {var:40s} compressed={b.obs_compressed} {ms:.5f} ms', flush=True)
                b.close()
                del b, pool
    for (cfg, var), v in res.items():
        print(f'== {cfg:11s} {var:40s} min {min(v):.5f} median {float(np.median(v)):.5f} max {max(v):.5f} ms')


if __name__ == '__main__':
    main()
