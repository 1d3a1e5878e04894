#!/usr/bin/env python
"""Step time of the cfg5 shape with wall-map pools, in one job, the arms alternated round by round.

    python tools/bench_map_pool.py [--rounds 3] [--steps 1000] [--burn 300] [--envs 1048576]

Arms (every one at --envs environments of the cfg5 shape: 20x20, 4 snakes, length 3, vision_range 5, Philox seed 0):
  no_map        SnakeBatch without a layout (the walled box, bench.py's workload)
  one_map       wall_map=layout 0 (snk_create_map)
  pool16        wall_maps=layouts 0..15, default assignment (env % 16), next_maps never rewritten
  pool256       wall_maps=layouts 0..255, likewise
  pool16_redraw pool16 with next_maps.random_(0, 16) before every step (the redraw kernel is inside the timed region)
  16x65536      sixteen single-map handles of envs / 16 environments each, layouts 0..15, stepped back to back: the
                one-handle-per-layout setup a pool replaces (one step = sixteen launches)
Layouts are the walled box with one to four random wall bars (seeded).  Times come from CUDA events around --steps
steps after --burn steps; each arm's batch is created fresh in every round.  Prints one JSON line per measurement and
the card's name and power limit.
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

KW = dict(height=20, width=20, num_snakes=4, snake_length=3, vision_range=5, frame_stack=1)
NPOOL = 251


def smi():
    q = 'name,power.limit,clocks.sm,clocks.max.sm'
    r = subprocess.run(['nvidia-smi', f'--query-gpu={q}', '--format=csv,noheader', '-i', '0'], capture_output=True, text=True)
    return r.stdout.strip() or r.stderr.strip()


def layouts(n, seed=7):
    rng = np.random.RandomState(seed)
    out = []
    for _ in range(n):
        m = np.ones((20, 20), dtype=np.uint8)
        m[1:-1, 1:-1] = 0
        for _ in range(rng.randint(1, 5)):
            r, c, ln = rng.randint(2, 17), rng.randint(2, 12), rng.randint(3, 7)
            if rng.rand() < 0.5:
                m[r, c:c + ln] = 1
            else:
                m[c:c + ln, r] = 1
        out.append(m)
    return np.stack(out)


def measure(arm, n_envs, steps, burn, maps):
    from marl_snake_b200 import SnakeBatch
    dev = torch.device('cuda', 0)
    if arm == '16x65536':
        n = n_envs // 16
        batches = [SnakeBatch(n, seed=0, env_id_offset=k * n, wall_map=maps[k], **KW) for k in range(16)]
    elif arm == 'no_map':
        batches = [SnakeBatch(n_envs, seed=0, **KW)]
    elif arm == 'one_map':
        batches = [SnakeBatch(n_envs, seed=0, wall_map=maps[0], **KW)]
    else:
        m = 256 if arm == 'pool256' else 16
        batches = [SnakeBatch(n_envs, seed=0, wall_maps=maps[:m], **KW)]
    redraw = arm == 'pool16_redraw'
    gen = torch.Generator(device=dev).manual_seed(1)
    acts = [torch.randint(0, 3, (NPOOL, b.num_envs, 4), dtype=torch.uint8, device=dev, generator=gen) for b in batches]
    for b in batches:
        b.reset()

    def step(t):
        for b, a in zip(batches, acts):
            if redraw:
                b.next_maps.random_(0, 16, generator=gen)
            b.step(a[t % NPOOL], want_info=False)
    for t in range(burn):
        step(t)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for t in range(steps):
        step(burn + t)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    errs = [b.device_errors() for b in batches]
    comp = all(b.obs_compressed for b in batches)
    for b in batches:
        b.close()
    del batches, acts
    torch.cuda.empty_cache()
    return dict(arm=arm, num_envs=n_envs, steps=steps, ms_per_step=ms, device_errors=max(errs), obs_compressed=comp)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--rounds', type=int, default=3)
    ap.add_argument('--steps', type=int, default=1000)
    ap.add_argument('--burn', type=int, default=300)
    ap.add_argument('--envs', type=int, default=1 << 20)
    ap.add_argument('--arms', default='no_map,one_map,pool16,pool256,pool16_redraw,16x65536')
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('needs a CUDA device')
    print(json.dumps(dict(gpu=smi())), flush=True)
    maps = layouts(256)
    res = {}
    for rnd in range(args.rounds):
        for arm in args.arms.split(','):
            r = measure(arm, args.envs, args.steps, args.burn, maps)
            r['round'] = rnd
            res.setdefault(arm, []).append(r['ms_per_step'])
            print(json.dumps(r), flush=True)
    summary = {arm: dict(min=min(v), median=sorted(v)[len(v) // 2], max=max(v)) for arm, v in res.items()}
    print(json.dumps(dict(summary=summary, gpu=smi())), flush=True)


if __name__ == '__main__':
    main()
