#!/usr/bin/env python
"""What the global state costs a step, in one job, the arms alternated round by round.

    python tools/bench_global_state.py [--rounds 3] [--shapes cfg5,cfg5_shard,cfg3,cfg4,cfg2,cfg2_many]

Arms, at every shape:
  step       SnakeBatch.step (or step_many) as bench.py runs it: NHWC observation, no global state
  grid       the same call with global_state=True: the step kernel also writes every env's grid (snk_step_grid)
  get_state  the plain call followed by snk_get_state with only the grid -- the route before the fused output
Shapes (BASELINE.json): cfg5 20x20 / 4 snakes / vision 5 at 1 048 576 envs and its 131 072-env shard of 8 GPUs, cfg3 the
same with frame_stack 4 at 65 536, cfg4 64x64 / 16 snakes / vision 7 at 16 384, cfg2 full-grid observation at 4 096,
stepped one call per step and through step_many (T = 64 steps per call; its arms write the last step's observation
and grid, and get_state runs once per call).  Each arm's batch is created fresh in every round; times come from
CUDA events around the timed steps after a burn-in.  Prints one JSON line per measurement and the card's name, power
limit and maximum SM clock (read-only nvidia-smi query).
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

CFG5 = dict(height=20, width=20, num_snakes=4, snake_length=3, vision_range=5)
SHAPES = {   # name: (kwargs, envs, timed steps, burn-in steps, steps per step_many call or 0)
    'cfg5': (CFG5, 1 << 20, 1000, 200, 0),
    'cfg5_shard': (CFG5, 131072, 4000, 500, 0),
    'cfg3': (dict(CFG5, frame_stack=4), 65536, 3000, 300, 0),
    'cfg4': (dict(height=64, width=64, num_snakes=16, snake_length=5, vision_range=7,
                  reward_dict={'fruit': 10.0, 'kill': 1.0, 'lose': -1.0, 'win': 0.1, 'time': -0.001}), 16384, 3000, 300, 0),
    'cfg2': (dict(height=20, width=20, num_snakes=4, snake_length=3), 4096, 10000, 1000, 0),
    'cfg2_many': (dict(height=20, width=20, num_snakes=4, snake_length=3), 4096, 64 * 160, 64 * 16, 64),
}
NPOOL = 64


def smi():
    q = 'name,power.limit,clocks.max.sm'
    r = subprocess.run(['nvidia-smi', f'--query-gpu={q}', '--format=csv,noheader', '-i', '0'], capture_output=True, text=True)
    return r.stdout.strip() or r.stderr.strip()


def measure(shape, arm):
    from marl_snake_b200 import SnakeBatch
    from marl_snake_b200._lib import SnkStateView, check, lib
    kw, n, steps, burn, T = SHAPES[shape]
    dev = torch.device('cuda', 0)
    b = SnakeBatch(n, seed=0, global_state=(arm == 'grid'), **kw)
    H, W = b.grid_shape
    ns = b.num_snakes
    grid = torch.empty((n, H, W), dtype=torch.uint8, device=dev) if arm == 'get_state' else None
    view = SnkStateView(grid=grid.data_ptr()) if grid is not None else None
    gen = torch.Generator(device=dev).manual_seed(1)
    acts = torch.randint(0, 3, (NPOOL if not T else T, n, ns), dtype=torch.uint8, device=dev, generator=gen)
    obs_last = torch.empty((n,) + b.obs_shape, dtype=torch.uint8, device=dev) if T else None
    rew = torch.empty((T, n, ns), dtype=torch.float64, device=dev) if T else None
    done = torch.empty((T, n, ns), dtype=torch.uint8, device=dev) if T else None
    b.reset()

    def call(t):
        if T:
            b.step_many(acts, obs=obs_last, rewards=rew, dones=done)
        else:
            b.step(acts[t % NPOOL], want_info=False)
        if view is not None:
            check(lib.snk_get_state(b._h, C.byref(view), C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)))
    per = T or 1
    for t in range(burn // per):
        call(t)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for t in range(steps // per):
        call(t)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / (steps // per * per)
    if arm == 'grid':
        assert torch.equal(b.global_state, b.get_state()['grid'])
    err = b.device_errors()
    b.close()
    del b, acts, grid
    torch.cuda.empty_cache()
    return dict(shape=shape, arm=arm, num_envs=n, steps=steps // per * per, steps_per_call=per, ms_per_step=ms,
                device_errors=err)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--rounds', type=int, default=3)
    ap.add_argument('--shapes', default=','.join(SHAPES))
    ap.add_argument('--arms', default='step,grid,get_state')
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('needs a CUDA device')
    print(json.dumps(dict(gpu=smi())), flush=True)
    res = {}
    for shape in args.shapes.split(','):
        for rnd in range(args.rounds):
            for arm in args.arms.split(','):
                r = measure(shape, arm)
                r['round'] = rnd
                res.setdefault(shape, {}).setdefault(arm, []).append(r['ms_per_step'])
                print(json.dumps(r), flush=True)
    summary = {shape: {arm: dict(min=min(v), median=sorted(v)[len(v) // 2], max=max(v)) for arm, v in arms.items()}
               for shape, arms in res.items()}
    for shape, arms in summary.items():
        if 'step' in arms:
            base = arms['step']['median']
            for arm, s in arms.items():
                s['vs_step'] = s['median'] / base - 1.0
    print(json.dumps(dict(summary=summary, gpu=smi())), flush=True)


if __name__ == '__main__':
    main()
