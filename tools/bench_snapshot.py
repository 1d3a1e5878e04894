#!/usr/bin/env python
"""What per-env snapshot and restore cost, in one job, the arms alternated round by round.

    python tools/bench_snapshot.py [--rounds 3] [--shapes cfg5,cfg3,cfg4,cfg2]

Arms, at every shape (one batch per shape and round; each arm timed with CUDA events over many calls after a burn-in):
  step            SnakeBatch.step as bench.py runs it (NHWC observation, no info)
  reset           a masked reset of every env with its observation (snk_reset with a mask of ones)
  snapshot        snk_snapshot of every env into a preallocated [N, snapshot_bytes] tensor
  restore         snk_restore of every env (src = arange) with the observation
  restore_8th     snk_restore of every eighth env with the observation (the other envs keep theirs)
  restore_bare    snk_restore of every env, no output at all: the copy kernel alone
Shapes (BASELINE.json): cfg5 20x20 / 4 snakes / vision 5 at 1 048 576 envs, cfg3 the same with frame_stack 4 at 65 536,
cfg4 64x64 / 16 snakes / vision 7 at 16 384, cfg2 full-grid observation at 4 096.  GB/s of the copy arms count the bytes
the copy kernels must move, from snk_snapshot_bytes: a snapshot reads the record and history (slot minus its 16-byte
header) and writes the slot; a restore reads the slot and writes the record and history.  Prints one JSON line per
measurement, a summary, and the card's name, power limit and maximum SM clock (read-only nvidia-smi query).
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
SHAPES = {   # name: (kwargs, envs, timed calls, burn-in calls)
    'cfg5': (CFG5, 1 << 20, 200, 20),
    'cfg3': (dict(CFG5, frame_stack=4), 65536, 1000, 100),
    'cfg4': (dict(height=64, width=64, num_snakes=16, snake_length=5, vision_range=7,
                  reward_dict={'fruit': 10.0, 'kill': 1.0, 'lose': -1.0, 'win': 0.1, 'time': -0.001}), 16384, 1000, 100),
    'cfg2': (dict(height=20, width=20, num_snakes=4, snake_length=3), 4096, 3000, 300),
}
ARMS = ('step', 'reset', 'snapshot', 'restore', 'restore_8th', 'restore_bare')
NPOOL = 64


def smi():
    q = 'name,power.limit,clocks.max.sm'
    r = subprocess.run(['nvidia-smi', f'--query-gpu={q}', '--format=csv,noheader', '-i', '0'], capture_output=True, text=True)
    return r.stdout.strip() or r.stderr.strip()


def measure(shape, arms):
    from marl_snake_b200 import SnakeBatch
    from marl_snake_b200._lib import check, lib
    kw, n, calls, burn = SHAPES[shape]
    dev = torch.device('cuda', 0)
    b = SnakeBatch(n, seed=0, **kw)
    ns, slot = b.num_snakes, b.snapshot_bytes
    gen = torch.Generator(device=dev).manual_seed(1)
    acts = torch.randint(0, 3, (NPOOL, n, ns), dtype=torch.uint8, device=dev, generator=gen)
    ones = torch.ones(n, dtype=torch.uint8, device=dev)
    snap = torch.empty((n, slot), dtype=torch.uint8, device=dev)
    src_all = torch.arange(n, dtype=torch.int32, device=dev)
    src_8th = torch.where(src_all % 8 == 0, src_all, torch.full_like(src_all, -1))
    b.reset()
    for t in range(8):
        b.step(acts[t], want_info=False)
    b.snapshot(out=snap)
    stream = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
    obs = b._obs

    def restore(src, out):
        check(lib.snk_restore(b._h, C.c_void_p(src.data_ptr()), n, C.c_void_p(snap.data_ptr()),
                              C.c_void_p(out.data_ptr()) if out is not None else None, None, None, stream))
    ops = {
        'step': lambda t: b.step(acts[t % NPOOL], want_info=False),
        'reset': lambda t: check(lib.snk_reset(b._h, C.c_void_p(ones.data_ptr()), C.c_void_p(obs.data_ptr()), stream)),
        'snapshot': lambda t: check(lib.snk_snapshot(b._h, None, n, C.c_void_p(snap.data_ptr()), stream)),
        'restore': lambda t: restore(src_all, obs),
        'restore_8th': lambda t: restore(src_8th, obs),
        'restore_bare': lambda t: restore(src_all, None),
    }
    copy_bytes = {'snapshot': n * (2 * slot - 16), 'restore_bare': n * (2 * slot - 16)}
    res = []
    for arm in arms:
        op = ops[arm]
        for t in range(burn):
            op(t)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for t in range(calls):
            op(t)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / calls
        r = dict(shape=shape, arm=arm, num_envs=n, snapshot_bytes=slot, calls=calls, ms_per_call=ms)
        if arm in copy_bytes:
            r['gb_per_s'] = copy_bytes[arm] / (ms * 1e-3) / 1e9
        res.append(r)
    err = b.device_errors()
    b.close()
    del b, acts, snap
    torch.cuda.empty_cache()
    for r in res:
        r['device_errors'] = err
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--rounds', type=int, default=3)
    ap.add_argument('--shapes', default=','.join(SHAPES))
    ap.add_argument('--arms', default=','.join(ARMS))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('needs a CUDA device')
    print(json.dumps(dict(gpu=smi())), flush=True)
    arms = args.arms.split(',')
    res = {}
    for shape in args.shapes.split(','):
        for rnd in range(args.rounds):
            order = arms[rnd % len(arms):] + arms[:rnd % len(arms)]      # a different arm goes first every round
            for r in measure(shape, order):
                r['round'] = rnd
                res.setdefault(shape, {}).setdefault(r['arm'], []).append(r)
                print(json.dumps(r), flush=True)
    summary = {}
    for shape, by_arm in res.items():
        summary[shape] = {}
        for arm, rs in by_arm.items():
            v = sorted(r['ms_per_call'] for r in rs)
            s = dict(min=v[0], median=v[len(v) // 2], max=v[-1])
            if 'gb_per_s' in rs[0]:
                s['gb_per_s_at_median'] = sorted(r['gb_per_s'] for r in rs)[len(rs) // 2]
            summary[shape][arm] = s
    print(json.dumps(dict(summary=summary, gpu=smi())), flush=True)


if __name__ == '__main__':
    main()
