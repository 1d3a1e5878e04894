#!/usr/bin/env python
"""Previous build against this one for the viewer-pair encode, alternating the two libsnk.so in one job.

    python tools/ab_encode_pairs.py OLD_LIB NEW_LIB [--rounds 3] [--out DIR]

Every measurement is a fresh process with SNK_LIB_PATH pointing at one build (the library is loaded once per process):
  1. bench.py --gpus 1 --steps 2000 --warmup 100 (no config block, no CPU arm), `--rounds` times per build, alternating; ms_per_step of each run;
  2. bench.py --dump-outputs for both builds, then a byte comparison of the files;
  3. tools/bench_configs.py cfg5_shard cfg5_full cfg1 cfg2 cfg3 cfg4 per build, alternating twice;
  4. the rules-only floor: bench_configs.py cfg5_full with BENCH_NO_OBS=1 (step(want_obs=False)) per build.
The card name, power limit and SM clocks are read before and after, and every record of the child processes is kept
under DIR (default ab_encode_pairs_out, relative to the working directory).
"""
import argparse
import filecmp
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def smi():
    q = 'name,power.limit,clocks.sm,clocks.max.sm,driver_version'
    r = subprocess.run(['nvidia-smi', f'--query-gpu={q}', '--format=csv,noheader', '-i', '0'],
                       capture_output=True, text=True)
    return r.stdout.strip() or r.stderr.strip()


def run(lib, args, env_extra=None, log=None):
    env = dict(os.environ, SNK_LIB_PATH=os.path.abspath(lib), **(env_extra or {}))
    r = subprocess.run([sys.executable] + args, cwd=ROOT, env=env, capture_output=True, text=True)
    if log:
        with open(log, 'a') as f:
            f.write(f'$ SNK_LIB_PATH={lib} {" ".join(args)}  (exit {r.returncode})\n{r.stdout}\n{r.stderr[-4000:]}\n')
    if r.returncode != 0:
        raise SystemExit(f'{args} with {lib} failed ({r.returncode}):\n{r.stderr[-3000:]}')
    return [json.loads(line) for line in r.stdout.splitlines() if line.startswith('{')]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('old')
    ap.add_argument('new')
    ap.add_argument('--rounds', type=int, default=3)
    ap.add_argument('--out', default='ab_encode_pairs_out')
    ap.add_argument('--parts', default='bench,dump,configs,rules', help='comma-separated subset of the four parts')
    args = ap.parse_args()
    parts = args.parts.split(',')
    os.makedirs(args.out, exist_ok=True)
    log = os.path.join(args.out, 'children.log')
    libs = {'old': args.old, 'new': args.new}
    print('gpu', smi(), flush=True)

    bench = {k: [] for k in libs}
    for rnd in range(args.rounds if 'bench' in parts else 0):
        for arm, lib in libs.items():
            rec = run(lib, ['bench.py', '--gpus', '1', '--steps', '2000', '--warmup', '100', '--no-configs',
                            '--no-cpu-baseline'], log=log)[-1]
            bench[arm].append(rec['ms_per_step'])
            print(f'bench round {rnd} {arm}: {rec["ms_per_step"]:.5f} ms/step  clocks {rec.get("clocks")}', flush=True)
            if rnd == 0:
                with open(os.path.join(args.out, f'bench_{arm}.json'), 'w') as f:
                    json.dump(rec, f)
    if 'bench' in parts:
        for arm, v in bench.items():
            s = sorted(v)
            print(f'== bench {arm}: min {s[0]:.5f} median {s[len(s) // 2]:.5f} max {s[-1]:.5f} ms', flush=True)
        print(f'every new run below every old run: {max(bench["new"]) < min(bench["old"])}', flush=True)

    if 'dump' in parts:
        dumps = {}
        for arm, lib in libs.items():
            dumps[arm] = os.path.join(args.out, f'dump_{arm}')
            run(lib, ['bench.py', '--gpus', '1', '--steps', '50', '--warmup', '10', '--no-configs', '--no-cpu-baseline',
                      '--dump-outputs', os.path.abspath(dumps[arm])], log=log)
        names = sorted(os.listdir(dumps['old']))
        same = names == sorted(os.listdir(dumps['new'])) and all(
            filecmp.cmp(os.path.join(dumps['old'], n), os.path.join(dumps['new'], n), shallow=False) for n in names)
        print(f'dump-outputs {names} byte-identical: {same}', flush=True)

    cfgs = ['cfg5_shard', 'cfg5_full', 'cfg1', 'cfg2', 'cfg3', 'cfg4']
    for rnd in range(2 if 'configs' in parts else 0):
        for arm, lib in libs.items():
            for rec in run(lib, ['tools/bench_configs.py'] + cfgs, log=log):
                t = f'{rec["ms_per_step"]:.5f} ms/step' if 'ms_per_step' in rec else f'{rec["us_per_step"]:.2f} us/step'
                print(f'configs round {rnd} {arm}: {rec.get("config")} {rec.get("num_envs")} envs {rec.get("mode", "")} {t}',
                      flush=True)
    for rnd in range(2 if 'rules' in parts else 0):
        for arm, lib in libs.items():
            for rec in run(lib, ['tools/bench_configs.py', 'cfg5_full'], env_extra={'BENCH_NO_OBS': '1'}, log=log):
                print(f'rules-only round {rnd} {arm}: cfg5_full {rec.get("mode", "")} {rec["ms_per_step"]:.5f} ms/step',
                      flush=True)
    print('gpu', smi(), flush=True)


if __name__ == '__main__':
    main()
