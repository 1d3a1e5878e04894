"""CPU timing of the reference's step path (TEST/BENCH INFRASTRUCTURE).

Used only by bench.py's `cpu_baseline` leg and its `--impl reference` arm.  Two kinds of worker:

  kind "reference"  the UNMODIFIED reference `SnakeEnv` from oracle/_ref (installed there by
                    `make -C oracle ref`, git-ignored, ships to the GPU box with the snapshot) behind the
                    structural gym stub -- `gym.make('Snake-v1', **kw)` exactly as make_snake does
                    (wrappers.py:206-209);
  kind "port"       oracle/snake_oracle.py, the restatement (caches the spawn-pose enumeration the
                    reference repeats on every reset and vectorises _encode, so it is ~10x faster).

Either way the run is shaped like the reference's vectorisation: one OS process per environment
(wrappers.py:211-212), reset on all(done) (wrappers.py:141-143), random actions, module-global NumPy RNG.
"""
import json
import multiprocessing as mp
import os
import sys
import time

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
REF_DIR = os.path.join(HERE, '_ref')


def usable_cores():
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        return max(1, os.cpu_count() or 1)


def reference_available():
    return os.path.exists(os.path.join(REF_DIR, 'marlenv', 'envs', 'snake_env.py'))


def reference_checkout():
    """Where the original project's checkout is looked for: SNK_REFERENCE_DIR, else the location BASELINE.json
    records for it (reference_path)."""
    if os.environ.get('SNK_REFERENCE_DIR'):
        return os.environ['SNK_REFERENCE_DIR']
    with open(os.path.join(os.path.dirname(HERE), 'BASELINE.json')) as f:
        return json.load(f)['reference_path']


def reference_search_path():
    """The sys.path entry that holds the unmodified reference package `marlenv`: `marlenv/` of the original project's
    checkout (reference_checkout()), else the install in oracle/_ref; None when neither is there.  A SNK_REFERENCE_DIR
    that names no checkout is an error rather than a silent skip of every test that needs the original."""
    path = os.path.join(reference_checkout(), 'marlenv')
    if os.path.exists(os.path.join(path, 'marlenv', 'envs', 'snake_env.py')):
        return path
    if os.environ.get('SNK_REFERENCE_DIR'):
        raise RuntimeError(f"SNK_REFERENCE_DIR={os.environ['SNK_REFERENCE_DIR']} is not a checkout of the original "
                           'project (no marlenv/marlenv/envs/snake_env.py under it)')
    return REF_DIR if reference_available() else None


def make_reference_env(kw):
    """gym.make('Snake-v1', **kw) on the unmodified reference installed in oracle/_ref."""
    for p in (REF_DIR, os.path.join(HERE, 'gym_stub')):
        if p in sys.path:
            sys.path.remove(p)
        sys.path.insert(0, p)
    for name in [m for m in sys.modules if m == 'marlenv' or m.startswith('marlenv.')]:
        if not (getattr(sys.modules[name], '__file__', '') or '').startswith(REF_DIR):
            del sys.modules[name]                    # the repo's import shim of the same name
    import gym
    import marlenv  # noqa: F401  (registers Snake-v1 with the stub's registry)
    assert marlenv.__file__.startswith(REF_DIR), marlenv.__file__
    return gym.make('Snake-v1', **kw)


def _worker(rank, kw, conn, kind):
    np.random.seed(1000 + rank)
    if kind == 'reference':
        env = make_reference_env(kw)
    else:
        from oracle.snake_oracle import OracleSnakeEnv
        env = OracleSnakeEnv(**kw)
    ns = env.num_snakes
    env.reset()
    act = np.random.RandomState(rank).randint(0, 3, size=(4096, ns))
    t = 0
    while True:
        msg = conn.recv()
        if msg is None:
            break
        n_steps = msg
        t0 = time.perf_counter()
        for _ in range(n_steps):
            _, _, done, _ = env.step([int(a) for a in act[t & 4095]])
            t += 1
            if all(done):
                env.reset()
        conn.send(time.perf_counter() - t0)
    conn.close()


class CpuPool:
    """P processes, one env each; run(n) advances every env by n steps and returns wall seconds."""

    def __init__(self, kw, procs=None, kind='port'):
        if kind == 'reference' and not reference_available():
            raise RuntimeError('oracle/_ref is missing: run `make -C oracle ref` where the original project is checked out')
        self.kind = kind
        self.procs = procs or usable_cores()
        ctx = mp.get_context('spawn')
        self.pipes, self.ps = [], []
        for r in range(self.procs):
            a, b = ctx.Pipe()
            p = ctx.Process(target=_worker, args=(r, kw, b, kind), daemon=True)
            p.start()
            self.pipes.append(a)
            self.ps.append(p)
        self.num_snakes = kw.get('num_snakes', 4)
        self.run(1)                      # wait until every worker has imported and reset

    def run(self, n_steps):
        t0 = time.perf_counter()
        for c in self.pipes:
            c.send(n_steps)
        for c in self.pipes:
            c.recv()
        return time.perf_counter() - t0

    def close(self):
        for c in self.pipes:
            c.send(None)
        for p in self.ps:
            p.join(timeout=5)
