"""What the compact record layout rests on (DESIGN.md section 3), checked on the CPU against the oracle and -- where
the original project is there (oracle.cpu_runner.reference_search_path) -- against the unmodified reference itself:

  after reset() and after every step(), the grid is exactly   wall layout + FRUIT cells + the bodies of the LIVE snakes
  (HEAD at coords[0], TAIL at coords[-1], BODY between), and the number of fruit cells never exceeds
  num_fruits + num_snakes // 2 within an episode (a fruit is only ever added without one being eaten when two or more
  heads meet on a fruit cell and die, snake_env.py:521-544).

That is why the kernel may keep the fruit cells and the bodies in HBM and rebuild the grid in shared memory, and why
num_fruits + num_snakes fruit slots are enough."""
import os
import sys

import numpy as np
import pytest

from oracle.cpu_runner import reference_search_path
from oracle.snake_oracle import OracleSnakeEnv

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SHAPES = [
    dict(height=20, width=20, num_snakes=4, snake_length=3, vision_range=5),
    dict(height=10, width=10, num_snakes=6, snake_length=2, num_fruits=12),                 # crowded: head-on meetings on fruit
    dict(height=8, width=14, num_snakes=5, snake_length=3, num_fruits=20, max_episode_steps=40),
    dict(height=16, width=16, num_snakes=8, snake_length=4, vision_range=3, num_fruits=6),
]


def implied_grid(walls, grid, bodies, alive):
    """walls + the grid's own FRUIT cells + live bodies; everything else must follow from these."""
    out = walls.copy()
    out[grid == 2] = 2
    for i, (cells, a) in enumerate(zip(bodies, alive)):
        if not a:
            continue
        for k, (r, c) in enumerate(cells):
            out[r, c] = (3 if k == 0 else 5 if k == len(cells) - 1 else 4) + 10 * i
    return out


def box_walls(H, W):
    w = np.ones((H, W), dtype=np.int64)
    w[1:-1, 1:-1] = 0
    return w


def drive(make_env, get_state, kw, seed, steps):
    np.random.seed(seed)
    env = make_env()
    H, W, ns = kw['height'], kw['width'], kw['num_snakes']
    nf = kw.get('num_fruits', int(round(0.8 * ns)))
    walls = box_walls(H, W)
    env.reset()
    rng = np.random.RandomState(seed + 1)
    most, over = 0, 0
    for t in range(steps):
        grid, bodies, alive = get_state(env)
        assert np.array_equal(np.asarray(grid), implied_grid(walls, np.asarray(grid), bodies, alive)), (kw, seed, t)
        n_fruit = int((np.asarray(grid) == 2).sum())
        assert n_fruit <= nf + ns // 2, (kw, seed, t, n_fruit)
        most = max(most, n_fruit)
        over += n_fruit > nf
        _, _, dones, _ = env.step([int(a) for a in rng.randint(0, 3, size=ns)])
        if all(dones):
            env.reset()
    return most, over


@pytest.mark.parametrize('kw', SHAPES, ids=lambda k: f"{k['height']}x{k['width']}x{k['num_snakes']}")
def test_oracle_grid_is_walls_fruits_and_live_bodies(kw):
    most = over = 0
    for seed in range(6):
        m, o = drive(lambda: OracleSnakeEnv(**kw), lambda e: (e.grid, [list(b) for b in e.body], e.alive), kw, seed, 300)
        most, over = max(most, m), over + o
    if kw.get('num_fruits') == 12:
        assert over > 0, 'the crowded 10x10 shape is there to push the fruit count past num_fruits at least once'


@pytest.mark.needs_reference
@pytest.mark.parametrize('kw', SHAPES, ids=lambda k: f"{k['height']}x{k['width']}x{k['num_snakes']}")
def test_reference_grid_is_walls_fruits_and_live_bodies(kw):
    ref_pkg = reference_search_path()
    sys.path.insert(0, ref_pkg)
    sys.path.insert(0, os.path.join(ROOT, 'oracle', 'gym_stub'))
    for m in [m for m in sys.modules if m == 'gym' or m.startswith('gym.') or m == 'marlenv' or m.startswith('marlenv.')]:
        del sys.modules[m]                   # this repository's `marlenv` import shim may already be loaded
    try:
        import gym
        import marlenv  # noqa: F401  (registers Snake-v1)
        assert marlenv.__file__.startswith(ref_pkg), marlenv.__file__
        for seed in range(3):
            drive(lambda: gym.make('Snake-v1', **kw),
                  lambda e: (e.grid, [list(s.coords) for s in e.snakes], [s.alive for s in e.snakes]), kw, seed, 300)
    finally:
        sys.path.remove(os.path.join(ROOT, 'oracle', 'gym_stub'))
        sys.path.remove(ref_pkg)
        for m in [m for m in sys.modules if m == 'gym' or m.startswith('gym.') or m == 'marlenv' or m.startswith('marlenv.')]:
            del sys.modules[m]
