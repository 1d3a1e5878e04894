#!/usr/bin/env python
"""Generate golden trajectories by running the UNMODIFIED reference.

Needs a checkout of the original project (tranthai189765/MARL-Snake) at SNK_REFERENCE_DIR or at BASELINE.json's
reference_path:

    python tests/golden/make_golden.py

Imports `marlenv.envs.snake_env.SnakeEnv` from <checkout>/marlenv behind the
structural gym stub in oracle/gym_stub, drives it with seeded random actions
under the reference's own auto-reset rule (wrappers.py:138-146) and records, per
step: actions, grid, rewards, dones, bit-packed observations, the signed
alive counter, terminal `info`, and the OUTPUTS of every RNG draw the env made
(accepted spawn-candidate indices, fruit ranks) in consumption order.  Also
records hand-built collision scenarios (SURVEY.md section 8a quirks) and the
spawn-candidate tables.  Output: tests/golden/*.npz (small, committed).
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, os.path.join(ROOT, 'oracle', 'gym_stub'))
sys.path.insert(0, ROOT)
from oracle.cpu_runner import reference_checkout  # noqa: E402
REF = reference_checkout()
sys.path.insert(0, os.path.join(REF, 'marlenv'))

import gym  # noqa: E402  (the stub)
import marlenv  # noqa: E402,F401  (registers Snake-v1)
from marlenv.core.snake import Snake, Direction  # noqa: E402
from marlenv.core.grid_util import dfs_sweep_empty, make_grid, make_grid_from_txt  # noqa: E402
import marlenv.envs.snake_env as ref_snake_env  # noqa: E402

ASSETS = os.path.join(REF, 'marlenv', 'marlenv', 'assets')


def load_asset_map(name, mapper=None):
    """A wall layout from the reference's assets, read by the reference's own loader (core/grid_util.py:23-33).
    The loader splits on '\\n' and so chokes on a final newline; such files are read from a scratch copy with the
    final newline removed (the map itself is unchanged)."""
    import tempfile
    mapper = mapper or {'#': 1, '.': 0}
    text = open(os.path.join(ASSETS, name)).read().rstrip('\n')
    with tempfile.NamedTemporaryFile('w', suffix='.txt', delete=False) as fp:
        fp.write(text)
    try:
        return make_grid_from_txt(fp.name, mapper)
    finally:
        os.unlink(fp.name)


class CustomWalls:
    """The reference's reset() always builds make_grid's walled box (snake_env.py:133) and has no parameter for a
    map; while installed, the `make_grid` name that reset() calls returns the custom layout instead.  Nothing else of
    the reference is touched: dfs_sweep_empty, random_empty_coords and the step rules work on whatever grid they get."""

    def __init__(self, wall_grid):
        self.grid = None if wall_grid is None else np.asarray(wall_grid)

    def __enter__(self):
        self._orig = ref_snake_env.make_grid
        if self.grid is not None:
            ref_snake_env.make_grid = lambda *a, **k: self.grid.copy()

    def __exit__(self, *exc):
        ref_snake_env.make_grid = self._orig

DIRS = [Direction.UP, Direction.RIGHT, Direction.DOWN, Direction.LEFT]


class DrawTap:
    """Logs outputs of np.random.permutation / randint while installed."""

    def __init__(self):
        self.events = []

    def __enter__(self):
        self._perm, self._randint = np.random.permutation, np.random.randint
        tap = self

        def permutation(n):
            out = tap._perm(n)
            tap.events.append(('perm', np.array(out)))
            return out

        def randint(low, high=None, size=None, dtype=int):
            out = tap._randint(low, high, size=size, dtype=dtype)
            tap.events.append(('randint', np.array(out).reshape(-1)))
            return out

        np.random.permutation, np.random.randint = permutation, randint
        return self

    def __exit__(self, *exc):
        np.random.permutation, np.random.randint = self._perm, self._randint

    def drain(self, ns):
        """Collapse to draw outputs: only the last permutation of a run is the accepted one."""
        out = []
        ev = self.events
        for k, (kind, val) in enumerate(ev):
            if kind == 'perm':
                if k + 1 < len(ev) and ev[k + 1][0] == 'perm':
                    continue                      # rejected attempt (overlap)
                out.extend(int(v) for v in val[:ns])
            else:
                out.extend(int(v) for v in val)
        self.events = []
        return out


def pack_obs(obs):
    """uint8 0/1 [..., 8*fs] -> uint8 [..., fs], channel c of a frame in bit c."""
    o = np.asarray(obs, dtype=np.uint8)
    fs = o.shape[-1] // 8
    o = o.reshape(*o.shape[:-1], fs, 8)
    return np.packbits(o, axis=-1, bitorder='little')[..., 0]


def snake_cells(env, W):
    """Per snake: alive flag, direction code, head-first cell indices (-1 padded)."""
    ns = env.num_snakes
    lens = [len(s.coords) if s.alive else 0 for s in env.snakes]
    L = max(lens + [1])
    cells = -np.ones((ns, L), dtype=np.int32)
    for i, s in enumerate(env.snakes):
        if s.alive:
            cells[i, :lens[i]] = [r * W + c for r, c in s.coords]
    alive = np.array([s.alive for s in env.snakes], dtype=np.uint8)
    dirs = np.array([DIRS.index(s.direction) for s in env.snakes], dtype=np.uint8)
    return alive, dirs, np.array(lens, dtype=np.int32), cells


ONLY = set(sys.argv[1:])          # `make_golden.py roll_human ...` regenerates just the named fixtures


def rollout(name, seed, num_envs, steps, env_id='Snake-v1', **kw):
    """Seeded random rollout of `num_envs` independent reference envs with auto-reset."""
    if ONLY and name not in ONLY:
        return
    ns = kw.get('num_snakes', 4)
    n_actions = 5 if kw.get('observer') == 'human' else 3
    walls = kw.get('wall_map')                      # nested list (H x W, 1 = wall) from load_asset_map, or None
    ref_kw = {k: v for k, v in kw.items() if k != 'wall_map'}
    per_env = []
    act_rng = np.random.RandomState(seed + 777)
    for e in range(num_envs):
        env = gym.make(env_id, **ref_kw)
        H, W = env.grid_shape
        np.random.seed(seed + e)
        tap = DrawTap()
        draws, draws_end = [], []
        with tap, CustomWalls(walls):
            obs0 = env.reset()
            draws.extend(tap.drain(ns))
            draws_end.append(len(draws))
            G, R, D, O, A, C, L = [], [], [], [], [], [], []
            info_step, info_rank, info_scores, info_steps, info_fruits, info_kills = [], [], [], [], [], []
            reset_grid = [env.grid.astype(np.uint8).copy()]
            for t in range(steps):
                a = act_rng.randint(0, n_actions, size=ns)
                obs, rew, done, info = env.step([int(x) for x in a])
                grid_after_step = env.grid.astype(np.uint8).copy()
                counter = env.alive_snakes
                if all(done):
                    obs = env.reset()
                    reset_grid.append(env.grid.astype(np.uint8).copy())
                draws.extend(tap.drain(ns))
                draws_end.append(len(draws))
                A.append(a.astype(np.uint8))
                G.append(grid_after_step)
                L.append(env.grid.astype(np.uint8).copy())     # live grid (after auto-reset)
                R.append(np.asarray(rew, dtype=np.float64))
                D.append(np.asarray(done, dtype=np.uint8))
                O.append(pack_obs(obs))
                C.append(counter)
                if info:
                    info_step.append(t)
                    info_rank.append(np.asarray(info['rank'], dtype=np.int32))
                    info_scores.append(np.asarray(info['episode_scores'], dtype=np.float64))
                    info_steps.append(np.asarray(info['episode_steps'], dtype=np.float64))
                    info_fruits.append(np.asarray(info['episode_fruits'], dtype=np.float64))
                    info_kills.append(np.asarray(info['episode_kills'], dtype=np.float64))
        zi = np.zeros((0, ns))
        per_env.append(dict(
            obs0=pack_obs(obs0), grid0=reset_grid[0], actions=np.stack(A), grid_step=np.stack(G),
            grid_live=np.stack(L), rewards=np.stack(R), dones=np.stack(D), obs=np.stack(O),
            counter=np.asarray(C, dtype=np.int32), draws=np.asarray(draws, dtype=np.int32),
            draws_end=np.asarray(draws_end, dtype=np.int32),
            info_step=np.asarray(info_step, dtype=np.int32),
            info_rank=np.stack(info_rank) if info_rank else zi.astype(np.int32),
            info_scores=np.stack(info_scores) if info_scores else zi,
            info_steps=np.stack(info_steps) if info_steps else zi,
            info_fruits=np.stack(info_fruits) if info_fruits else zi,
            info_kills=np.stack(info_kills) if info_kills else zi))
    out = {}
    for e, d in enumerate(per_env):
        for k, v in d.items():
            out[f'e{e}_{k}'] = v
    out['meta_kind'] = np.array('rollout')
    out['meta_env_id'] = np.array(env_id)
    out['meta_kwargs'] = np.array(repr(kw))
    out['meta_seed'] = np.array(seed)
    out['meta_num_envs'] = np.array(num_envs)
    out['meta_steps'] = np.array(steps)
    path = os.path.join(HERE, f'{name}.npz')
    np.savez_compressed(path, **out)
    n_term = sum(len(d['info_step']) for d in per_env)
    print(f'{name}: {num_envs} envs x {steps} steps, {n_term} episodes ended, '
          f'{os.path.getsize(path) / 1024:.1f} KiB')


# ----------------------------------------------------------------------------- scenarios
def build_env(H, W, snakes, fruits=(), counter=None, **kw):
    """Reference env forced into a hand-built state. snakes: list of head-first (r,c) lists or None(dead)."""
    ns = len(snakes)
    env = gym.make('Snake-v1', height=H, width=W, num_snakes=ns, snake_length=2, **kw)
    np.random.seed(0)
    env.reset()
    grid = make_grid(H, W, empty_value=0, wall_value=1)
    env.snakes = []
    for i, cells in enumerate(snakes):
        if cells is None:
            s = Snake(i, [(1, 1), (1, 2)])
            s.alive = False
            env.snakes.append(s)
            continue
        s = Snake(i, [tuple(c) for c in cells])
        env.snakes.append(s)
        for c in s.coords:
            grid[c] = 4 + 10 * i
        grid[s.head_coord] = 3 + 10 * i
        grid[s.tail_coord] = 5 + 10 * i
    for f in fruits:
        grid[tuple(f)] = 2
    env.grid = grid
    env.alive_snakes = counter if counter is not None else sum(c is not None for c in snakes)
    env._reset_epi_stats()
    env.episode_length = 0
    env.obs.clear()
    first = env._encode(env.grid, vision_range=env.vision_range)
    for _ in range(env.frame_stack):
        env.obs.append(first)
    return env


SCENARIOS = []


def scenario(fn):
    SCENARIOS.append(fn)
    return fn


REW = {'fruit': 10.0, 'kill': 3.0, 'lose': -0.5, 'win': 7.0, 'time': -0.001}


@scenario
def head_on_empty():
    # two heads into the same empty cell: both die, nobody is credited (C2)
    return dict(H=8, W=8, snakes=[[(3, 2), (3, 1)], [(3, 4), (3, 5)], [(6, 3), (6, 2)]],
                actions=[[0, 0, 0], [0, 0, 0]])


@scenario
def head_on_fruit():
    # two heads onto a fruit: both die, fruit stays, fruit_taken still draws one more (C3)
    return dict(H=8, W=8, snakes=[[(3, 2), (3, 1)], [(3, 4), (3, 5)], [(6, 3), (6, 2)]],
                fruits=[(3, 3)], actions=[[0, 0, 0], [0, 0, 0]])


@scenario
def head_swap():
    # adjacent heads moving into each other's head cell: both die, both get a kill (C2)
    return dict(H=8, W=8, snakes=[[(3, 3), (3, 2)], [(3, 4), (3, 5)], [(6, 3), (6, 2)]],
                actions=[[0, 0, 0], [0, 0, 0]])


@scenario
def self_bite():
    # snake 0 (length 5) turns into its own body: reward kill+lose to itself (C2)
    return dict(H=9, W=9, snakes=[[(3, 3), (3, 4), (4, 4), (4, 3), (4, 2)], [(7, 6), (7, 7)]],
                actions=[[1, 0], [0, 0]])


@scenario
def body_hit_credit_dead_owner():
    # 0 hits 1's body while 1 itself dies on the wall the same step; 1 is still paid the kill
    return dict(H=8, W=8, snakes=[[(3, 1), (4, 1)], [(1, 2), (2, 2), (3, 2), (4, 2)], [(6, 5), (6, 4)]],
                actions=[[2, 0, 0], [0, 0, 0]])


@scenario
def tail_follow_ok():
    # moving into another snake's tail cell is legal when that snake does not grow (C1, U1)
    return dict(H=8, W=8, snakes=[[(3, 2), (3, 1)], [(3, 5), (3, 4), (3, 3)], [(6, 5), (6, 4)]],
                actions=[[0, 0, 0], [0, 0, 0], [0, 0, 0]])


@scenario
def tail_follow_reverse_index():
    # same with the follower having the higher index (update order must not matter)
    return dict(H=8, W=8, snakes=[[(3, 5), (3, 4), (3, 3)], [(3, 2), (3, 1)], [(6, 5), (6, 4)]],
                actions=[[0, 0, 0], [0, 0, 0], [0, 0, 0]])


@scenario
def tail_growth_kill():
    # 1 eats a fruit so its tail stays; 0 moves into that tail and is killed by the growth rule (C4)
    return dict(H=8, W=8, snakes=[[(3, 2), (3, 1)], [(3, 5), (3, 4), (3, 3)], [(6, 5), (6, 4)]],
                fruits=[(3, 6)], actions=[[0, 0, 0], [0, 0, 0]])


@scenario
def tail_growth_double_count():
    # two snakes collide head-on in the cell that is the tail of a fruit eater: the counter is
    # decremented twice per victim and under-runs (C4); with 4 snakes counter reaches 0 while 2 live
    return dict(H=9, W=9, snakes=[[(3, 2), (3, 1)], [(3, 4), (3, 5)], [(5, 3), (4, 3), (3, 3)],
                                  [(7, 6), (7, 5)]],
                fruits=[(6, 3)], actions=[[0, 0, 0, 0], [0, 0, 0, 0], [0, 0, 0, 0]])


@scenario
def win_every_step():
    # counter == 1 pays the win reward on every step it holds (C5)
    return dict(H=8, W=8, snakes=[[(3, 2), (3, 1)], None, None], counter=1,
                actions=[[0, 0, 0], [2, 0, 0], [0, 0, 0]])


@scenario
def wall_and_step_cap():
    return dict(H=7, W=7, snakes=[[(1, 4), (1, 3)], [(4, 2), (4, 3)]], kw=dict(max_episode_steps=3),
                actions=[[0, 0], [0, 0], [0, 0], [0, 0]])


@scenario
def len2_and_die_with_overwritten_tail():
    # 1 (len 2) dies on the wall while 0's head takes 1's tail cell: tail cell must survive as HEAD_0
    return dict(H=8, W=8, snakes=[[(2, 4), (2, 3)], [(1, 5), (2, 5)], [(6, 5), (6, 4)]],
                actions=[[0, 0, 0], [0, 0, 0]])


@scenario
def die_with_overwritten_tail_reverse():
    return dict(H=8, W=8, snakes=[[(1, 5), (2, 5)], [(2, 4), (2, 3)], [(6, 5), (6, 4)]],
                actions=[[0, 0, 0], [0, 0, 0]])


@scenario
def eat_and_grow_crop_stack():
    # growth, respawn draw, egocentric crop near a corner, frame stack of 3
    return dict(H=8, W=10, snakes=[[(1, 2), (1, 1)], [(6, 7), (6, 8)]], fruits=[(1, 3), (6, 6)],
                kw=dict(vision_range=2, frame_stack=3),
                actions=[[0, 0], [0, 0], [2, 1], [0, 0], [2, 2]])


@scenario
def human_absolute_actions():
    # observer='human' (:610-632): 0 heads RIGHT, 1 heads UP.  Step 1: 'up' turns 0; 1 is already vertical
    # and ignores it.  Step 2: 'left' turns 0, 'right' turns 1.  Step 3: 0 moves horizontally and ignores
    # 'left', 'down' turns 1.  Step 4: the unknown action 7 is a no-op (no KeyError) and 0 runs into the wall.
    return dict(H=9, W=9, snakes=[[(5, 3), (5, 2), (5, 1)], [(5, 6), (6, 6), (7, 6)]],
                kw=dict(observer='human', vision_range=2),
                actions=[[4, 4], [1, 2], [1, 3], [7, 0]])


def run_scenarios():
    if ONLY and 'scenarios' not in ONLY:
        return
    out = {}
    names = []
    for fn in SCENARIOS:
        sc = fn()
        name = fn.__name__
        names.append(name)
        kw = dict(reward_dict=REW)
        kw.update(sc.get('kw', {}))
        env = build_env(sc['H'], sc['W'], sc['snakes'], sc.get('fruits', ()), sc.get('counter'), **kw)
        H, W = env.grid_shape
        alive, dirs, lens, cells = snake_cells(env, W)
        pre = f'{name}__'
        out[pre + 'H'] = np.array(H)
        out[pre + 'W'] = np.array(W)
        out[pre + 'kw'] = np.array(repr(kw))
        out[pre + 'grid0'] = env.grid.astype(np.uint8)
        out[pre + 'alive0'] = alive
        out[pre + 'dir0'] = dirs
        out[pre + 'len0'] = lens
        out[pre + 'cells0'] = cells
        out[pre + 'counter0'] = np.array(env.alive_snakes)
        tap = DrawTap()
        G, R, D, O, C, draws, draws_end = [], [], [], [], [], [], []
        np.random.seed(1234)
        with tap:
            for a in sc['actions']:
                obs, rew, done, info = env.step(list(a))
                draws.extend(tap.drain(env.num_snakes))
                draws_end.append(len(draws))
                G.append(env.grid.astype(np.uint8).copy())
                R.append(np.asarray(rew, dtype=np.float64))
                D.append(np.asarray(done, dtype=np.uint8))
                O.append(pack_obs(obs))
                C.append(env.alive_snakes)
        out[pre + 'actions'] = np.asarray(sc['actions'], dtype=np.uint8)
        out[pre + 'grid'] = np.stack(G)
        out[pre + 'rewards'] = np.stack(R)
        out[pre + 'dones'] = np.stack(D)
        out[pre + 'obs'] = np.stack(O)
        out[pre + 'counter'] = np.asarray(C, dtype=np.int32)
        out[pre + 'draws'] = np.asarray(draws, dtype=np.int32)
        out[pre + 'draws_end'] = np.asarray(draws_end, dtype=np.int32)
        print(f'scenario {name}: rewards {[list(np.round(r, 4)) for r in R]} counter {C}')
    out['names'] = np.array(names)
    np.savez_compressed(os.path.join(HERE, 'scenarios.npz'), **out)


def spawn_tables():
    if ONLY and 'spawn_tables' not in ONLY:
        return
    out = {}
    for (H, W, k) in [(20, 20, 3), (8, 8, 2), (10, 14, 4), (12, 12, 5), (7, 9, 6)]:
        grid = make_grid(H, W, empty_value=0, wall_value=1)
        cands = np.asarray(dfs_sweep_empty(grid, k), dtype=np.int16)
        out[f'c_{H}_{W}_{k}'] = cands
        print(f'spawn table {H}x{W} k={k}: {len(cands)} candidates')
    # spawn tables on the reference's asset maps (custom wall layouts, SURVEY N4)
    for name, k, mapper in [('12x12.txt', 4, None), ('20x20_cross.txt', 3, None),
                            ('40x40_ml2.txt', 3, {'#': 1, '.': 0, 'O': 1})]:
        grid = load_asset_map(name, mapper)
        cands = np.asarray(dfs_sweep_empty(grid, k), dtype=np.int16)
        tag = name.split('.')[0]
        out[f'map_{tag}__walls'] = (grid != 0).astype(np.uint8)
        out[f'map_{tag}__k'] = np.array(k)
        out[f'map_{tag}__cands'] = cands
        print(f'spawn table on {name} k={k}: {len(cands)} candidates')
    # turn table, probed from the reference's trigonometric _next_direction
    env = gym.make('Snake-v1')
    out['turn'] = np.array([[DIRS.index(env._next_direction(d, a)) for a in range(3)] for d in DIRS],
                           dtype=np.int8)
    np.savez_compressed(os.path.join(HERE, 'spawn_tables.npz'), **out)


def render_frames():
    """Pixels of the reference's three drawings -- render_fancy (snake_env.py:165-263), render('rgb_array')
    (grid_util.py:164-174) and one render('gif') frame (:177-185) -- together with the state they were drawn from."""
    if ONLY and 'render' not in ONLY:
        return
    out, names = {}, []
    cases = [('r20', dict(height=20, width=20, num_snakes=4, snake_length=5), 30, [0, 7, 19, 33]),
             ('r12', dict(height=12, width=16, num_snakes=6, snake_length=3, num_fruits=5), 40, [0, 9, 15]),
             ('r9', dict(height=9, width=9, num_snakes=2, snake_length=3), 17, [0, 4])]
    for tag, kw, cs, when in cases:
        env = gym.make('Snake-v1', **kw)
        np.random.seed(31 + cs)
        env.reset()
        rng = np.random.RandomState(cs)
        H, W = env.grid_shape
        for t in range(max(when) + 1):
            if t in when:
                name = f'{tag}_t{t}'
                names.append(name)
                alive, dirs, lens, cells = snake_cells(env, W)
                out[f'{name}__grid'] = env.grid.astype(np.uint8).copy()
                out[f'{name}__alive'], out[f'{name}__dir'], out[f'{name}__len'] = alive, dirs, lens
                out[f'{name}__cells'] = cells
                out[f'{name}__cell_size'] = np.array(cs)
                out[f'{name}__fancy'] = np.asarray(env.render_fancy(cell_size=cs))
                out[f'{name}__rgb'] = np.asarray(env.render('rgb_array'))
                env.frame_buffer = []
                env.render('gif')
                out[f'{name}__gif'] = np.asarray(env.frame_buffer[0])
            _, _, done, _ = env.step([int(a) for a in rng.randint(0, 3, size=env.num_snakes)])
            if all(done):
                env.reset()
    out['names'] = np.array(names)
    path = os.path.join(HERE, 'render.npz')
    np.savez_compressed(path, **out)
    print(f'render: {len(names)} frames, {os.path.getsize(path) / 1024:.1f} KiB')


if __name__ == '__main__':
    render_frames()
    custom = {'fruit': 1.0, 'kill': 2.0, 'lose': 3.0, 'win': 4.0, 'time': 0.1}
    cfg4_rew = {'fruit': 10.0, 'kill': 1.0, 'lose': -1.0, 'win': 0.1, 'time': -0.001}
    spawn_tables()
    run_scenarios()
    rollout('roll_cfg1', 100, 8, 200, height=20, width=20, num_snakes=4, snake_length=3,
            vision_range=5, frame_stack=1)
    rollout('roll_full', 200, 4, 120, height=20, width=20, num_snakes=4, snake_length=3)
    rollout('roll_fs4', 300, 4, 150, height=20, width=20, num_snakes=4, snake_length=3,
            vision_range=5, frame_stack=4)
    rollout('roll_big', 400, 2, 120, height=16, width=16, num_snakes=6, snake_length=5,
            vision_range=7, reward_dict=cfg4_rew)
    rollout('roll_single', 500, 4, 150, height=10, width=10, num_snakes=1, snake_length=3,
            num_fruits=4, reward_dict=custom)
    rollout('roll_cap', 600, 6, 60, height=8, width=8, num_snakes=2, snake_length=2,
            max_episode_steps=7, reward_dict=custom)
    rollout('roll_rect', 700, 4, 120, height=10, width=14, num_snakes=3, snake_length=4,
            vision_range=3, frame_stack=2, reward_dict=cfg4_rew)
    rollout('roll_coop', 900, 4, 120, env_id='SnakeCoop-v1', height=12, width=12, num_snakes=3, snake_length=3,
            vision_range=3, frame_stack=2, reward_dict=cfg4_rew)
    rollout('roll_crowd', 800, 4, 100, height=9, width=9, num_snakes=5, snake_length=3,
            vision_range=2, num_fruits=6, reward_dict=cfg4_rew)
    rollout('roll_cfg4', 1100, 1, 90, height=64, width=64, num_snakes=16, snake_length=5, vision_range=7,
            max_episode_steps=45, reward_dict=cfg4_rew)            # BASELINE cfg4 shape; the cap forces one auto-reset
    cross = load_asset_map('20x20_cross.txt')
    rollout('roll_map_cross', 1200, 4, 150, height=20, width=20, num_snakes=4, snake_length=3, vision_range=5,
            wall_map=cross.tolist())                                   # assets/20x20_cross.txt, the cfg1 shape otherwise
    small = load_asset_map('12x12.txt')
    rollout('roll_map_12', 1300, 4, 120, height=12, width=12, num_snakes=3, snake_length=4, frame_stack=2,
            num_fruits=5, reward_dict=cfg4_rew, wall_map=small.tolist())   # assets/12x12.txt, full-grid observation
    ml2 = load_asset_map('40x40_ml2.txt', {'#': 1, '.': 0, 'O': 1})
    rollout('roll_map_ml2', 1400, 2, 100, height=40, width=40, num_snakes=8, snake_length=3, vision_range=4,
            max_episode_steps=35, num_fruits=10, reward_dict=cfg4_rew, wall_map=ml2.tolist())   # direction-plane record (> 6 snakes)
    rollout('roll_human', 1000, 4, 150, height=12, width=12, num_snakes=3, snake_length=3,
            vision_range=4, observer='human', reward_dict=cfg4_rew)
