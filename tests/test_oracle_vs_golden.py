"""Pins oracle/snake_oracle.py to the reference: committed golden vectors (always) and the
live reference under the same np.random seed (where the original project is there: its checkout at
SNK_REFERENCE_DIR or BASELINE.json's reference_path, or its install in oracle/_ref)."""
import functools
import hashlib
import os
import sys

import numpy as np
import pytest

from golden_util import GOLDEN_DIR, ROLLOUTS, Rollout, load_map_spawn_tables, load_scenarios, load_spawn_tables, unpack_obs
from oracle.cpu_runner import reference_search_path
from oracle.snake_oracle import (CoopOracleSnakeEnv, OracleSnakeEnv, ReplayDraws, RecordingDraws, TURN,
                                 spawn_candidates, competition_rank)


def test_spawn_tables_and_turn_table():
    tables, turn = load_spawn_tables()
    for (H, W, k), ref in tables.items():
        mine = spawn_candidates(H, W, k)
        assert mine.shape == ref.shape, (H, W, k)
        assert np.array_equal(mine, ref), (H, W, k)
    assert np.array_equal(np.asarray(TURN), turn)


def test_spawn_tables_on_the_reference_asset_maps():
    """dfs_sweep_empty on custom wall layouts (assets/12x12.txt, 20x20_cross.txt, 40x40_ml2.txt; SURVEY N4)."""
    maps = load_map_spawn_tables()
    assert set(maps) == {'12x12', '20x20_cross', '40x40_ml2'}
    for name, (walls, k, ref) in maps.items():
        mine = spawn_candidates(walls.shape[0], walls.shape[1], k, walls)
        assert mine.shape == ref.shape and np.array_equal(mine, ref), name


@pytest.mark.parametrize('name', ROLLOUTS)
def test_rollout_replay(name):
    g = Rollout(name)
    for e in range(g.num_envs):
        ge = g.env[e]
        cls = CoopOracleSnakeEnv if g.done_mode else OracleSnakeEnv
        env = cls(draws=ReplayDraws(ge['draws']), **g.kwargs)
        obs = env.reset()
        assert np.array_equal(obs, unpack_obs(ge['obs0']))
        assert np.array_equal(env.grid, ge['grid0'])
        assert env.draws.pos == ge['draws_end'][0]
        k = 0
        for t in range(g.steps):
            obs, rew, done, info = env.step([int(a) for a in ge['actions'][t]])
            assert np.array_equal(env.grid, ge['grid_step'][t]), (name, e, t)
            assert env.alive_counter == ge['counter'][t], (name, e, t)
            if info:
                assert ge['info_step'][k] == t
                assert list(info['rank']) == list(ge['info_rank'][k])
                assert np.array_equal(info['episode_scores'], ge['info_scores'][k])
                assert np.array_equal(info['episode_steps'], ge['info_steps'][k])
                assert np.array_equal(info['episode_fruits'], ge['info_fruits'][k])
                assert np.array_equal(info['episode_kills'], ge['info_kills'][k])
                k += 1
            if all(done):
                obs = env.reset()
            assert np.array_equal(np.asarray(rew), ge['rewards'][t]), (name, e, t)
            assert np.array_equal(np.asarray(done, dtype=np.uint8), ge['dones'][t]), (name, e, t)
            assert np.array_equal(obs, unpack_obs(ge['obs'][t])), (name, e, t)
            assert np.array_equal(env.grid, ge['grid_live'][t])
            assert env.draws.pos == ge['draws_end'][t + 1]
        assert k == len(ge['info_step'])


@pytest.mark.parametrize('sc', load_scenarios(), ids=lambda s: s.name)
def test_scenarios(sc):
    env = OracleSnakeEnv(height=sc.H, width=sc.W, num_snakes=sc.num_snakes, snake_length=2,
                         draws=ReplayDraws(sc.draws), **sc.kwargs)
    env.import_state(sc.grid0, sc.alive0, sc.dir0, sc.len0, sc.cells0, sc.counter0)
    for t, a in enumerate(sc.actions):
        obs, rew, done, info = env.step([int(x) for x in a])
        assert np.array_equal(env.grid, sc.grid[t]), (sc.name, t)
        assert np.array_equal(np.asarray(rew), sc.rewards[t]), (sc.name, t)
        assert np.array_equal(np.asarray(done, dtype=np.uint8), sc.dones[t])
        assert env.alive_counter == sc.counter[t]
        assert np.array_equal(obs, unpack_obs(sc.obs[t])), (sc.name, t)
        assert env.draws.pos == sc.draws_end[t]


def test_rank_rule():
    assert list(competition_rank([0.0, 1000.5])) == [2, 1]
    assert list(competition_rank([3.0, 3.0, 1.0, 5.0])) == [2, 2, 4, 1]


def test_reward_dict_keys_and_action_errors():
    with pytest.raises(KeyError):
        OracleSnakeEnv(reward_dict={'fruit': 1.0})
    env = OracleSnakeEnv(num_snakes=2)
    np.random.seed(3)
    env.reset()
    with pytest.raises(AssertionError):
        env.step([0])
    with pytest.raises(KeyError):
        env.step([0, 3])


# ------------------------------------------------------------------ the cases run against the live reference
SAME_SEED = [
    dict(height=20, width=20, num_snakes=4, snake_length=3, vision_range=5),
    dict(height=12, width=9, num_snakes=3, snake_length=4, vision_range=2, frame_stack=3,
         reward_dict={'fruit': 1.5, 'kill': 2.0, 'lose': -3.0, 'win': 4.0, 'time': 0.1}),
    dict(height=8, width=8, num_snakes=5, snake_length=2, num_fruits=7, max_episode_steps=25),
]
WALL_MAPS = [
    ('12x12', dict(num_snakes=3, snake_length=4, vision_range=3, frame_stack=2)),
    ('20x20_cross', dict(num_snakes=4, snake_length=3, vision_range=5)),
]
FINISHED = [
    dict(height=9, width=9, num_snakes=3, snake_length=3, vision_range=2, max_episode_steps=6, num_fruits=2),
    dict(height=8, width=10, num_snakes=2, snake_length=2, frame_stack=2, num_fruits=1),
]
LIVE_GOLDEN = os.path.join(GOLDEN_DIR, 'live_cases.npz')


def small_fuzz_configs(n, seed):
    """Seeded random small shapes (the reference re-enumerates every spawn pose on each reset, so grids stay
    <= 13 cells wide); shared with the host-simulation fuzz.  num_fruits >= 1: with 0 the reference's reset
    executes `grid[None, None] = FRUIT` (snake_env.py:147-148 has no None guard), which paints the WHOLE grid,
    walls included, and the snakes then walk out of the array -- a crash path, not a behaviour to match."""
    rng = np.random.RandomState(seed)
    out = []
    while len(out) < n:
        H, W = int(rng.randint(6, 14)), int(rng.randint(6, 14))
        ns, K = int(rng.randint(1, 7)), int(rng.randint(2, 5))
        if ns * K * 5 > (H - 2) * (W - 2):
            continue
        kw = dict(height=H, width=W, num_snakes=ns, snake_length=K,
                  vision_range=[None, 1, 2, 3, 4][rng.randint(0, 5)], frame_stack=int([1, 1, 2, 3][rng.randint(0, 4)]),
                  num_fruits=int(rng.randint(1, 9)), max_episode_steps=int([10000, 15, 6][rng.randint(0, 3)]),
                  observer=['snake', 'snake', 'human'][rng.randint(0, 3)],
                  reward_dict={'fruit': float(rng.randint(1, 9)), 'kill': 0.25 * rng.randint(0, 9),
                               'lose': -0.125 * rng.randint(0, 9), 'win': 0.5 * rng.randint(0, 5),
                               'time': -0.001 * rng.randint(0, 5)})
        out.append((kw, ['Snake-v1', 'Snake-v1', 'SnakeCoop-v1'][rng.randint(0, 3)]))
    return out


def wall_map_kw(name, kw):
    walls, _, _ = load_map_spawn_tables()[name]
    return dict(height=walls.shape[0], width=walls.shape[1], wall_map=walls.astype(np.int64), **kw)


@functools.lru_cache(maxsize=None)
def live_cases():
    """name -> (kw, env_id, steps, n_actions, reset_on_done) of every case the live-reference tests run."""
    cases = {f'same_seed_{i}': (kw, 'Snake-v1', 400, 3, True) for i, kw in enumerate(SAME_SEED)}
    for name, kw in WALL_MAPS:
        cases[f'wall_map_{name}'] = (wall_map_kw(name, kw), 'Snake-v1', 250, 3, True)
    for i, kw in enumerate(FINISHED):
        cases[f'finished_{i}'] = (kw, 'Snake-v1', 60, 3, False)
    for i, (kw, env_id) in enumerate(small_fuzz_configs(24, 777)):
        cases[f'fuzz_{i}'] = (kw, env_id, 150, 5 if kw['observer'] == 'human' else 3, True)
    return cases


def trajectory(make, ns, steps, n_actions=3, reset_on_done=True):
    """The live comparison's protocol: np.random.seed(42), make, reset, then `steps` steps of RandomState(5) actions,
    resetting on all(done) when reset_on_done.  Returns [reset obs, (obs, rewards, dones, info keys, info values,
    grid) per step]."""
    acts = np.random.RandomState(5).randint(0, n_actions, size=(steps, ns))
    np.random.seed(42)
    env = make()
    out = [env.reset()]
    for a in acts:
        o, r, d, info = env.step([int(x) for x in a])
        if all(d) and reset_on_done:
            o = env.reset()
        out.append((o, list(r), list(d), sorted(info.keys()),
                    [list(np.asarray(info[k], dtype=np.float64)) for k in sorted(info.keys())],
                    np.asarray(env.grid).copy()))
    return out


def digests(traj):
    """8-byte SHA-256 prefixes, one row for the reset observation and one per step over (obs, rewards, dones,
    info, grid) in fixed dtypes: a whole trajectory pinned in a few bytes per step."""
    def h(*arrays, text=''):
        m = hashlib.sha256(text.encode())
        for x in arrays:
            m.update(repr(x.shape).encode() + x.tobytes())
        return np.frombuffer(m.digest()[:8], np.uint8)
    rows = [h(np.asarray(traj[0], np.uint8))]
    for o, r, d, keys, vals, grid in traj[1:]:
        rows.append(h(np.asarray(o, np.uint8), np.asarray(r, np.float64), np.asarray(d, np.uint8),
                      np.asarray([x for v in vals for x in v], np.float64), np.asarray(grid, np.int64),
                      text=repr([(k, len(v)) for k, v in zip(keys, vals)])))
    return np.stack(rows)


def oracle_record(name):
    """The oracle's trajectory of one live case as stored in tests/golden/live_cases.npz."""
    kw, env_id, steps, n_actions, reset_on_done = live_cases()[name]
    cls = CoopOracleSnakeEnv if env_id == 'SnakeCoop-v1' else OracleSnakeEnv
    traj = trajectory(lambda: cls(**kw), kw['num_snakes'], steps, n_actions, reset_on_done)
    return {'digest': digests(traj), 'rewards': np.asarray([t[1] for t in traj[1:]], np.float64),
            'dones': np.asarray([t[2] for t in traj[1:]], np.uint8)}


@pytest.mark.parametrize('name', sorted(live_cases()))
def test_live_reference_cases_against_stored_trajectories(name):
    """Every case of the live-reference tests below, on every run: the oracle against the trajectory stored for it
    in tests/golden/live_cases.npz (made by tests/golden/make_live_cases.py from this oracle; the live tests check
    the oracle against the original project wherever it is installed)."""
    want = np.load(LIVE_GOLDEN)
    got = oracle_record(name)
    assert np.array_equal(got['rewards'], want[f'{name}_rewards']), name
    assert np.array_equal(got['dones'], want[f'{name}_dones']), name
    bad = np.flatnonzero((got['digest'] != want[f'{name}_digest']).any(1))
    assert got['digest'].shape == want[f'{name}_digest'].shape and bad.size == 0, \
        f'{name}: first differing row {bad[:1]} (row 0 = reset, row t + 1 = step t)'


# ------------------------------------------------------------------ live reference (reference_search_path)
def _drop_gym_and_marlenv():
    for m in [m for m in sys.modules if m == 'gym' or m.startswith('gym.') or m == 'marlenv' or m.startswith('marlenv.')]:
        del sys.modules[m]


def _compare_with_live_reference(kw, env_id='Snake-v1', steps=400, n_actions=3, reset_on_done=True):
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    ref_pkg = reference_search_path()
    sys.path.insert(0, os.path.join(root, 'oracle', 'gym_stub'))
    sys.path.insert(1, ref_pkg)
    _drop_gym_and_marlenv()                  # this repository's `marlenv` import shim may already be loaded
    try:
        import gym
        import marlenv  # noqa: F401
        assert marlenv.__file__.startswith(ref_pkg), marlenv.__file__
        walls = kw.get('wall_map')
        ref_kw = {k: v for k, v in kw.items() if k != 'wall_map'}
        if walls is not None:     # the reference has no map parameter: its reset() gets the layout from `make_grid`
            import marlenv.envs.snake_env as ref_snake_env
            ref_snake_env.make_grid = lambda *a, **k: np.asarray(walls).copy()

        cls = CoopOracleSnakeEnv if env_id == 'SnakeCoop-v1' else OracleSnakeEnv
        ns = kw['num_snakes']
        ref = trajectory(lambda: gym.make(env_id, **ref_kw), ns, steps, n_actions, reset_on_done)
        mine = trajectory(lambda: cls(**kw), ns, steps, n_actions, reset_on_done)
        assert np.array_equal(ref[0], mine[0])
        for t, (a, b) in enumerate(zip(ref[1:], mine[1:])):
            assert np.array_equal(a[0], b[0]), (t, kw)
            assert a[1] == b[1] and a[2] == b[2] and a[3] == b[3] and a[4] == b[4], (t, kw)
            assert np.array_equal(a[5], b[5]), (t, kw)
    finally:
        sys.path.remove(os.path.join(root, 'oracle', 'gym_stub'))
        sys.path.remove(ref_pkg)
        _drop_gym_and_marlenv()


@pytest.mark.needs_reference
@pytest.mark.parametrize('kw', SAME_SEED)
def test_same_seed_as_live_reference(kw):
    _compare_with_live_reference(kw)


@pytest.mark.needs_reference
@pytest.mark.parametrize('name,kw', WALL_MAPS)
def test_custom_wall_map_same_seed_as_live_reference(name, kw):
    """SURVEY N4: the oracle on a custom wall layout against the reference whose reset() is handed the same layout."""
    _compare_with_live_reference(wall_map_kw(name, kw), steps=250)


@pytest.mark.needs_reference
@pytest.mark.parametrize('kw', FINISHED)
def test_stepping_a_finished_env_like_the_live_reference(kw):
    """No reset after the episode ends (SURVEY E1, probe g3): the reference keeps stepping -- capped episodes
    move on, dead snakes return 0 / True, info is emitted again every step."""
    _compare_with_live_reference(kw, steps=60, reset_on_done=False)


@pytest.mark.needs_reference
@pytest.mark.parametrize('case', range(24))
def test_oracle_fuzz_vs_live_reference(case):
    """The oracle against the unmodified reference under the same np.random seed on seeded random shapes,
    both env ids and both observers."""
    kw, env_id = small_fuzz_configs(24, 777)[case]
    _compare_with_live_reference(kw, env_id, steps=150, n_actions=5 if kw['observer'] == 'human' else 3)


def test_recording_roundtrip():
    rec = RecordingDraws()
    np.random.seed(9)
    env = OracleSnakeEnv(num_snakes=3, vision_range=3, draws=rec)
    acts = np.random.RandomState(1).randint(0, 3, size=(150, 3))
    trace = [env.reset()]
    for a in acts:
        o, r, d, _ = env.step(list(a))
        if all(d):
            o = env.reset()
        trace.append(o)
    env2 = OracleSnakeEnv(num_snakes=3, vision_range=3, draws=ReplayDraws(rec.log))
    trace2 = [env2.reset()]
    for a in acts:
        o, r, d, _ = env2.step(list(a))
        if all(d):
            o = env2.reset()
        trace2.append(o)
    assert all(np.array_equal(a, b) for a, b in zip(trace, trace2))
