"""CPU oracle for the Snake-v1 step path  --  TEST INFRASTRUCTURE, NOT PRODUCT CODE.

A from-scratch restatement (NumPy + small Python loops) of the algorithm in the
reference `tranthai189765/MARL-Snake` (fork of kc-ml2/marlenv).  Only `tests/`,
`__graft_entry__.smoke()` and `bench.py`'s cpu_baseline / `--impl reference` leg
may import this module; the product path (marl-snake_b200/) never does and fails
loudly when its CUDA library is missing.

Parity status: PINNED.  `tests/test_oracle_vs_golden.py` checks this file
against trajectories recorded from the *unmodified* reference
(`tests/golden/*.npz`, produced by `tests/golden/make_golden.py` which imports
the original project's checkout (SNK_REFERENCE_DIR, default BASELINE.json's
reference_path) behind `oracle/gym_stub`).  Where the original is there (that
checkout or its install in oracle/_ref) the same test module
additionally runs it live under the same `np.random.seed` and compares every step.

Reference lines each function follows (paths relative to marlenv/marlenv/ of the
original project):

  spawn_candidates      core/grid_util.py:73-115   dfs_sweep_empty/_dfs_helper/_head_blocked
  OracleSnakeEnv.reset  envs/snake_env.py:131-159, 576-596; core/snake.py:53-74;
                        core/grid_util.py:14-20, 126-133
  OracleSnakeEnv.step   envs/snake_env.py:301-414 (+ _check_collision :521-544,
                        _update_grid :546-566, Snake.move core/snake.py:96-107)
  turn table            envs/snake_env.py:598-608 (_next_direction)
  encode / crop / stack envs/snake_env.py:444-519
  auto-reset            wrappers.py:138-146 (VectorOracle)

RNG: the reference draws from the module-global legacy `np.random`
(snake_env.py:581, grid_util.py:130).  `NumpyGlobalDraws` issues exactly the
same calls in the same order, so under one `np.random.seed(s)` the oracle and
the reference produce identical trajectories.  `RecordingDraws` logs the draw
*outputs* (accepted spawn-candidate indices, fruit ranks) and `ReplayDraws`
feeds such a log back; that log is what the CUDA replay mode consumes.
"""
from collections import deque
from functools import lru_cache

import numpy as np

EMPTY, WALL, FRUIT, HEAD, BODY, TAIL = 0, 1, 2, 3, 4, 5     # core/snake.py:5-11
# direction codes: 0 UP, 1 RIGHT, 2 DOWN, 3 LEFT as (dr, dc)   core/snake.py:33-37
DELTA = ((-1, 0), (0, 1), (1, 0), (0, -1))
# action 0 keeps, 1 turns left (code-1), 2 turns right (code+1)  snake_env.py:598-608
TURN = tuple(tuple(((d + s) % 4) for s in (0, -1, 1)) for d in range(4))
# neighbour order used by the spawn DFS, as (dr, dc)   core/grid_util.py:7-11
DFS_SHIFTS = ((0, 1), (1, 0), (0, -1), (-1, 0))

DEFAULT_REWARD = {'fruit': 10.0, 'kill': 0.0, 'lose': -0.5, 'win': 0.0, 'time': -0.001}
REWARD_KEYS = DEFAULT_REWARD.keys()
DEFAULT_MAX_EPISODE_STEPS = 1e4


# --------------------------------------------------------------------------- spawn table
def spawn_candidates(height, width, length, wall_map=None):
    """All spawn poses in the reference's enumeration order; wall_map (H x W, nonzero = wall) replaces make_grid's
    walled box by a custom layout (dfs_sweep_empty takes whatever grid reset() built, snake_env.py:578)."""
    key = None if wall_map is None else np.ascontiguousarray(np.asarray(wall_map) != 0, dtype=np.uint8).tobytes()
    return _spawn_candidates(height, width, length, key)


@lru_cache(maxsize=None)
def _spawn_candidates(height, width, length, wall_bytes):
    """

    Returns an int array [n_cand, length, 2] of (row, col), head first.
    Follows core/grid_util.py:73-115 on the empty walled grid of make_grid
    (:14-20): start cells row-major, neighbours in DFS_SHIFTS order, a pose is
    dropped when all four neighbours of its first cell are wall / own body /
    the cell about to be appended (_head_blocked, :102-110).
    """
    free = np.zeros((height, width), dtype=bool)
    if wall_bytes is None:
        free[1:height - 1, 1:width - 1] = True
    else:
        free = np.frombuffer(wall_bytes, dtype=np.uint8).reshape(height, width) == 0
    out = []

    def head_boxed(path, extra):
        r0, c0 = path[0]
        for dr, dc in DFS_SHIFTS:
            n = (r0 + dr, c0 + dc)
            if 0 <= n[0] < height and 0 <= n[1] < width and free[n] and n not in path and n != extra:
                return False
        return True

    def grow(path):
        if len(path) == length:
            out.append(list(path))
            return
        r, c = path[-1]
        for dr, dc in DFS_SHIFTS:
            n = (r + dr, c + dc)
            if 0 <= n[0] < height and 0 <= n[1] < width and free[n] and n not in path:
                if not head_boxed(path, n):
                    path.append(n)
                    grow(path)
                    path.pop()

    for r in range(height):
        for c in range(width):
            if free[r, c]:
                grow([(r, c)])
    return np.asarray(out, dtype=np.int32).reshape(len(out), length, 2)


# --------------------------------------------------------------------------- draw sources
class NumpyGlobalDraws:
    """Issues the reference's own np.random calls (same stream under the same seed)."""

    def spawn(self, n_cand, ns, no_overlap):
        while True:                                   # snake_env.py:579-586
            pick = np.random.permutation(n_cand)[:ns]
            if no_overlap(pick):
                return [int(p) for p in pick]

    def fruit(self, n_empty, k):
        return [int(v) for v in np.random.randint(0, n_empty, size=k)]   # grid_util.py:130


class RecordingDraws:
    """Wraps a draw source and logs the outputs in consumption order."""

    def __init__(self, inner=None):
        self.inner = inner or NumpyGlobalDraws()
        self.log = []

    def spawn(self, n_cand, ns, no_overlap):
        pick = self.inner.spawn(n_cand, ns, no_overlap)
        self.log.extend(pick)
        return pick

    def fruit(self, n_empty, k):
        ranks = self.inner.fruit(n_empty, k)
        self.log.extend(ranks)
        return ranks


class ReplayDraws:
    """Feeds back a RecordingDraws log."""

    def __init__(self, log):
        self.log = [int(v) for v in log]
        self.pos = 0

    def _take(self, k):
        if self.pos + k > len(self.log):
            raise IndexError('replay log exhausted')
        out = self.log[self.pos:self.pos + k]
        self.pos += k
        return out

    def spawn(self, n_cand, ns, no_overlap):
        pick = self._take(ns)
        assert no_overlap(pick), 'replayed spawn overlaps'
        return pick

    def fruit(self, n_empty, k):
        ranks = self._take(k)
        assert all(0 <= r < n_empty for r in ranks), 'replayed fruit rank out of range'
        return ranks


def next_direction_global(direction, action):
    """observer='human': absolute actions 0 noop, 1 left, 2 right, 3 down, 4 up.  A snake moving
    horizontally may only turn down/up, one moving vertically only left/right; anything else (including
    values outside 0..4) keeps the direction -- no KeyError on this path.  snake_env.py:610-632."""
    UP, RIGHT, DOWN, LEFT = 0, 1, 2, 3
    dr, dc = DELTA[direction]
    if dr == 0:                       # the reference's `direction.value[0] == 0`: moving left or right
        if action == 3:
            return DOWN
        if action == 4:
            return UP
    elif dc == 0:
        if action == 1:
            return LEFT
        if action == 2:
            return RIGHT
    return direction


# --------------------------------------------------------------------------- the env
class OracleSnakeEnv:
    """One Snake-v1 environment; same ctor kwargs / reset / step contract as SnakeEnv."""

    def __init__(self, height=20, width=20, num_snakes=4, snake_length=3, vision_range=None,
                 frame_stack=1, observer='snake', draws=None, wall_map=None, **kwargs):
        # wall_map: H x W, nonzero = wall -- reset() starts from this layout instead of make_grid's walled box
        # (the array make_grid_from_txt returns for an assets/*.txt map, core/grid_util.py:23-33)
        self.wall_map = None
        if wall_map is not None:
            self.wall_map = (np.asarray(wall_map) != 0).astype(np.int64)
            height, width = self.wall_map.shape
        reward_dict = kwargs.pop('reward_dict', DEFAULT_REWARD)
        if reward_dict.keys() != REWARD_KEYS:                              # snake_env.py:76-80
            raise KeyError(f'reward dict keys must correspond to {REWARD_KEYS}')
        if observer not in ('snake', 'human'):
            raise ValueError("observer must be 'snake' (three relative actions) or 'human' (five absolute)")
        self.observer = observer
        self.reward_dict = reward_dict
        self.max_episode_steps = kwargs.pop('max_episode_steps', DEFAULT_MAX_EPISODE_STEPS)
        self.num_snakes = num_snakes
        self.num_fruits = kwargs.pop('num_fruits', int(round(num_snakes * 0.8)))
        self.grid_shape = (height, width)
        self.snake_length = snake_length
        self.vision_range = vision_range
        self.frame_stack = frame_stack
        self.obs_ch = 8 * frame_stack
        self.draws = draws or NumpyGlobalDraws()
        hw = (2 * vision_range + 1,) * 2 if vision_range else self.grid_shape
        self.obs_shape = (num_snakes, *hw, self.obs_ch)

    # ---- reset ---------------------------------------------------------------------------
    def reset(self):
        H, W = self.grid_shape
        ns = self.num_snakes
        if self.wall_map is None:
            grid = np.zeros((H, W), dtype=np.int64)
            grid[0, :] = grid[H - 1, :] = WALL
            grid[:, 0] = grid[:, W - 1] = WALL
        else:
            grid = self.wall_map * WALL
        cands = spawn_candidates(H, W, self.snake_length, self.wall_map)

        def no_overlap(pick):                                              # snake_env.py:568-574
            cells = cands[list(pick)].reshape(-1, 2)
            return len({(int(r), int(c)) for r, c in cells}) == len(cells)

        pick = self.draws.spawn(len(cands), ns, no_overlap)
        self.body = []          # per snake: deque of (r, c), head first
        self.dir = []
        for i, p in enumerate(pick):
            cells = [(int(r), int(c)) for r, c in cands[p]]
            self.body.append(deque(cells))
            d = (cells[0][0] - cells[1][0], cells[0][1] - cells[1][1])     # core/snake.py:58-61
            self.dir.append(DELTA.index(d))
            for rc in cells:
                grid[rc] = BODY + 10 * i
            grid[cells[0]] = HEAD + 10 * i
            grid[cells[-1]] = TAIL + 10 * i
        self.grid = grid
        self._place_fruit(self.num_fruits)
        self.alive = [True] * ns
        self.alive_counter = ns                                            # snake_env.py:150
        frame = self._encode()
        self.frames = deque([frame] * self.frame_stack, maxlen=self.frame_stack)
        self._zero_stats()
        self.episode_length = 0
        return self._stacked()

    def _place_fruit(self, k):
        if not k:
            return
        rows, cols = np.where(self.grid == EMPTY)                          # grid_util.py:127
        if len(rows) == 0:
            return
        ranks = self.draws.fruit(len(rows), k)
        self.grid[rows[ranks], cols[ranks]] = FRUIT

    def _zero_stats(self):
        ns = self.num_snakes
        self.epi_scores = np.zeros(ns)
        self.epi_steps = np.zeros(ns)
        self.epi_fruits = np.zeros(ns)
        self.epi_kills = np.zeros(ns)

    # ---- step ----------------------------------------------------------------------------
    def step(self, actions):
        ns = self.num_snakes
        if isinstance(actions, int):
            actions = [actions]
        assert len(actions) == ns
        actions = [a.item() if isinstance(a, np.ndarray) else a for a in actions]
        grid = self.grid
        was_alive = list(self.alive)

        # 1. turn + head advance, grouped by target cell in first-arrival order  (:318-330)
        arrivals = {}
        for i in range(ns):
            if was_alive[i]:
                if self.observer == 'human':
                    self.dir[i] = next_direction_global(self.dir[i], actions[i])
                else:
                    self.dir[i] = TURN[self.dir[i]][{0: 0, 1: 1, 2: 2}[actions[i]]]   # KeyError like the ref
                hr, hc = self.body[i][0]
                dr, dc = DELTA[self.dir[i]]
                arrivals.setdefault((hr + dr, hc + dc), []).append(i)

        # 2. collisions on the pre-move grid  (:521-544)
        died = [False] * ns
        ate = [False] * ns
        kills = [0] * ns
        won = [False] * ns
        fruit_taken = 0
        dead_set = set()
        eaters = []
        for cell, who in arrivals.items():
            code = int(grid[cell])
            kind = code % 10
            if len(who) > 1 or kind in (WALL, BODY, HEAD):
                dead_set.update(who)
                if kind == FRUIT:
                    fruit_taken += 1
                if kind in (BODY, HEAD):
                    kills[code // 10] += 1
            elif kind == FRUIT:
                eaters.extend(who)
                fruit_taken += 1

        # 3. death bookkeeping, tail-growth rule, win rule  (:334-352)
        self.alive_counter -= len(dead_set)
        for i in dead_set:
            died[i] = True
            self.alive[i] = False
        for e in eaters:
            tail = self.body[e][-1]
            for d in arrivals.get(tail, ()):
                died[d] = True
                self.alive[d] = False
                self.alive_counter -= 1
                kills[e] += 1
            ate[e] = True
        if self.alive_counter == 1 and ns > 1:
            for i in range(ns):
                if self.alive[i]:
                    won[i] = True
                    break

        # 4. rewards + grid update, snake by snake in index order  (:358-374, :546-566)
        rd = self.reward_dict
        rews, dones, fruits_f, kills_f = [], [], [], []
        for i in range(ns):
            if not was_alive[i]:
                rews.append(0.)
                fruits_f.append(0)
                kills_f.append(0)
            else:
                r = rd['time'] * self.alive[i]
                r += rd['fruit'] * ate[i]
                r += rd['lose'] * died[i]
                r += rd['kill'] * kills[i]
                r += rd['win'] * won[i]
                rews.append(r)
                fruits_f.append(float(ate[i]))
                kills_f.append(float(kills[i]))
                self._move_on_grid(i, ate[i])
            dones.append(not self.alive[i])

        # 5. fruit respawn  (:377-379)
        self._place_fruit(fruit_taken)

        # 6. observation  (:381, :461-472)
        self.frames.append(self._encode())
        obs = self._stacked()

        # 7. episode statistics, step cap, terminal info  (:385-412)
        mask = 1. - np.asarray(dones)
        self.epi_scores = self.epi_scores + mask * np.asarray(rews)
        self.epi_steps = self.epi_steps + mask * np.ones(ns)
        self.epi_fruits = self.epi_fruits + mask * np.asarray(fruits_f)
        self.epi_kills = self.epi_kills + mask * np.asarray(kills_f)
        info = {}
        self.episode_length += 1
        if self.episode_length >= self.max_episode_steps:
            dones = [True] * ns
        if self._done_fn(dones):
            info['rank'] = list(competition_rank(self.epi_scores))
            info.update(episode_scores=self.epi_scores, episode_steps=self.epi_steps,
                        episode_fruits=self.epi_fruits, episode_kills=self.epi_kills)
            self._zero_stats()
        return obs, rews, dones, info

    def _done_fn(self, dones):
        return all(dones)

    def _move_on_grid(self, i, grew):
        grid = self.grid
        body = self.body[i]
        tag = 10 * i
        if self.alive[i]:
            hr, hc = body[0]
            grid[hr, hc] = BODY + tag
            dr, dc = DELTA[self.dir[i]]
            body.appendleft((hr + dr, hc + dc))
            if not grew:
                old_tail = body.pop()
                if grid[old_tail] == TAIL + tag:          # may already hold another head (:555)
                    grid[old_tail] = EMPTY
            grid[body[0]] = HEAD + tag
            grid[body[-1]] = TAIL + tag
        else:
            cells = list(body)
            if grid[cells[-1]] // 10 != i:                # tail cell taken over by a head (:562)
                cells = cells[:-1]
            for rc in cells:
                grid[rc] = EMPTY
            # the reference still advances the dead body (core/snake.py:96-107); nothing
            # reads it afterwards, so the oracle just drops it.
            body.clear()

    # ---- observation -----------------------------------------------------------------------
    def _encode(self):
        """Per-viewer 8-channel one-hot, optionally cropped around the own head (:474-519)."""
        grid = self.grid
        ns = self.num_snakes
        H, W = self.grid_shape
        kind = grid % 10
        owner = grid // 10
        is_snake = (grid != EMPTY) & (grid != WALL) & (grid != FRUIT)
        full = np.zeros((ns, H, W, 8), dtype=np.uint8)
        full[..., 0] = grid == WALL
        full[..., 1] = grid == FRUIT
        for v in range(ns):
            mine = is_snake & (owner == v)
            other = is_snake & ~mine
            for k, part in enumerate((HEAD, BODY, TAIL)):
                full[v, :, :, 2 + k] = other & (kind == part)
                full[v, :, :, 5 + k] = mine & (kind == part)
        vr = self.vision_range
        if not vr:
            return full
        side = 2 * vr + 1
        out = np.zeros((ns, side, side, 8), dtype=np.uint8)
        for v in range(ns):
            flat = int(full[v, :, :, 5].argmax())          # 0 when the viewer has no head (:500)
            hr, hc = divmod(flat, W)
            r0, r1 = max(hr - vr, 0), min(hr + vr, H - 1)
            c0, c1 = max(hc - vr, 0), min(hc + vr, W - 1)
            out[v, r0 - hr + vr:r1 - hr + vr + 1, c0 - hc + vr:c1 - hc + vr + 1] = \
                full[v, r0:r1 + 1, c0:c1 + 1]
        return out

    def _stacked(self):
        return np.concatenate(list(self.frames), axis=-1).astype(np.uint8)   # oldest -> newest

    # ---- state export used by the parity harness ---------------------------------------------
    def export_state(self):
        ns = self.num_snakes
        W = self.grid_shape[1]
        head = np.full(ns, -1, dtype=np.int32)
        tail = np.full(ns, -1, dtype=np.int32)
        length = np.zeros(ns, dtype=np.int32)
        for i in range(ns):
            if self.alive[i]:
                head[i] = self.body[i][0][0] * W + self.body[i][0][1]
                tail[i] = self.body[i][-1][0] * W + self.body[i][-1][1]
                length[i] = len(self.body[i])
        return dict(grid=self.grid.astype(np.uint8), head=head, tail=tail, length=length,
                    dir=np.asarray(self.dir, dtype=np.int32),
                    alive=np.asarray(self.alive, dtype=np.uint8),
                    alive_counter=int(self.alive_counter),
                    episode_length=int(self.episode_length))


    def import_state(self, grid, alive, dirs, lens, cells, alive_counter, episode_length=0):
        """Force a hand-built state (scenario tests). cells[i] = head-first flat cell indices."""
        H, W = self.grid_shape
        self.grid = np.asarray(grid, dtype=np.int64).reshape(H, W).copy()
        self.alive = [bool(a) for a in alive]
        self.dir = [int(d) for d in dirs]
        self.body = [deque((int(c) // W, int(c) % W) for c in cells[i][:int(lens[i])])
                     for i in range(self.num_snakes)]
        self.alive_counter = int(alive_counter)
        self.episode_length = int(episode_length)
        self._zero_stats()
        frame = self._encode()
        self.frames = deque([frame] * self.frame_stack, maxlen=self.frame_stack)
        return self._stacked()


class CoopOracleSnakeEnv(OracleSnakeEnv):
    """SnakeCoop-v1: any(dones) ends the episode and turns every done True (envs/coop_snake_env.py:14-22)."""

    def step(self, actions):
        obs, rews, dones, info = super().step(actions)
        if self._done_fn(dones):
            dones = [True] * self.num_snakes
        return obs, rews, dones, info

    def _done_fn(self, dones):
        return any(dones)


def competition_rank(scores):
    """Standard competition ranking on descending score, ties share (snake_env.py:397-404)."""
    scores = np.asarray(scores, dtype=np.float64)
    return np.array([1 + int(np.sum(scores > s)) for s in scores])


class VectorOracle:
    """N independent oracle envs with the reference worker's auto-reset (wrappers.py:138-146):
    after a step whose dones are all True the returned observation is the reset one while
    reward / done / info stay those of the terminal step."""

    def __init__(self, num_envs, draws=None, **kwargs):
        self.envs = [OracleSnakeEnv(draws=(draws[i] if draws else None), **kwargs)
                     for i in range(num_envs)]
        self.num_envs = num_envs

    def reset(self):
        return np.stack([e.reset() for e in self.envs])

    def step(self, actions):
        obs, rews, dones, infos = [], [], [], []
        for e, a in zip(self.envs, actions):
            o, r, d, info = e.step(list(a))
            if all(d):
                o = e.reset()
            obs.append(o)
            rews.append(r)
            dones.append(d)
            infos.append(info)
        return np.stack(obs), np.asarray(rews, dtype=np.float64), np.asarray(dones, dtype=bool), infos


# --------------------------------------------------------------------------- Philox draw source
def philox4x32_10(counter, key):
    """Philox4x32-10 (Salmon et al., SC'11): counter 4x u32, key 2x u32 -> 4x u32."""
    M0, M1, W0, W1 = 0xD2511F53, 0xCD9E8D57, 0x9E3779B9, 0xBB67AE85
    c0, c1, c2, c3 = counter
    k0, k1 = key
    for _ in range(10):
        p0, p1 = M0 * c0, M1 * c2
        c0, c1, c2, c3 = ((p1 >> 32) ^ c1 ^ k0) & 0xFFFFFFFF, p1 & 0xFFFFFFFF, \
                         ((p0 >> 32) ^ c3 ^ k1) & 0xFFFFFFFF, p0 & 0xFFFFFFFF
        k0, k1 = (k0 + W0) & 0xFFFFFFFF, (k1 + W1) & 0xFFFFFFFF
    return c0, c1, c2, c3


class PhiloxDraws:
    """The device's counter-based stream (DESIGN.md 'RNG'): word(seed; env, event, purpose, idx) with
    counter = {env_lo, env_hi ^ 'SNK1', event, purpose << 24 | idx // 4}, bounded draw = mulhi(word, n).
    `event` is bumped by the driver once per step and per explicit reset (tick())."""
    STEP_FRUIT, SPAWN, RESET_FRUIT = 0, 1, 2

    def __init__(self, seed, env_id):
        self.key = (seed & 0xFFFFFFFF, (seed >> 32) & 0xFFFFFFFF)
        self.env_id = env_id
        self.event = 0
        self.in_reset = False

    def tick(self):
        self.event = (self.event + 1) & 0xFFFFFFFF

    def _below(self, purpose, idx, n):
        ctr = (self.env_id & 0xFFFFFFFF, ((self.env_id >> 32) & 0xFFFFFFFF) ^ 0x534E4B31, self.event,
               (purpose << 24) | (idx >> 2))
        return (philox4x32_10(ctr, self.key)[idx & 3] * n) >> 32

    def spawn(self, n_cand, ns, no_overlap):
        self.in_reset = True
        attempt = 0
        while True:
            pick = [self._below(self.SPAWN, attempt * ns + i, n_cand) for i in range(ns)]
            if no_overlap(pick):
                return pick
            attempt += 1

    def fruit(self, n_empty, k):
        purpose = self.RESET_FRUIT if self.in_reset else self.STEP_FRUIT
        self.in_reset = False
        return [self._below(purpose, j, n_empty) for j in range(k)]
