"""Egocentric frame_stack-1 observations (the ENC_REG encode: viewer pairs on 16-byte aligned blocks, one viewer at a
time otherwise) against a vectorised restatement of the oracle's SnakeEnv._encode, for every environment of the batch,
computed from get_state()."""
import numpy as np
import pytest
import torch

from marl_snake_b200 import SnakeBatch

pytestmark = pytest.mark.gpu

EMPTY, WALL, FRUIT, HEAD, BODY, TAIL = 0, 1, 2, 3, 4, 5          # oracle/snake_oracle.py
CFG5 = dict(height=20, width=20, num_snakes=4, snake_length=3, vision_range=5)
CHUNK = 1 << 17


def expected_obs(grid, head, alive, V):
    """oracle.SnakeEnv._encode for a batch: grid uint8 [n, H, W] cell codes, head int32 [n, ns] (-1: no head),
    alive [n, ns] -> uint8 [n, ns, 2V+1, 2V+1, 8]."""
    n, H, W = grid.shape
    ns = head.shape[1]
    side = 2 * V + 1
    pad = torch.zeros((n, H + 2 * V, W + 2 * V), dtype=torch.uint8, device=grid.device)     # EMPTY: all channels 0
    pad[:, V:V + H, V:V + W] = grid
    h = torch.where(alive.bool(), head.long(), torch.zeros_like(head, dtype=torch.long))      # no head: cell (0, 0)
    hr, hc = h // W, h % W
    k = torch.arange(side, device=grid.device)
    rows = (hr[..., None] + k)[:, :, :, None]                     # padded row of window row i = hr - V + i + V
    cols = (hc[..., None] + k)[:, :, None, :]
    win = pad[torch.arange(n, device=grid.device)[:, None, None, None], rows, cols].long()    # [n, ns, side, side]
    kind, owner = win % 10, win // 10
    snake = win >= HEAD
    mine = snake & (owner == torch.arange(ns, device=grid.device)[None, :, None, None])
    other = snake & ~mine
    ch = [win == WALL, win == FRUIT] + [other & (kind == p) for p in (HEAD, BODY, TAIL)] + \
         [mine & (kind == p) for p in (HEAD, BODY, TAIL)]
    return torch.stack(ch, dim=-1).to(torch.uint8)


def check_all(b, obs, what):
    st = b.get_state()
    V = b.vision_range
    for lo in range(0, b.num_envs, CHUNK):
        hi = min(lo + CHUNK, b.num_envs)
        want = expected_obs(st['grid'][lo:hi], st['head'][lo:hi], st['alive'][lo:hi], V)
        got = obs[lo:hi]
        if not torch.equal(got, want):
            bad = (got != want).flatten(1).any(1).nonzero()[:5, 0] + lo
            raise AssertionError(f'{what}: observations differ from the oracle encode, first envs {bad.tolist()}')
    assert b.device_errors() == 0, what


def run_sequence(b, steps=24, seed=5):
    """reset, steps with auto-reset, a masked reset, a set_state round trip: every env checked after each."""
    N, ns = b.num_envs, b.num_snakes
    check_all(b, b.reset(), 'reset')
    g = torch.Generator(device='cuda').manual_seed(seed)
    finished = 0
    for t in range(steps):
        a = torch.randint(0, 3, (N, ns), dtype=torch.uint8, device='cuda', generator=g)
        obs, _, _, info = b.step(a)
        finished += int(info['finished'].sum())
        if t % 6 == 5 or t == steps - 1:
            check_all(b, obs, f'step {t}')
    assert finished > 0                                           # auto-resets happened inside the checked steps
    mask = (torch.arange(N, device='cuda') % 3 == 1).to(torch.uint8)
    check_all(b, b.reset(mask), 'masked reset')
    a = torch.randint(0, 3, (N, ns), dtype=torch.uint8, device='cuda', generator=g)
    b.step(a)
    st = b.get_state(max_cells=max(2, int(b.get_state()['length'].max())))
    args = [st[k].cpu().numpy() for k in ('grid', 'alive', 'dir', 'length', 'cells', 'alive_counter', 'episode_length')]
    cells, length = args[4], args[3]
    cells[np.arange(cells.shape[-1]) >= length[..., None]] = 0
    check_all(b, b.set_state(*args), 'set_state')


def _cross_map(n=16):
    m = np.zeros((n, n), dtype=np.uint8)
    m[0, :] = m[-1, :] = m[:, 0] = m[:, -1] = 1
    m[n // 2, 3:n - 3] = 1
    m[3:n - 3, n // 2] = 1
    return m


def test_cfg5_full_every_env_matches_the_oracle_encode():
    b = SnakeBatch(1 << 20, seed=3, **CFG5)
    assert b._obs.data_ptr() % 16 == 0                            # the viewer-pair path
    run_sequence(b)
    b.close()


def test_8_byte_aligned_buffer_matches_the_oracle_encode():
    N = 1 << 17
    b = SnakeBatch(N, seed=4, **CFG5)
    n = b._obs.numel()
    raw = torch.empty(n + 32, dtype=torch.uint8, device=b.device)
    off = 8 if raw.data_ptr() % 16 == 0 else 16 - raw.data_ptr() % 16 + 8
    b._obs = raw[off:off + n].view(b._obs.shape)
    assert b._obs.data_ptr() % 16 == 8                            # one viewer at a time
    run_sequence(b)
    b.close()


@pytest.mark.parametrize('num_snakes', [2, 3])
def test_two_and_three_snakes_match_the_oracle_encode(num_snakes):
    b = SnakeBatch(1 << 17, seed=6, **dict(CFG5, num_snakes=num_snakes))
    run_sequence(b)
    b.close()


def test_wall_map_matches_the_oracle_encode():
    b = SnakeBatch(50000, seed=7, wall_map=_cross_map(), num_snakes=4, vision_range=4, done_mode='any')
    run_sequence(b)
    b.close()


def test_step_many_every_step_equals_single_steps():
    N, T = 1 << 16, 6
    many = SnakeBatch(N, seed=8, **CFG5)
    single = SnakeBatch(N, seed=8, **CFG5)
    assert torch.equal(many.reset(), single.reset())
    g = torch.Generator(device='cuda').manual_seed(9)
    acts = torch.randint(0, 3, (T, N, 4), dtype=torch.uint8, device='cuda', generator=g)
    obs = torch.empty((T, N) + many.obs_shape, dtype=torch.uint8, device='cuda')
    assert obs.data_ptr() % 16 == 0
    _, rew, done, _ = many.step_many(acts, obs=obs)
    for t in range(T):
        o, r, d, _ = single.step(acts[t])
        assert torch.equal(obs[t], o) and torch.equal(rew[t], r) and torch.equal(done[t].bool(), d), f'step {t}'
    check_all(single, obs[T - 1], 'step_many last step')
    many.close()
    single.close()
