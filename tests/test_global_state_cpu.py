"""CPU-side checks of the global-state calls (snk_reset_grid / snk_step_grid / snk_step_many_grid): they are exported
through the C ABI, refuse a null handle, and SnakeBatch.step_many checks the shape of a caller's global_state tensor
before it calls the library."""
import ctypes as C

import pytest
import torch

GRID_CALLS = ('snk_reset_grid', 'snk_step_grid', 'snk_step_many_grid')


def test_grid_calls_are_exported():
    import marl_snake_b200 as m
    from marl_snake_b200._lib import PROTOTYPES
    for name in GRID_CALLS:
        assert name in PROTOTYPES and hasattr(m.lib, name), name


def test_grid_calls_refuse_a_null_handle():
    import marl_snake_b200 as m
    buf = (C.c_uint8 * 64)()
    p = C.cast(buf, C.c_void_p)
    assert m.lib.snk_reset_grid(None, None, None, None, p, None) == -1
    assert 'null handle' in m.lib.snk_last_error().decode()
    assert m.lib.snk_step_grid(None, p, None, None, p, p, p, None, None) == -1
    assert 'null handle' in m.lib.snk_last_error().decode()
    assert m.lib.snk_step_many_grid(None, 2, p, None, None, p, 1, p, p, None, None) == -1
    assert 'null handle' in m.lib.snk_last_error().decode()


def fake_batch(N=6, ns=2, H=9, W=10, fs=1):
    """A SnakeBatch shell on the CPU with just what step_many's argument checks read (they run before any library
    call, so no handle is needed)."""
    from marl_snake_b200 import SnakeBatch
    b = object.__new__(SnakeBatch)
    b.num_envs, b.num_snakes, b.device = N, ns, torch.device('cpu')
    b.grid_shape = (H, W)
    b.obs_shape = (ns, 5, 5, 8 * fs)
    b.bits_shape = (ns, 5, 5, fs)
    b.global_state = None
    b._h = C.c_void_p()
    return b


@pytest.mark.parametrize('shape,msg', [
    ((3, 6, 9, 9), 'global_state must have shape'),           # wrong grid
    ((6, 90), 'global_state must have shape'),                # flat rows are not accepted
    ((2, 6, 9, 10), 'global_state must have shape'),          # T = 2 against 3 steps of actions
    ((1, 6, 9, 10), 'global_state must have shape'),          # [1, N, H, W] only for T == 1
])
def test_step_many_global_state_shapes_are_checked(shape, msg):
    b = fake_batch()
    acts = torch.zeros((3, 6, 2), dtype=torch.uint8)
    with pytest.raises(ValueError, match=msg):
        b.step_many(acts, global_state=torch.zeros(shape, dtype=torch.uint8))


def test_step_many_global_state_dtype_and_layout_are_checked():
    b = fake_batch()
    acts = torch.zeros((3, 6, 2), dtype=torch.uint8)
    with pytest.raises(ValueError, match='contiguous uint8'):
        b.step_many(acts, global_state=torch.zeros((6, 9, 10), dtype=torch.int32))
    with pytest.raises(ValueError, match='contiguous uint8'):
        b.step_many(acts, global_state=torch.zeros((6, 10, 9), dtype=torch.uint8).transpose(1, 2))


def test_step_many_outputs_must_agree_on_every_step():
    b = fake_batch()
    acts = torch.zeros((3, 6, 2), dtype=torch.uint8)
    every_obs = torch.zeros((3, 6) + b.obs_shape, dtype=torch.uint8)
    with pytest.raises(ValueError, match='all hold every step or all hold the last step only'):
        b.step_many(acts, obs=every_obs, global_state=torch.zeros((6, 9, 10), dtype=torch.uint8))
