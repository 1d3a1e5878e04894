"""CPU-side checks of the C-ABI library: it loads without a GPU, exports every symbol include/snk.h
declares, validates configurations before touching CUDA, and its host-side spawn table equals the
reference's dfs_sweep_empty enumeration (golden tables)."""
import ctypes as C
import os
import re
import shutil
import subprocess

import numpy as np
import pytest

from golden_util import load_spawn_tables

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
    import marl_snake_b200 as m
    header = open(os.path.join(ROOT, 'include', 'snk.h')).read()
    header = re.sub(r'/\*.*?\*/', '', header, flags=re.S)
    declared = set(re.findall(r'\b(snk_[a-z_0-9]+)\s*\(', header))
    assert len(declared) >= 20
    for name in declared:
        assert hasattr(m.lib, name), f'{name} declared in snk.h but not exported by libsnk.so'
    from marl_snake_b200._lib import PROTOTYPES
    assert declared == set(PROTOTYPES), declared ^ set(PROTOTYPES)
    assert m.lib.snk_abi_version() == 1


def test_config_struct_matches_header_layout():
    from marl_snake_b200._lib import SnkConfig
    # 14 int32, 2 uint64, 6 double, naturally aligned
    assert C.sizeof(SnkConfig) == 14 * 4 + 2 * 8 + 6 * 8
    assert SnkConfig.seed.offset == 56 and SnkConfig.max_episode_steps.offset == 72


def test_invalid_configs_are_rejected_without_cuda():
    from hostsim_util import make_config
    import marl_snake_b200 as m
    h = C.c_void_p()
    for bad in (dict(num_snakes=26), dict(snake_length=1), dict(snake_length=26), dict(height=3),
                dict(frame_stack=0), dict(num_fruits=33), dict(height=300, width=300)):
        cfg = make_config(4, dict(bad))
        assert m.lib.snk_create(C.byref(cfg), C.byref(h)) == -1, bad
        assert len(m.lib.snk_last_error()) > 0
    cfg = make_config(4, {})
    cfg.abi_version = 99
    assert m.lib.snk_create(C.byref(cfg), C.byref(h)) == -1


def test_spawn_table_matches_reference_enumeration():
    import marl_snake_b200 as m
    tables, _ = load_spawn_tables()
    for (H, W, k), ref in tables.items():
        n = m.lib.snk_spawn_count(H, W, k)
        assert n == len(ref), (H, W, k)
        out = np.zeros((n, k), dtype=np.int32)
        assert m.lib.snk_spawn_cells(H, W, k, out.ctypes.data_as(C.c_void_p), n) == 0
        want = ref[..., 0].astype(np.int32) * W + ref[..., 1]
        assert np.array_equal(out, want), (H, W, k)
    assert m.lib.snk_spawn_count(64, 64, 5) == 362344          # SURVEY probe for the cfg4 shape
    # the pose count explodes with the length; the enumeration gives up instead of running for hours
    assert m.lib.snk_spawn_count(40, 40, 25) == -1 and b'spawn poses' in m.lib.snk_last_error()
    from hostsim_util import make_config
    h = C.c_void_p()
    assert m.lib.snk_create(C.byref(make_config(4, dict(height=40, width=40, snake_length=25))), C.byref(h)) == -1


@pytest.mark.parametrize('n,threads,misalign', [(0, 1, 0), (1, 1, 0), (7, 1, 0), (121 * 4, 1, 0), (100003, 1, 0),
                                                 (100003, 4, 0), (1 << 20, 8, 0), (4099, 3, 8), (4099, 1, 3)])
@pytest.mark.parametrize('scalar', [False, True])
def test_widen_bits_host_is_little_endian_unpackbits(monkeypatch, n, threads, misalign, scalar):
    """Host half of the packed transport: byte u, bit c -> obs byte 8*u + c (channel order of
    snake_env.py:484-492).  Any size, any thread count, any output alignment, AVX-512 or the scalar table."""
    import marl_snake_b200 as m
    if scalar:
        monkeypatch.setenv('SNK_NO_AVX512', '1')
    rng = np.random.RandomState(n + threads)
    bits = rng.randint(0, 256, size=n).astype(np.uint8)
    buf = np.full(8 * n + 64 + misalign, 0xAB, dtype=np.uint8)
    out = buf[misalign:misalign + 8 * n]
    assert m.lib.snk_widen_bits_host(bits.ctypes.data_as(C.c_void_p), out.ctypes.data_as(C.c_void_p), n, threads) == 0
    assert np.array_equal(out, np.unpackbits(bits, bitorder='little'))
    assert (buf[:misalign] == 0xAB).all() and (buf[misalign + 8 * n:] == 0xAB).all()      # nothing written outside


def test_no_cpu_fallback():
    import torch
    import marl_snake_b200 as m
    if torch.cuda.is_available():
        pytest.skip('GPU present')
    with pytest.raises(RuntimeError):
        m.SnakeBatch(4)
    with pytest.raises(KeyError):
        m.SnakeBatch(4, reward_dict={'fruit': 1.0})


def test_product_never_imports_the_oracle():
    pkg = os.path.join(ROOT, 'marl-snake_b200')
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith(('.py', '.cu', '.cuh', '.cpp', '.h')):
                text = open(os.path.join(dirpath, f)).read()
                assert 'import oracle' not in text and 'from oracle' not in text and 'hostsim' not in text.replace(
                    'tests/hostsim', ''), f


def test_reference_import_paths_resolve():
    """`from marlenv.marlenv.wrappers import make_snake, RenderGUI` (test_env.py:1) and `import marlenv`."""
    import sys
    saved = {k: v for k, v in sys.modules.items() if k == 'marlenv' or k.startswith('marlenv.')}
    for k in saved:
        del sys.modules[k]
    try:
        from marlenv.marlenv.wrappers import make_snake, RenderGUI
        import marlenv
        import marl_snake_b200 as m
        assert make_snake is m.make_snake and RenderGUI is m.RenderGUI
        assert marlenv.envs.SnakeEnv is m.SnakeEnv and marlenv.wrappers.make_snake is m.make_snake
    finally:
        for k in [k for k in sys.modules if k == 'marlenv' or k.startswith('marlenv.')]:
            del sys.modules[k]
        sys.modules.update(saved)


def _tile_kernels():
    """(registers, stack bytes) of every snk_tile_kernel instance of the in-tree library, keyed by its template
    arguments (ns, W, oh, ow, fs, coop, enc, variant; 0 for a generic dimension).  cuobjdump reads them; no GPU needed."""
    if not shutil.which('cuobjdump'):
        pytest.skip('cuobjdump not on PATH')
    import marl_snake_b200 as m
    out = subprocess.run(['cuobjdump', '-res-usage', m.LIB_PATH], capture_output=True, text=True, timeout=300).stdout
    found = re.findall(r'Function \S*snk_tile_kernelILi(\d+)ELi(\d+)ELi(\d+)ELi(\d+)ELi(\d+)ELb(\d)ELi(\d+)ELi(\d+)EE\S*:'
                       r'\s*\n\s*REG:(\d+) STACK:(\d+)', out)
    tiles = {tuple(int(a) for a in f[:8]): (int(f[8]), int(f[9])) for f in found}
    assert len(tiles) == len(found)
    return tiles


def test_hot_kernel_instances_keep_their_register_budget():
    """The occupancy of the benchmarked kernel instances is part of the measured numbers: the rare-event functions
    (fruit placement, reset) are out of line, and what they keep live raises the register count of EVERY instance
    (a four-words-per-load fruit scan once took cfg2 from 48 to 62 and cfg5 from 88 to 102 registers -- 0.756 -> 0.836 ms)."""
    tiles = _tile_kernels()
    budget = {                                    # (registers, stack bytes) ceilings
        'cfg5 warp-private, capped': (tiles[4, 20, 11, 11, 1, 0, 1, 0], (64, 16)),
        'cfg5 warp-private, uncapped (the bench line)': (tiles[4, 20, 11, 11, 1, 0, 1, 3], (88, 0)),
        'cfg2 cooperative': (tiles[4, 20, 20, 20, 1, 1, 2, 0], (48, 16)),
        'cfg3 cooperative': (tiles[4, 20, 11, 11, 4, 1, 0, 0], (64, 0)),
        'cfg4 cooperative': (tiles[16, 64, 15, 15, 1, 1, 3, 0], (64, 0)),
    }
    for what, ((reg, stack), (max_reg, max_stack)) in budget.items():
        assert reg <= max_reg and stack <= max_stack, (what, reg, stack)


def test_grid_instances_keep_the_register_budget():
    """The cfg5 step with the global state runs its own instance (variant 8): still the viewer-pair encode within 64
    registers and a small stack.  Every instance a default launch selects is there with its budget, and no specialised
    instance that only a forced tile mode or encode could reach: those calls run the generic instance of their flavour."""
    tiles = _tile_kernels()
    reg, stack = tiles[4, 20, 11, 11, 1, 0, 1, 8]
    assert reg <= 64 and stack <= 16, (reg, stack)
    assert tiles[4, 20, 11, 11, 1, 0, 1, 0] == (64, 8)
    assert tiles[4, 20, 11, 11, 1, 0, 1, 3] == (88, 0)
    for var in (0, 1, 2, 4, 5, 6, 8, 10, 12, 14):
        assert (4, 20, 11, 11, 1, 1, 1, var) in tiles            # the cooperative ones
    assert not [k for k in tiles if k[:5] == (4, 20, 11, 11, 1) and k[6] == 0], 'cfg5 ENC_LEGACY'
    assert not [k for k in tiles if k[:5] == (16, 64, 15, 15, 1) and k[6] == 0], 'cfg4 ENC_LEGACY'
    assert not [k for k in tiles if k[:5] == (4, 20, 11, 11, 4) and k[5] == 0], 'cfg3 warp-private'
    assert not [k for k in tiles if k[:5] == (4, 20, 11, 11, 4) and k[7] in (2, 6)], 'cfg3 several steps per launch'
    per_var = {}
    for k in tiles:
        per_var[k[7]] = per_var.get(k[7], 0) + 1
    # generic REG, DIRECT and LEGACY in both tile modes and PAD cooperative (7), cfg5 REG and cfg2 DIRECT in both (4),
    # cfg3 LEGACY and cfg4 PAD cooperative (2, cfg3 without variants 2 and 6); variant 3 exists warp-private only
    assert per_var == {0: 13, 1: 13, 2: 12, 3: 5, 4: 13, 5: 13, 6: 12, 8: 13, 10: 13, 12: 13, 14: 13}, per_var
