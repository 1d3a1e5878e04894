"""CPU-side checks of the wall-map pool (snk_create_maps): the new calls are exported through the C ABI, and bad pools
are refused with a message naming the map at fault before any CUDA call."""
import ctypes as C

import numpy as np

from golden_util import load_map_spawn_tables
from hostsim_util import make_config


def box(h, w):
    b = np.ones((h, w), dtype=np.uint8)
    b[1:-1, 1:-1] = 0
    return b


def create_maps(maps, num_envs=4, ids=None, **kw):
    import marl_snake_b200 as m
    maps = np.ascontiguousarray(maps, dtype=np.uint8)
    cfg = make_config(num_envs, dict(kw, height=maps.shape[1], width=maps.shape[2]), rng_mode=0)
    h = C.c_void_p()
    ids_p = None if ids is None else np.ascontiguousarray(ids, dtype=np.uint8).ctypes.data_as(C.c_void_p)
    rc = m.lib.snk_create_maps(C.byref(cfg), len(maps), maps.ctypes.data_as(C.c_void_p), ids_p, C.byref(h))
    msg = m.lib.snk_last_error().decode() if rc else ''    # a successful call leaves the last failure's message
    if rc == 0:
        m.lib.snk_destroy(h)
    return rc, msg


def test_pool_calls_are_exported():
    import marl_snake_b200 as m
    from marl_snake_b200._lib import DEV_ERRORS, PROTOTYPES
    for name in ('snk_create_maps', 'snk_map_ids_dev', 'snk_num_maps'):
        assert name in PROTOTYPES and hasattr(m.lib, name)
    assert 128 in DEV_ERRORS
    assert m.lib.snk_num_maps(None) == 0
    p, q = C.c_void_p(), C.c_void_p()
    assert m.lib.snk_map_ids_dev(None, C.byref(p), C.byref(q)) == -1


def test_bad_pools_are_rejected_naming_the_map():
    import marl_snake_b200 as m
    b = box(12, 12)
    open_border = b.copy()
    open_border[0, 5] = 0
    rc, msg = create_maps(np.stack([b, b, open_border]))
    assert rc == -1 and 'wall map 2' in msg and 'border cell (0, 5)' in msg
    # a map with room for fewer spawn poses than snakes
    full = np.ones((12, 12), dtype=np.uint8)
    full[5, 3:6] = 0
    rc, msg = create_maps(np.stack([b, full]))
    assert rc == -1 and 'wall map 1' in msg and 'spawn poses' in msg
    rc, msg = create_maps(np.stack([b, b]), ids=[0, 1, 2, 0])
    assert rc == -1 and 'map_ids[2]' in msg
    cfg = make_config(4, dict(height=12, width=12), rng_mode=0)
    h = C.c_void_p()
    walls = np.ascontiguousarray(np.stack([b] * 2))
    for n in (0, 257):
        assert m.lib.snk_create_maps(C.byref(cfg), n, walls.ctypes.data_as(C.c_void_p), None, C.byref(h)) == -1
        assert 'num_maps' in m.lib.snk_last_error().decode()
    assert m.lib.snk_create_maps(C.byref(cfg), 2, None, None, C.byref(h)) == -1


def test_asset_map_pool_passes_the_host_checks():
    # every asset map is a valid pool member: the checks above reject none of them (creation then needs a device)
    for name, (walls, k, cands) in load_map_spawn_tables().items():
        pool = np.stack([walls, box(*walls.shape)])
        rc, msg = create_maps(pool, snake_length=k)
        assert 'wall map' not in msg and 'map_ids' not in msg, (name, msg)
