#!/usr/bin/env python
"""Does the cfg5 observation block write faster into compressible device memory?  (DESIGN.md section 4)

    python tools/obs_compression_probe.py [--out DIR] [--trials 5]

One run answers, on cuda:0:
  1. device support: CU_DEVICE_ATTRIBUTE_GENERIC_COMPRESSION_SUPPORTED, and the compressionType that
     cuMemGetAllocationPropertiesFromHandle reads back for a CU_MEM_ALLOCATION_COMP_GENERIC allocation;
  2. bare write rate: a 4.06 GB block (1,048,576 cfg5 observations) written into a plain cudaMalloc buffer and into a
     compressible one (snk_alloc_obs), alternating, with three contents -- a real cfg5 observation block captured
     after a burn-in and tiled, all zeros, random 0/1 bytes -- each with st.global.cs and plain stores;
  3. the real step: SnakeBatch.step at cfg5 (1,048,576 envs) with its observation buffer plain and compressible,
     alternating in one process, and the two buffers' outputs compared byte for byte from the same seed.  (Since the
     step picks the 64-register instance for a compressible block, this now times both changes together.)
Prints and writes DIR/obs_compression_probe.json and .txt; records the card and its power limit.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

ENV_KW = dict(height=20, width=20, num_snakes=4, snake_length=3, vision_range=5, frame_stack=1)   # bench.py cfg5
N = 1 << 20
PATTERN_ENVS = 2048                      # 2048 x 3872 B = 7.9 MB of real observations, tiled 512 times


def build_probe(tmp):
    so = os.path.join(tmp, 'obs_compression_probe.so')
    subprocess.check_call(['nvcc', '-O3', '-gencode', 'arch=compute_100a,code=sm_100a', '-shared', '-Xcompiler',
                           '-fPIC', '-o', so, os.path.join(ROOT, 'tools', 'obs_compression_probe.cu'), '-lcuda'])
    p = C.CDLL(so)
    p.probe_tile_write.restype = C.c_float
    p.probe_tile_write.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_int, C.c_int, C.c_int]
    p.probe_compression_props.restype = None
    p.probe_compression_props.argtypes = [C.c_int, C.c_size_t, C.POINTER(C.c_longlong * 4)]
    return p


class _DeviceBlock:
    """A uint8 device block from snk_alloc_obs, as a torch tensor (torch keeps this owner alive)."""

    def __init__(self, lib, nbytes):
        self.lib, self.ptr, comp = lib, C.c_void_p(), C.c_int(0)
        rc = lib.snk_alloc_obs(0, nbytes, C.byref(self.ptr), C.byref(comp))
        if rc:
            raise RuntimeError(lib.snk_last_error().decode())
        self.compressed = bool(comp.value)
        self.__cuda_array_interface__ = dict(shape=(nbytes,), typestr='|u1', data=(self.ptr.value, False), version=2)

    def __del__(self):
        self.lib.snk_free_obs(self.ptr)


def card():
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm,clocks.max.mem,driver_version',
                        '--format=csv,noheader', '-i', '0'], capture_output=True, text=True)
    return q.stdout.strip()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', default='.', help='directory for obs_compression_probe.json / .txt')
    ap.add_argument('--trials', type=int, default=5)
    ap.add_argument('--reps', type=int, default=10, help='tile writes per timed trial')
    ap.add_argument('--steps', type=int, default=200, help='steps per timed trial of the real step')
    args = ap.parse_args()
    import numpy as np
    import torch
    from marl_snake_b200 import SnakeBatch, lib

    os.makedirs(args.out, exist_ok=True)
    lines, res = [], {'card': card()}

    def say(s):
        print(s, flush=True)
        lines.append(s)

    say(f'card (name, power limit, max SM / mem clocks, driver): {res["card"]}')
    tmp = tempfile.mkdtemp(prefix='obs_comp_probe_')
    probe = build_probe(tmp)
    torch.cuda.set_device(0)

    # ---- 1. device support ---------------------------------------------------------------------------------------
    obs_env = 4 * 11 * 11 * 8
    total = N * obs_env
    props = (C.c_longlong * 4)()
    probe.probe_compression_props(0, total, C.byref(props))
    res['props'] = dict(generic_compression_supported=int(props[0]), granularity=int(props[1]),
                        granted_compression_type=int(props[2]), first_error=int(props[3]))
    say(f'1. device attribute GENERIC_COMPRESSION_SUPPORTED = {props[0]}, granularity with COMP_GENERIC = '
        f'{props[1]} B, compressionType read back = {props[2]} (1 = CU_MEM_ALLOCATION_COMP_GENERIC), '
        f'first CUresult error = {props[3]}')

    # ---- capture a real cfg5 observation block ---------------------------------------------------------------------
    gen = torch.Generator(device='cuda').manual_seed(1234)
    pool = list(torch.randint(0, 3, (509, N, 4), dtype=torch.uint8, device='cuda', generator=gen).unbind(0))
    batch = SnakeBatch(N, device=0, seed=0, rng='philox', auto_reset=True, **ENV_KW)
    batch.reset()
    for t in range(256):
        batch.step(pool[t % 509], want_info=False)
    torch.cuda.synchronize()
    real = batch._obs.reshape(-1)[:PATTERN_ENVS * obs_env].clone()
    nz = real.view(-1, 8).sum(1)
    say(f'real pattern: {PATTERN_ENVS} envs x {obs_env} B after a 256-step burn-in; nonzero bytes '
        f'{int((real != 0).sum()) / real.numel():.4f}, 8-byte groups with a one {float((nz > 0).float().mean()):.4f}, '
        f'max ones per group {int(nz.max())}')
    patterns = {'real_obs': real,
                'zeros': torch.zeros_like(real),
                'random01': torch.randint(0, 2, real.shape, dtype=torch.uint8, device='cuda', generator=gen)}
    ntiles = N // PATTERN_ENVS

    # ---- 2. bare write rate ------------------------------------------------------------------------------------------
    plain = torch.empty(total, dtype=torch.uint8, device='cuda')
    comp_owner = _DeviceBlock(lib, total)
    comp = torch.as_tensor(comp_owner, device='cuda')
    say(f'2. compressible block: snk_alloc_obs granted compression = {comp_owner.compressed}; '
        f'{total / 1e9:.3f} GB per write, {args.reps} writes per trial, {args.trials} trials per buffer, alternating')
    res['alloc_compressed'] = comp_owner.compressed
    res['bare'] = {}
    for pname, pat in patterns.items():
        for cs in (1, 0):
            for buf in (plain, comp):                                  # warm up both
                probe.probe_tile_write(buf.data_ptr(), pat.data_ptr(), pat.numel(), ntiles, cs, 2)
            ms = {'plain': [], 'compressible': []}
            for _ in range(args.trials):
                for bname, buf in (('plain', plain), ('compressible', comp)):
                    t = probe.probe_tile_write(buf.data_ptr(), pat.data_ptr(), pat.numel(), ntiles, cs, args.reps)
                    ms[bname].append(t / args.reps)
            assert torch.equal(plain[:real.numel()], comp[:real.numel()]) and torch.equal(plain[-1024:], comp[-1024:])
            key = f'{pname}/{"st.global.cs" if cs else "st.global"}'
            res['bare'][key] = ms
            say(f'   {key:24s} plain {min(ms["plain"]):.4f}-{max(ms["plain"]):.4f} ms '
                f'({total / min(ms["plain"]) / 1e6:.0f} GB/s)   compressible {min(ms["compressible"]):.4f}-'
                f'{max(ms["compressible"]):.4f} ms ({total / min(ms["compressible"]) / 1e6:.0f} GB/s)')

    # ---- 3. the real step -----------------------------------------------------------------------------------------
    # outputs: two batches from the same seed, one writing the plain buffer, one the compressible buffer
    a = SnakeBatch(N, device=0, seed=7, rng='philox', auto_reset=True, **ENV_KW)
    b = SnakeBatch(N, device=0, seed=7, rng='philox', auto_reset=True, **ENV_KW)
    a._obs = torch.empty_like(a._obs)                                  # SnakeBatch's own buffer may be compressible
    b._obs = comp.view(a._obs.shape)
    same = torch.equal(a.reset(), b.reset())
    for t in range(64):
        oa, ra, da, _ = a.step(pool[t], want_info=False)
        ob, rb, db, _ = b.step(pool[t], want_info=False)
        same = same and torch.equal(oa, ob) and torch.equal(ra, rb) and torch.equal(da, db)
    a.close(); b.close()
    del a, b
    res['step_outputs_equal'] = bool(same)
    say(f'3. step outputs byte-equal, plain vs compressible buffer, reset + 64 steps at {N} envs: {same}')
    bufs = {'plain': torch.empty_like(batch._obs), 'compressible': comp.view(batch._obs.shape)}
    step_no = 256
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ms = {'plain': [], 'compressible': []}
    for trial in range(args.trials + 1):
        for bname in ('plain', 'compressible'):
            batch._obs = bufs[bname]
            for _ in range(20):
                batch.step(pool[step_no % 509], want_info=False)
                step_no += 1
            ev0.record()
            for _ in range(args.steps):
                batch.step(pool[step_no % 509], want_info=False)
                step_no += 1
            ev1.record()
            torch.cuda.synchronize()
            if trial:                                                  # trial 0 warms both up
                ms[bname].append(ev0.elapsed_time(ev1) / args.steps)
    res['step_ms'] = ms
    res['device_errors'] = batch.device_errors()
    for bname, v in ms.items():
        say(f'   step, obs {bname:12s}: {min(v):.4f}-{max(v):.4f} ms per step (median {float(np.median(v)):.4f}) '
            f'over {args.trials} x {args.steps} steps')
    say(f'   device errors: {res["device_errors"]}; card after: {card()}')
    with open(os.path.join(args.out, 'obs_compression_probe.json'), 'w') as f:
        json.dump(res, f, indent=1)
    with open(os.path.join(args.out, 'obs_compression_probe.txt'), 'w') as f:
        f.write('\n'.join(lines) + '\n')


if __name__ == '__main__':
    main()
