#!/usr/bin/env python
"""bench.py -- agent-steps/s of the Snake-v1 step path on N B200s (one process per GPU).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

A "step" is one pass of the hot path over the whole batch: ONE launch of snk_tile_kernel stepping every
environment of the shard (rules + auto-reset + observation render).  Workload (config.workload): BASELINE
cfg5 shape -- 20x20 grid, 4 snakes, length 3, vision_range 5, frame_stack 1, auto-reset, Philox seed 0,
uniform random actions -- with 1,048,576 environments per GPU (weak scaling; no collective on the step
path, one NCCL all-reduce of the 8-double statistics vector after the timed region).

Prints ONE JSON line (rank 0): value = device-timed whole-job throughput with state and actions
resident in HBM; e2e = the same metric through the C ABI's host-buffer call (snk_step_host: pinned
actions H2D, step, obs + rewards + dones D2H, synchronise); roofline = the kernel against measured HBM
peak; cpu_baseline = the unmodified reference SnakeEnv (oracle/_ref; the oracle port when that install is
missing) on this box's host cores, run as the reference vectorises (one process per env).

--dump-outputs DIR writes, after the timed region, what the last timed step returned to its caller for a fixed
sample of DUMP_ENVS environments (seeded choice, sorted): obs.npy float32 [n, ns, oh, ow, 8], rewards.npy float64
[n, ns], dones.npy float32 [n, ns].  The batch, the actions and the number of steps before the timed region are
fixed by the arguments, so two builds run with the same arguments can be compared output for output.
"""
import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

ENV_KW = dict(height=20, width=20, num_snakes=4, snake_length=3, vision_range=5, frame_stack=1)
WORKLOAD = 'cfg5: 20x20, 4 snakes, len 3, vision_range 5, frame_stack 1, auto-reset, random actions'
BURN_IN = 256          # steps before warm-up so the alive / reset mix is stationary (mean episode ~68)
CLOCK_RAMP_S = 1.0     # untimed stepping after the CPU legs so the GPU is back at its load clocks
DUMP_ENVS, DUMP_SEED = 2048, 0     # --dump-outputs sample: 2048 x 3872 float32 observations = 32 MB


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=2000, help='timed steps')
    ap.add_argument('--warmup', type=int, default=100)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--envs-per-gpu', type=int, default=1 << 20)
    ap.add_argument('--envs-total', type=int, default=0,
                    help='strong scaling: this many environments in total, sharded over the ranks '
                         '(BASELINE cfg5 read literally: 1048576); default 0 = weak scaling, --envs-per-gpu each')
    ap.add_argument('--e2e-steps', type=int, default=8)
    ap.add_argument('--cpu-seconds', type=float, default=12.0)
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-configs', action='store_true', help='skip the per-config block (cfg1-cfg4, strong scaling)')
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help='write the last timed step\'s obs / rewards / dones of a fixed sample of environments '
                         'as DIR/<name>.npy (rank 0)')
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error('--steps must be at least 1 and --warmup at least 0')
    if args.dump_outputs and args.impl != 'ours':
        ap.error('--dump-outputs needs --impl ours')
    return args


def dump_outputs(out_dir, obs, rew, done):
    """The caller-visible outputs of one step (obs uint8, rewards float64, dones bool, all [N, ns, ...] on the
    device) for a seeded sample of environments, as .npy files in float32 / float64."""
    import numpy as np
    import torch
    N = obs.shape[0]
    idx = np.sort(np.random.RandomState(DUMP_SEED).choice(N, size=min(N, DUMP_ENVS), replace=False))
    sel = torch.as_tensor(idx, device=obs.device)
    os.makedirs(out_dir, exist_ok=True)
    for name, x, dtype in (('obs', obs, np.float32), ('rewards', rew, np.float64), ('dones', done, np.float32)):
        np.save(os.path.join(out_dir, name + '.npy'), x.index_select(0, sel).cpu().numpy().astype(dtype))


# ------------------------------------------------------------------------------ CPU legs
def cpu_leg(seconds, kind, chunk=None):
    """The reference's CPU step path on all host cores for about `seconds`: kind 'reference' = the UNMODIFIED
    reference SnakeEnv installed in oracle/_ref (make -C oracle ref), kind 'port' = the oracle restatement.
    Returns a cpu_baseline dict."""
    from oracle.cpu_runner import CpuPool
    chunk = chunk or (40 if kind == 'reference' else 250)
    pool = CpuPool(ENV_KW, kind=kind)
    pool.run(chunk)
    total, wall = 0, 0.0
    while wall < seconds:
        wall += pool.run(chunk)
        total += chunk
    pool.close()
    ns = ENV_KW['num_snakes']
    what = ('unmodified reference SnakeEnv (oracle/_ref, gym stubbed)' if kind == 'reference'
            else 'oracle port (oracle/snake_oracle.py)')
    return {'value': total * pool.procs * ns / wall, 'unit': 'agent-steps/s', 'cores': pool.procs, 'kind': kind,
            'sample': f'{what}: {pool.procs} processes x 1 env (reference vectorisation, wrappers.py:211-212), '
                      f'{total} env-steps each incl. resets, {wall:.1f} s wall, Python {sys.version.split()[0]}'}


def reference_kind():
    from oracle.cpu_runner import reference_available
    return 'reference' if reference_available() else 'port'


def cpu_native_leg(seconds=4.0):
    """Extra context, single thread: the device rule source compiled for the host (tests/hostsim, test
    infrastructure).  Runs in a SUBPROCESS so that no test code is loaded into the measuring process."""
    import subprocess
    try:
        out = subprocess.run([sys.executable, os.path.join(ROOT, 'tools', 'cpu_native_leg.py'), str(seconds)],
                             capture_output=True, text=True, timeout=120)
        return json.loads(out.stdout.strip().splitlines()[-1])
    except Exception as exc:      # noqa: BLE001
        return {'unavailable': repr(exc)}


def reference_arm(args):
    """--impl reference: the reference's own CPU implementation of the path on all host cores -- the unmodified
    reference from oracle/_ref when it was installed (kind "reference"), else the oracle port (kind "port").
    One 'step' = every worker process advances its env by `chunk` env-steps (auto-reset included)."""
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    from oracle.cpu_runner import CpuPool
    kind = reference_kind()
    chunk = 40 if kind == 'reference' else 250
    pool = CpuPool(ENV_KW, kind=kind)
    for _ in range(max(args.warmup, 1)):
        pool.run(chunk)
    t = 0.0
    for _ in range(args.steps):
        t += pool.run(chunk)
    pool.close()
    ns = ENV_KW['num_snakes']
    val = args.steps * chunk * pool.procs * ns / t
    sample = (f'{"unmodified reference SnakeEnv from oracle/_ref" if kind == "reference" else "oracle port"}: '
              f'{pool.procs} processes x 1 env, {chunk} env-steps per bench step incl. resets')
    out = {
        'impl': 'reference', 'metric': 'agent_steps_per_sec', 'value': val, 'unit': 'agent-steps/s',
        'n_gpus': args.gpus, 'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': 1e3 * t / args.steps,
        'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'u8', 'data': 'synthetic',
        # the arm's config: the same workload; each bench step is a bounded SAMPLE of it (one env per host core)
        'config': {'workload': WORKLOAD, 'envs_per_gpu': args.envs_per_gpu, 'global_envs': args.envs_per_gpu * args.gpus,
                   'parallelism': f'env-shard x{args.gpus}',
                   'sample_envs': pool.procs, 'env_steps_per_bench_step': chunk},
        'cpu_baseline': {'value': val, 'unit': 'agent-steps/s', 'cores': pool.procs, 'kind': kind, 'sample': sample},
        'e2e': {'value': val, 'unit': 'agent-steps/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
        'gpu_launches': 0}
    if kind == 'reference':           # the port beside it: how much faster the restatement is than the reference
        out['cpu_port'] = cpu_leg(4.0, 'port')
    print(json.dumps(out), file=RESULT_OUT, flush=True)


# ------------------------------------------------------------------------------ clocks
class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons of one GPU through NVML while the timed region runs."""
    BAD = {'hw_slowdown': 0x8, 'hw_thermal_slowdown': 0x40, 'sw_thermal_slowdown': 0x20,
           'hw_power_brake_slowdown': 0x80}
    NOTE = {'sw_power_cap': 0x4}

    def __init__(self, index, period=0.002):
        super().__init__(daemon=True)
        self.index, self.period = index, period
        self.samples, self.reasons = [], 0
        self.stop_flag = threading.Event()
        self.ok = False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception:
            self.max_mhz = None

    def run(self):
        if not self.ok:
            return
        while not self.stop_flag.is_set():
            try:
                self.samples.append(self.nv.nvmlDeviceGetClockInfo(self.h, self.nv.NVML_CLOCK_SM))
                self.reasons |= int(self.nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h))
            except Exception:
                pass
            time.sleep(self.period)

    def summary(self):
        if not self.samples:
            return {'sm_mhz': None, 'sm_max_mhz': self.max_mhz, 'reasons': ['unsampled']}
        s = sorted(self.samples)
        names = [n for n, b in {**self.BAD, **self.NOTE}.items() if self.reasons & b]
        return {'sm_mhz': s[len(s) // 2], 'sm_max_mhz': self.max_mhz, 'reasons': names, 'samples': len(s)}


# ------------------------------------------------------------------------------ our arm
def ours(args):
    import torch
    import torch.distributed as dist
    from marl_snake_b200 import SnakeBatch, allreduce_stats

    rank = int(os.environ.get('RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    if world > 1:
        dist.init_process_group('nccl', device_id=torch.device('cuda', local))
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)

    # CPU baseline first (rank 0, N=1 only), before the GPU is busy
    cpu = cpu_port = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        kind = reference_kind()
        cpu = cpu_leg(args.cpu_seconds, kind)
        if kind == 'reference':
            cpu_port = cpu_leg(5.0, 'port')
        cpu_native = cpu_native_leg()

    ns = ENV_KW['num_snakes']
    if args.envs_total:
        if args.envs_total % world:
            raise SystemExit('--envs-total must be a multiple of the number of GPUs')
        N = args.envs_total // world
    else:
        N = args.envs_per_gpu
    def make_batch():
        return SnakeBatch(N, device=local, seed=0, rng='philox', auto_reset=True, env_id_offset=rank * N, **ENV_KW)
    gen = torch.Generator(device=dev).manual_seed(1234 + rank)
    # A short action cycle would trap snakes in closed orbits (net turn of the cycle != 0 closes the
    # path after 4 cycles) and empty the workload of deaths and resets; 509 distinct tensors make the
    # cycle far longer than any snake lives (mean episode ~70 steps).
    NPOOL = 509
    pool = list(torch.randint(0, 3, (NPOOL, N, ns), dtype=torch.uint8, device=dev, generator=gen).unbind(0))   # one launch
    # The CPU baseline legs above leave the GPU idle for ~20 s and it drops to its idle clocks; a quarter of a second
    # of burn-in does not always bring the memory clock back (seen: 1.02 ms per step instead of 0.87).  Step for about
    # a second of wall time first, on a batch that is then thrown away: the step count of a wall-time loop varies
    # from run to run, and the measured batch must start from the same state every run.
    batch = make_batch()
    batch.reset()
    t_ramp, step_no = time.perf_counter(), 0
    while time.perf_counter() - t_ramp < CLOCK_RAMP_S:
        for _ in range(64):
            batch.step(pool[step_no % NPOOL], want_info=False)
            step_no += 1
        torch.cuda.synchronize()
    # Creating and resetting the measured batch idles the GPU for a few milliseconds only, and its burn-in and warm-up
    # (>= 356 steps, ~0.27 s at the default size) run back to back into the timed region; on a B200 (1000 W limit) this
    # order measured the same step time as ramping the measured batch itself (0.7675-0.7685 ms against 0.7676-0.7677).
    batch.close()
    del batch
    batch = make_batch()
    batch.reset()
    step_no = 0
    for t in range(BURN_IN + args.warmup):
        batch.step(pool[step_no % NPOOL], want_info=False)
        step_no += 1
    torch.cuda.synchronize()

    sampler = ClockSampler(local)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    sampler.start()
    # `ncu --profile-from-start off` lists exactly the launches of the timed region (a no-op without a profiler)
    torch.cuda.cudart().cudaProfilerStart()
    ev0.record()
    for t in range(args.steps):
        last = batch.step(pool[(step_no + t) % NPOOL], want_info=False)   # one kernel launch per step, current stream
    ev1.record()
    torch.cuda.synchronize()
    torch.cuda.cudart().cudaProfilerStop()
    sampler.stop_flag.set()
    ms = ev0.elapsed_time(ev1)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, *last[:3])
    del last
    if world > 1:
        dist.barrier()
        tms = torch.tensor([ms], device=dev, dtype=torch.float64)
        dist.all_reduce(tms, op=dist.ReduceOp.MAX)
        ms = float(tms.item())
    errs = batch.device_errors()
    st_after = batch.stats()

    # end-of-rollout statistics all-reduce (the only collective; outside the step path)
    stats = allreduce_stats(batch.stats_tensor().clone())
    stats_host = stats.cpu().tolist()

    # e2e: the reference-shaped call with HOST buffers (pinned), copies inside the timed region.  Default
    # transport of the C ABI for a block this size: channel bits over PCIe, widened to the reference's 0/1
    # bytes by the host cores (shared by the ranks of the box); the straight NHWC copy is timed beside it.
    K2 = max(1, args.e2e_steps)
    cores = len(os.sched_getaffinity(0)) if hasattr(os, 'sched_getaffinity') else (os.cpu_count() or 1)
    host_threads = max(1, cores // world)
    h_act = [p.cpu().pin_memory() for p in pool[:4]]
    h_obs = torch.empty((N,) + batch.obs_shape, dtype=torch.uint8).pin_memory()
    h_rew = torch.empty((N, ns), dtype=torch.float64).pin_memory()
    h_done = torch.empty((N, ns), dtype=torch.uint8).pin_memory()

    def time_host_steps(mode):
        batch.set_host_transport(mode, threads=host_threads)
        for t in range(2):
            batch.step_host(h_act[t % 4], h_obs, h_rew, h_done)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for t in range(K2):
            batch.step_host(h_act[t % 4], h_obs, h_rew, h_done)
        torch.cuda.synchronize()
        sec = time.perf_counter() - t0
        if world > 1:
            ts = torch.tensor([sec], device=dev, dtype=torch.float64)
            dist.all_reduce(ts, op=dist.ReduceOp.MAX)
            sec = float(ts.item())
        assert int(h_obs.max()) == 1 and bool((h_done <= 1).all())
        return sec

    e2e_raw_s = time_host_steps('raw')
    # context only: a host caller that consumes channel bits as they are (snk_step_host_bits, no widening)
    h_bits = torch.empty((N,) + batch.obs_shape[:-1] + (batch.obs_shape[-1] // 8,), dtype=torch.uint8).pin_memory()
    for t in range(2):
        batch.step_host_bits(h_act[t % 4], h_bits, h_rew, h_done)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for t in range(K2):
        batch.step_host_bits(h_act[t % 4], h_bits, h_rew, h_done)
    torch.cuda.synchronize()
    e2e_bits_s = time.perf_counter() - t0
    if world > 1:
        ts = torch.tensor([e2e_bits_s], device=dev, dtype=torch.float64)
        dist.all_reduce(ts, op=dist.ReduceOp.MAX)
        e2e_bits_s = float(ts.item())
    # the two ends of the packed transport on their own: (a) the device leg -- the step kernel emitting channel bits
    # (no NHWC block), CUDA events; (b) the host leg -- widening a block of channel bits that is already in host
    # memory into the caller's uint8 NHWC buffer with this rank's threads, i.e. the host-DRAM ceiling of the call
    d_act = [pool[t] for t in range(4)]
    for t in range(3):
        batch.step_bits(d_act[t % 4], want_info=False)
    evb0, evb1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    evb0.record()
    for t in range(20):
        batch.step_bits(d_act[t % 4], want_info=False)
    evb1.record()
    torch.cuda.synchronize()
    dev_leg_ms = evb0.elapsed_time(evb1) / 20
    import ctypes as C
    from marl_snake_b200 import lib as snk_lib
    n_units = h_bits.numel()
    if world > 1:
        dist.barrier()
    t0 = time.perf_counter()
    for t in range(3):
        snk_lib.snk_widen_bits_host(C.c_void_p(h_bits.data_ptr()), C.c_void_p(h_obs.data_ptr()), n_units, host_threads)
    widen_s = (time.perf_counter() - t0) / 3
    if world > 1:
        ts = torch.tensor([widen_s], device=dev, dtype=torch.float64)
        dist.all_reduce(ts, op=dist.ReduceOp.MAX)
        widen_s = float(ts.item())
    del h_bits
    e2e_s = time_host_steps('packed')
    # the delivered block against the device state of the same step: the window centre of a live snake is
    # its own head (channel 5), a dead snake's window sits on wall cell (0,0)  (byte parity: tests/)
    V = ENV_KW['vision_range']
    alive_now = batch.get_state()['alive'].cpu().bool()
    assert torch.equal(h_obs[:, :, V, V, 5].bool(), alive_now), 'packed transport: observation/state mismatch'
    assert int(h_obs[:8192].view(-1, 8).sum(1).max()) == 1

    # ---- the other BASELINE configs (driver-visible): cfg1 single-env latency through make_snake, cfg2 / cfg3 /
    #      cfg4 device-timed (1 GPU runs only); for N > 1 the strong-scaling reading of cfg5 (1,048,576 envs in
    #      total, sharded over the ranks, max over ranks).
    del h_obs, h_rew, h_done
    mean_ep = st_after['episode_steps_sum'] / max(st_after['episodes'], 1.0)
    algo_rec_bytes = batch.algorithmic_bytes_per_env_step()
    obs_shape = batch.obs_shape
    batch.close()
    del batch, pool
    torch.cuda.empty_cache()
    sys.path.insert(0, os.path.join(ROOT, 'tools'))
    import bench_configs as bc
    configs = {}
    if not args.no_configs:
        if world == 1:
            configs['cfg1'] = bc.measure_single_env()
            configs['cfg2'] = bc.measure('cfg2', steps=2000)
            configs['cfg2_graph'] = bc.measure('cfg2', steps=2000, graph=True)
            if hasattr(SnakeBatch, 'step_many'):
                configs['cfg2_step_many'] = bc.measure('cfg2', steps=2048, many=32)
            configs['cfg3'] = bc.measure('cfg3', steps=300)
            configs['cfg4'] = bc.measure('cfg4', steps=300)
            configs['cfg5_shard_131072'] = bc.measure('cfg5_shard', steps=400)
            try:                              # SURVEY N1: env + reference DQN + packed replay ring, all on the device
                configs['n1_rollout_cfg3'] = bc.measure_rollout()
            except Exception as exc:          # noqa: BLE001  (cuDNN / memory trouble must not cost the headline line)
                configs['n1_rollout_cfg3'] = {'unavailable': repr(exc)[:300]}
        else:
            total = 1 << 20
            kw = dict(bc.CONFIGS['cfg5_full'])
            kw['num_envs'] = total // world
            dist.barrier()
            r = bc.measure('cfg5_strong', steps=400, kw=kw, device=local, env_id_offset=rank * (total // world))
            tms = torch.tensor([r['ms_per_step']], device=dev, dtype=torch.float64)
            dist.all_reduce(tms, op=dist.ReduceOp.MAX)
            ms_strong = float(tms.item())
            scale = r['ms_per_step'] / ms_strong
            rf = r['roofline']
            configs['cfg5_strong'] = {
                'config': 'cfg5 read literally: 1,048,576 envs in total, %d per GPU' % (total // world),
                'scaling': 'strong', 'n_gpus': world, 'ms_per_step': ms_strong,
                'agent_steps_per_sec': total * ns / (ms_strong * 1e-3),
                'roofline_per_gpu': {'frac': rf['frac'] * scale, 'frac_record': rf['frac_record'] * scale,
                                     'achieved': rf['achieved'] * scale, 'peak': rf['peak'], 'unit': 'GB/s'}}

    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, 'MEASURED_PEAKS.json')))
        except Exception:
            pass
        peak = float(peaks.get('hbm_gbs', 6650.0))
        bytes_rec = algo_rec_bytes                      # what the kernel moves: 2 x 544-byte record + obs + I/O
        bytes_per_env = bc.survey_bytes_per_env_step(ENV_KW)   # SURVEY 8(d): 2*H*W + ns*(O + P + 38) = 4 824
        obs_bytes = 1
        for x in obs_shape:
            obs_bytes *= x
        rec_bytes = (bytes_rec - obs_bytes - 10 * ns) // 2
        per_launch = bytes_per_env * N
        achieved = per_launch / (ms / args.steps * 1e-3) / 1e9
        achieved_rec = bytes_rec * N / (ms / args.steps * 1e-3) / 1e9
        traffic = None
        try:
            traffic = bc.traffic_per_launch('cfg5_full')
        except Exception:
            pass
        value = N * world * ns * args.steps / (ms * 1e-3)
        out = {
            'metric': 'agent_steps_per_sec', 'value': value, 'unit': 'agent-steps/s', 'n_gpus': world,
            'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': ms / args.steps,
            'higher_is_better': True, 'scaling': 'strong' if args.envs_total else 'weak', 'vs_baseline': None,
            'dtype': 'u8', 'data': 'synthetic',
            'config': {'workload': WORKLOAD, 'envs_per_gpu': N, 'global_envs': N * world, 'burn_in_steps': BURN_IN, 'clock_ramp_s': CLOCK_RAMP_S,
                       'l2': 'no flush: per-step working set (records %.0f MB read + written, obs %.0f MB written) '
                             'exceeds the 126 MB L2' % (N * rec_bytes / 1e6, N * obs_bytes / 1e6),
                       'parallelism': f'env-shard x{world}', 'rng': 'philox seed 0',
                       'tile_envs': os.environ.get('SNK_TILE_ENVS', 'auto'), 'threads': os.environ.get('SNK_THREADS', 'auto'),
                       'mean_episode_steps_rank0': mean_ep,
                       'device_errors': errs},
            'roofline': {'bound': 'hbm', 'achieved': achieved, 'peak': peak, 'unit': 'GB/s',
                         'frac': achieved / peak, 'frac_of_nominal_8000_gbs': achieved / 8000.0, 'traffic': traffic,
                         'peak_source': 'MEASURED_PEAKS.json hbm_gbs (measured)' if peaks else 'fallback 6650',
                         'algorithmic_bytes_per_env_step': bytes_per_env,
                         'bytes_formula': 'SURVEY.md 8(d): 2*H*W + ns*(O + P + 38) with a 400-byte state',
                         'record_bytes_per_env_step': bytes_rec, 'achieved_record': achieved_rec,
                         'frac_record': achieved_rec / peak, 'hbm_record_bytes': rec_bytes,
                         'note': 'frac = SURVEY bytes / time / peak; the model reads and writes a 400-byte grid per env-step, '
                                 'the resident record holds no grid (rebuilt in shared memory), so the step moves '
                                 'record_bytes_per_env_step and frac can exceed 1; frac_record is the physical utilisation',
                         'kernel': 'snk_tile_kernel',
                         'launch_ms': ms / args.steps},
            'configs': configs,
            'e2e': {'value': N * world * ns * K2 / e2e_s, 'unit': 'agent-steps/s',
                    # bytes that cross PCIe per step per rank: actions in; channel-bit observations, float64
                    # rewards and dones out.  The call delivers N*obs_bytes of uint8 NHWC into the host buffer.
                    'h2d_bytes_per_step': N * ns, 'd2h_bytes_per_step': N * obs_bytes // 8 + N * ns * 9,
                    'host_obs_bytes_delivered_per_step': N * obs_bytes,
                    'steps': K2, 'ms_per_step': 1e3 * e2e_s / K2,
                    'api': 'snk_step_host (C ABI, pinned host buffers), packed transport: the step kernel emits channel '
                           'bits, %d MB over PCIe in chunks, %d host threads per rank widen to uint8 NHWC'
                           % (obs_bytes * N // 8 // 1000000, host_threads),
                    'host_threads_per_rank': host_threads,
                    'bits_format': {'value': N * world * ns * K2 / e2e_bits_s, 'ms_per_step': 1e3 * e2e_bits_s / K2,
                                    'd2h_bytes_per_step': N * obs_bytes // 8 + N * ns * 9,
                                    'note': 'snk_step_host_bits: the same call delivering channel bits as they are (one '
                                            'byte per cell, bit c = channel c; np.packbits of the reference format) -- no '
                                            'host widening, PCIe-bound'},
                    'device_leg_ms': dev_leg_ms,
                    'device_leg_note': 'step kernel emitting channel bits (snk_step_bits), CUDA events, per step',
                    'host_widen_only_ms': 1e3 * widen_s,
                    'host_dram_ceiling': {'value': N * world * ns / widen_s, 'unit': 'agent-steps/s',
                                          'note': 'all ranks widening a resident bit block into their uint8 NHWC host '
                                                  'buffers at once, no GPU, no PCIe: what the box\'s host memory system '
                                                  'allows for the reference format (%d threads per rank)' % host_threads},
                    'raw_transport': {'value': N * world * ns * K2 / e2e_raw_s, 'ms_per_step': 1e3 * e2e_raw_s / K2,
                                      'd2h_bytes_per_step': N * obs_bytes + N * ns * 9}},
            'gpu_launches': args.steps * world,       # timed region of `value`: one snk_tile_kernel per step per rank
            'clocks': sampler.summary(),
            'rollout_stats': dict(zip(('episodes', 'return_sum', 'episode_steps_sum', 'fruits_sum', 'kills_sum',
                                       'deaths'), stats_host[:6])),
        }
        if cpu:
            out['cpu_baseline'] = cpu
            if cpu_port:
                out['cpu_port'] = cpu_port
            out['cpu_native_1thread'] = cpu_native
        print(json.dumps(out), file=RESULT_OUT, flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == '__main__':
    # stdout must carry exactly ONE JSON line.  Libraries write there too (NCCL prints its version banner to
    # stdout when NCCL_DEBUG is set), so file descriptor 1 is pointed at stderr for the whole run and the
    # result line goes to a private duplicate of the original stdout.
    RESULT_OUT = os.fdopen(os.dup(1), 'w')
    sys.stdout.flush()
    os.dup2(2, 1)
    a = parse()
    if a.impl == 'reference':
        reference_arm(a)
    else:
        ours(a)
