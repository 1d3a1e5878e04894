"""GPU-resident rollout plumbing for value-based callers (SURVEY N1).

The reference's DQN trainer runs one tiny forward per live snake, moves every observation host -> device
and synchronises with `.item()` per action (train_dqn.py:163-173, 277-308) and keeps its replay buffer in
a Python deque (:89-100).  With the environment on the GPU the whole loop can stay there: batched
epsilon-greedy straight from the device observation, transitions written into a device ring buffer, no
host synchronisation per step.  Everything here is torch tensor plumbing around `SnakeBatch.step`; the
game itself stays in the CUDA library.
"""
import ctypes as C

import torch

from ._lib import check, lib


def epsilon_greedy(q_values, epsilon, generator=None):
    """q_values: float [B, n_actions] on the GPU -> uint8 actions [B]; with probability epsilon uniform."""
    B, n = q_values.shape
    greedy = q_values.argmax(dim=1)
    explore = torch.rand(B, device=q_values.device, generator=generator) < epsilon
    rand = torch.randint(0, n, (B,), device=q_values.device, generator=generator)
    return torch.where(explore, rand, greedy).to(torch.uint8)


def unpack_obs(bits):
    """Inverse of SnakeBatch.pack_obs on the device: uint8 [..., F] channel-bit bytes -> uint8 0/1 [..., 8*F]."""
    shifts = torch.arange(8, device=bits.device, dtype=torch.uint8)
    return ((bits.unsqueeze(-1) >> shifts) & 1).reshape(*bits.shape[:-1], bits.shape[-1] * 8)


class DeviceReplayBuffer:
    """Fixed-capacity ring of transitions in device memory; observations stay uint8 (NHWC).  With
    `pack=batch` (a SnakeBatch) observations are stored as channel bits -- one byte per (cell, frame), an
    eighth of the memory -- packed by the library's kernel on push and widened again on sample."""

    def __init__(self, capacity, obs_shape, device, pack=None):
        self.capacity, self.size, self.pos, self.pack = int(capacity), 0, 0, pack
        stored = (*obs_shape[:-1], obs_shape[-1] // 8) if pack is not None else tuple(obs_shape)
        self.obs = torch.empty((capacity, *stored), dtype=torch.uint8, device=device)
        self.next_obs = torch.empty_like(self.obs)
        self.action = torch.empty(capacity, dtype=torch.uint8, device=device)
        self.reward = torch.empty(capacity, dtype=torch.float32, device=device)
        self.done = torch.empty(capacity, dtype=torch.bool, device=device)

    def push(self, obs, action, reward, next_obs, done):
        """Append a batch of transitions (any leading batch size <= capacity), wrapping around."""
        n = obs.shape[0]
        if n == 0:
            return
        if n > self.capacity:
            obs, action, reward, next_obs, done = (t[-self.capacity:] for t in (obs, action, reward, next_obs, done))
            n = self.capacity
        if self.pack is not None:
            obs, next_obs = self.pack.pack_obs(obs.contiguous()), self.pack.pack_obs(next_obs.contiguous())
        idx = (self.pos + torch.arange(n, device=obs.device)) % self.capacity
        self.obs[idx], self.next_obs[idx] = obs, next_obs
        self.action[idx], self.reward[idx], self.done[idx] = action, reward.to(torch.float32), done
        self.pos = (self.pos + n) % self.capacity
        self.size = min(self.size + n, self.capacity)

    def sample(self, batch_size, generator=None):
        idx = torch.randint(0, self.size, (batch_size,), device=self.obs.device, generator=generator)
        obs, next_obs = self.obs[idx], self.next_obs[idx]
        if self.pack is not None:
            obs, next_obs = unpack_obs(obs), unpack_obs(next_obs)
        return obs, self.action[idx], self.reward[idx], next_obs, self.done[idx]


class GraphedSteps:
    """T environment steps captured once in a CUDA graph and replayed with a single launch call.

    A step is one kernel with no host synchronisation, so a short batch (BASELINE cfg2: 4 096 envs, ~20 us of
    work per step) is bound by launch latency; replaying a captured sequence removes the per-step launch
    overhead (profiles/README.md: 21 -> 19 us per step).  `actions` is a uint8 CUDA tensor [T, N, ns] that
    the caller refills between replays; after a replay the batch's own obs / reward / done buffers hold the
    last step's outputs and, when `keep` is true, `rewards[T, N, ns]` / `dones[T, N, ns]` hold every step's."""

    def __init__(self, batch, actions, keep=True):
        if actions.dtype != torch.uint8 or actions.dim() != 3 or tuple(actions.shape[1:]) != (batch.num_envs, batch.num_snakes):
            raise ValueError('actions must be a uint8 CUDA tensor of shape [T, num_envs, num_snakes]')
        self.batch, self.actions, self.T = batch, actions, actions.shape[0]
        self.rewards = torch.empty((self.T, batch.num_envs, batch.num_snakes), dtype=torch.float64, device=actions.device) if keep else None
        self.dones = torch.empty((self.T, batch.num_envs, batch.num_snakes), dtype=torch.bool, device=actions.device) if keep else None
        stream = torch.cuda.Stream(device=actions.device)
        stream.wait_stream(torch.cuda.current_stream(actions.device))
        self.graph = torch.cuda.CUDAGraph()
        mark = (batch._mutations, batch._obs_stale)
        with torch.cuda.stream(stream):
            with torch.cuda.graph(self.graph, stream=stream):
                for t in range(self.T):
                    obs, rew, done, _ = batch.step(actions[t], want_info=False)
                    if keep:
                        self.rewards[t].copy_(rew)
                        self.dones[t].copy_(done)
        torch.cuda.current_stream(actions.device).wait_stream(stream)
        batch._mutations, batch._obs_stale = mark              # capturing ran nothing
        self.obs = obs

    def replay(self):
        """Run the T captured steps (asynchronous; outputs are valid on the current stream afterwards)."""
        b = self.batch
        stream = torch.cuda.current_stream(b.device)
        self.graph.replay()
        # the replayed kernels bypass the library: report the stream so that a following host-buffer call waits for them
        check(lib.snk_note_stream(b._h, C.c_void_p(stream.cuda_stream)))
        b._mutated(None)
        return self.obs, self.rewards, self.dones


@torch.no_grad()
def collect(batch, q_net, steps, buffer=None, epsilon=0.1, generator=None, early_death=None, max_steps=None,
            to_input=None):
    """Run `steps` env steps of `batch` (SnakeBatch, auto-reset on) with a shared per-snake Q network -- the
    inner loop of the reference trainer (train_dqn.py:277-308) for every environment of the batch at once:

      * one batched forward over all [N*ns] observations (float NCHW built from the uint8 NHWC observation, as
        train_dqn.py:118,168 does per snake; `to_input` overrides the conversion), epsilon-greedy on the device;
        snakes that are already dead send action 0 (:281-282);
      * a transition (obs_i, action_i, r_i, next_obs_i, next_done_i) is pushed for every snake that was alive
        BEFORE the step and for no other (:290-298), in (env, snake) order; with `early_death=(threshold, penalty)`
        a snake that dies while its episode is younger than `threshold` steps gets `penalty` added (:293-295);
      * an episode that ended was reset inside the step (the vector worker's rule, wrappers.py:141-143): its
        `next_obs` is the first observation of the next episode and all of its snakes are alive again;
      * with `max_steps`, an episode that reaches that many steps is cut and restarted without a done flag, as the
        trainer's `step < MAX_STEPS_PER_EPISODE` loop condition does (:275, 270) -- one masked reset launch per step.

    The alive mask and the per-env episode age are read back from the device state (`snk_get_state`) when the batch
    was stepped, reset, restored or replayed by anything else since the last call, so consecutive calls continue the
    same rollout.  The observations come from the batch's own buffer, which step(), full reset(), set_state() and
    GraphedSteps.replay() keep current; after any other stepping or resetting call (step_bits, step_many, the
    host-buffer calls, reset(bits=True), load_checkpoint, step(want_obs=False)) collect raises ValueError until
    reset() or step() renders it again.  A batch that was never reset is reset by the first call.
    Returns the number of transitions written (a device scalar); nothing is copied to the host."""
    N, ns = batch.num_envs, batch.num_snakes
    if batch._obs_stale is not None:
        if batch._mutations:
            raise ValueError(f"collect: the batch's observation buffer is out of date after {batch._obs_stale}; "
                             'call reset() or step() to restore it')
        batch.reset()
    if batch._rollout_mark != batch._mutations:  # first call, or the batch was changed by another call in between
        st = batch.get_state()
        batch._rollout_alive, batch._rollout_age = st['alive'].bool(), st['episode_length']
    obs = batch._obs
    alive, age = batch._rollout_alive, batch._rollout_age
    written = torch.zeros((), dtype=torch.int64, device=obs.device)
    for _ in range(steps):
        flat = obs.reshape(N * ns, *obs.shape[2:])
        q = q_net(to_input(flat) if to_input is not None else flat.permute(0, 3, 1, 2).float())
        actions = epsilon_greedy(q.float(), epsilon, generator).reshape(N, ns)
        actions = torch.where(alive, actions, torch.zeros_like(actions))
        prev = flat.clone() if buffer is not None else None
        obs, rew, done, info = batch.step(actions)
        if buffer is not None:
            m = alive.reshape(-1)
            if early_death is not None:
                threshold, penalty = early_death
                rew = rew + (done & (age < threshold)[:, None]).to(rew.dtype) * penalty
            buffer.push(prev[m], actions.reshape(-1)[m], rew.reshape(-1)[m],
                        obs.reshape(N * ns, *obs.shape[2:])[m], done.reshape(-1)[m])
            written += m.sum()
        # a finished env was reset inside the step: all of its snakes are alive again, its age is 0
        fin = info['finished'].bool()
        alive = torch.where(fin[:, None], torch.ones_like(done), ~done)
        age = torch.where(fin, torch.zeros_like(age), age + 1)
        if max_steps is not None:
            cut = age >= max_steps
            obs = batch.reset(mask=cut)
            alive, age = alive | cut[:, None], torch.where(cut, torch.zeros_like(age), age)
    batch._rollout_alive, batch._rollout_age, batch._rollout_mark = alive, age, batch._mutations
    return written
