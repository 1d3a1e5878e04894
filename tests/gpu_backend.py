"""Adapter: libsnk.so (through marl_snake_b200.SnakeBatch, i.e. through the C ABI) behind the same
little interface the parity drivers use for the host simulation."""
import numpy as np
import torch


class GpuBackend:
    def __init__(self, num_envs, kw, rng_mode=1, auto_reset=1, seed=0, env_id_offset=0, done_mode=0, plain_obs=False):
        """plain_obs: step into a plain torch buffer through snk_step instead of the batch's observation block, which
        is compressible where the device grants it (and there the step runs the capped instance)."""
        from marl_snake_b200 import SnakeBatch
        self.b = SnakeBatch(num_envs, rng='replay' if rng_mode else 'philox', auto_reset=bool(auto_reset),
                            seed=seed, env_id_offset=env_id_offset, done_mode='any' if done_mode else 'all', **kw)
        self.N, self.ns = num_envs, self.b.num_snakes
        self.plain = None
        if plain_obs:
            dev = self.b.device
            self.plain = dict(obs=torch.empty((self.N,) + self.b.obs_shape, dtype=torch.uint8, device=dev),
                              rew=torch.empty((self.N, self.ns), dtype=torch.float64, device=dev),
                              done=torch.empty((self.N, self.ns), dtype=torch.uint8, device=dev),
                              fin=torch.empty((self.N,), dtype=torch.uint8, device=dev))

    def set_replay(self, draws):
        self.b.set_replay(draws)

    def reset(self):
        return self.b.reset().cpu().numpy()

    def step(self, actions, around=None):
        """around: with plain_obs, a context-manager factory entered around the launch alone (its value is kept in
        self.around_value), e.g. a launch witness."""
        a = torch.as_tensor(np.ascontiguousarray(actions, dtype=np.uint8).reshape(self.N, self.ns)).to(self.b.device)
        if self.plain is not None:
            import ctypes as C
            from marl_snake_b200._lib import SnkStepExtra, check, lib
            p = self.plain
            x = SnkStepExtra(p['fin'].data_ptr(), None, None, None, None, None)
            import contextlib
            with (around or contextlib.nullcontext)() as self.around_value:
                check(lib.snk_step(self.b._h, C.c_void_p(a.data_ptr()), C.c_void_p(p['obs'].data_ptr()),
                                   C.c_void_p(p['rew'].data_ptr()), C.c_void_p(p['done'].data_ptr()), C.byref(x),
                                   self.b._stream()))
            return (p['obs'].cpu().numpy(), p['rew'].cpu().numpy(), p['done'].cpu().numpy().astype(bool),
                    dict(finished=p['fin'].cpu().numpy().astype(bool)))
        obs, rew, done, info = self.b.step(a)
        return (obs.cpu().numpy(), rew.cpu().numpy(), done.cpu().numpy(),
                {k: v.cpu().numpy() for k, v in info.items()})

    def grid(self):
        st = self.b.get_state()
        cur = self.b.replay_cursors() if self.b.rng == 'replay' else np.zeros(self.N, np.int32)
        return st['grid'].cpu().numpy().reshape(self.N, -1), st['alive_counter'].cpu().numpy(), cur

    def set_state(self, grid, alive, dir, length, cells, counter, ep_len=None):
        return self.b.set_state(grid, alive, dir, length, cells, counter, ep_len).cpu().numpy()

    def errors(self):
        return self.b.device_errors()

    def close(self):
        self.b.close()
