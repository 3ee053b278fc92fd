"""Host binding of the GPU replay buffer (include/agar_replay.h): mirrors src/model/replay_buffer.py's
ReplayBuffer / PrioritizedReplayBuffer for batches of transitions that stay on the GPU.  Randomness is injected
(uniforms in [0, 1)) exactly where the reference calls random.randint / random.random."""
import ctypes

from . import env as _env


def _bind(lib):
    if getattr(lib, "_replay_bound", False):
        return lib
    vp, i32, dbl = ctypes.c_void_p, ctypes.c_int, ctypes.c_double
    lib.agar_replay_create.argtypes = [i32, i32, i32, i32, dbl, dbl, i32, ctypes.POINTER(vp)]
    lib.agar_replay_destroy.argtypes = [vp]
    lib.agar_replay_last_error.argtypes = [vp]
    lib.agar_replay_last_error.restype = ctypes.c_char_p
    lib.agar_replay_size.argtypes = [vp, vp]
    lib.agar_replay_next_idx.argtypes = [vp, vp]
    lib.agar_replay_add_batch.argtypes = [vp] + [vp] * 6 + [i32, vp]
    lib.agar_replay_gather.argtypes = [vp, vp, i32] + [vp] * 5 + [vp]
    lib.agar_replay_sample_uniform.argtypes = [vp, vp, i32, vp] + [vp] * 5 + [vp]
    lib.agar_replay_sample_prioritized.argtypes = [vp, vp, i32, vp, vp] + [vp] * 5 + [vp]
    lib.agar_replay_update_priorities.argtypes = [vp, vp, vp, i32, vp]
    lib.agar_replay_error_flags.argtypes = [vp, vp]
    lib.agar_replay_launch_count.argtypes = [vp]
    lib.agar_replay_launch_count.restype = ctypes.c_int64
    lib._replay_bound = True
    return lib


def trajectory_transitions(traj):
    """(obs_t, action, reward, obs_tp1, done, valid) of every transition in a recorded rollout (env.Trajectory): decision d's
    observation and action, then the reward, observation, done and valid read after decision d + 1's observation -- the
    alignment of the per-tick loops (step_observe, then add_batch).  Contiguous views, no copies.  It holds when every decision
    is one bot turn (n_frames == frame_skip + 1); any other trajectory is refused."""
    missing = [f for f in ("obs", "action", "reward", "done", "valid") if getattr(traj, f) is None]
    if missing:
        raise ValueError("add_trajectory needs the %s fields recorded" % ", ".join(missing))
    if traj.n_frames != traj.frame_skip + 1:
        raise ValueError("add_trajectory needs one bot turn per decision (n_frames == frame_skip + 1 == %d); this trajectory "
                         "has n_frames = %s" % (traj.frame_skip + 1, traj.n_frames))
    return traj.obs[:-1], traj.action, traj.reward[1:], traj.obs[1:], traj.done[1:], traj.valid[1:]


class GpuReplayBuffer(object):
    """ReplayBuffer(size) / PrioritizedReplayBuffer(size, alpha, beta) on one GPU."""

    def __init__(self, size, state_len, action_len=4, prioritized=False, alpha=0.6, beta=0.4, device=0):
        import torch
        if not torch.cuda.is_available():
            raise _env.AgarError("no CUDA device: the replay buffer has no CPU fallback")
        self.torch = torch
        self.lib = _bind(_env.load_library())
        self.device = torch.device("cuda", device)
        self.size_max, self.state_len, self.action_len, self.prioritized = size, state_len, action_len, bool(prioritized)
        self.h = ctypes.c_void_p()
        rc = self.lib.agar_replay_create(size, state_len, action_len, int(prioritized), alpha, beta, self.device.index,
                                         ctypes.byref(self.h))
        if rc != 0:
            raise _env.AgarError("agar_replay_create failed (%d): %s" % (rc, self.lib.agar_replay_last_error(None).decode()))

    def _stream(self):
        return ctypes.c_void_p(self.torch.cuda.current_stream(self.device).cuda_stream)

    def _check(self, rc):
        if rc != 0:
            raise _env.AgarError("replay call failed (%d): %s" % (rc, self.lib.agar_replay_last_error(self.h).decode()))

    def _p(self, t):
        return ctypes.c_void_p(t.data_ptr()) if t is not None else ctypes.c_void_p()

    def close(self):
        if getattr(self, "h", None) and self.h.value:
            self.lib.agar_replay_destroy(self.h)
            self.h = ctypes.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __len__(self):
        return int(self.lib.agar_replay_size(self.h, self._stream()))

    @property
    def next_idx(self):
        return int(self.lib.agar_replay_next_idx(self.h, self._stream()))

    @property
    def error_flags(self):
        """Sticky AGAR_RP_ERR_* bits (1 sampled a too-small buffer, 2 index out of range, 4 priority <= 0)."""
        return int(self.lib.agar_replay_error_flags(self.h, self._stream()))

    def raise_on_error(self):
        """The reference raises / asserts in these cases (replay_buffer.py:66,116,203-204); call after a sync point."""
        f = self.error_flags
        if f:
            raise _env.AgarError("replay buffer error flags %d (1 = sampled from a buffer that is too small, 2 = index out of "
                                 "range, 4 = priority <= 0)" % f)

    @property
    def launch_count(self):
        return int(self.lib.agar_replay_launch_count(self.h))

    def add_batch(self, obs_t, action, reward, obs_tp1, done, valid=None):
        """ReplayBuffer.add for every transition with valid != 0, in index order.  Tensors on this device."""
        t = self.torch
        n = int(reward.numel())
        obs_t = obs_t.reshape(n, self.state_len).contiguous().float()
        obs_tp1 = obs_tp1.reshape(n, self.state_len).contiguous().float()
        action = action.reshape(n, -1)[:, :self.action_len].contiguous().float()
        reward = reward.reshape(n).contiguous().float()
        done = done.reshape(n).contiguous().to(t.uint8)
        valid = None if valid is None else valid.reshape(n).contiguous().to(t.uint8)
        self._check(self.lib.agar_replay_add_batch(self.h, self._p(obs_t), self._p(action), self._p(reward), self._p(obs_tp1),
                                                   self._p(done), self._p(valid), n, self._stream()))

    def add_trajectory(self, traj):
        """Every transition of a recorded rollout (AgarBatch.rollout) in one add_batch of D x E x A transitions, in
        (decision, env, agent) order: see trajectory_transitions for the alignment and what is refused."""
        self.add_batch(*trajectory_transitions(traj))

    def _outs(self, batch):
        t = self.torch
        return (t.empty((batch, self.state_len), dtype=t.float32, device=self.device),
                t.empty((batch, self.action_len), dtype=t.float32, device=self.device),
                t.empty((batch,), dtype=t.float32, device=self.device),
                t.empty((batch, self.state_len), dtype=t.float32, device=self.device),
                t.empty((batch,), dtype=t.uint8, device=self.device))

    def gather(self, idx):
        idx = idx.to(self.device, self.torch.int32).contiguous()
        o = self._outs(int(idx.numel()))
        self._check(self.lib.agar_replay_gather(self.h, self._p(idx), int(idx.numel()), *[self._p(x) for x in o], self._stream()))
        return o

    def sample(self, uniforms):
        """ReplayBuffer.sample / PrioritizedReplayBuffer.sample with the caller's uniforms (float64 in [0, 1))."""
        t = self.torch
        u = t.as_tensor(uniforms, dtype=t.float64, device=self.device).contiguous()
        batch = int(u.numel())
        idx = t.empty((batch,), dtype=t.int32, device=self.device)
        o = self._outs(batch)
        if self.prioritized:
            w = t.empty((batch,), dtype=t.float64, device=self.device)
            self._check(self.lib.agar_replay_sample_prioritized(self.h, self._p(u), batch, self._p(idx), self._p(w),
                                                                *[self._p(x) for x in o], self._stream()))
            return o + (w, idx)
        self._check(self.lib.agar_replay_sample_uniform(self.h, self._p(u), batch, self._p(idx), *[self._p(x) for x in o],
                                                        self._stream()))
        return o + (idx,)

    def update_priorities(self, idx, priorities):
        t = self.torch
        idx = t.as_tensor(idx, device=self.device).to(t.int32).contiguous()
        pr = t.as_tensor(priorities, dtype=t.float64, device=self.device).contiguous()
        self._check(self.lib.agar_replay_update_priorities(self.h, self._p(idx), self._p(pr), int(idx.numel()), self._stream()))
