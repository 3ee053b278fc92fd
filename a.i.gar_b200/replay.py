"""Host binding of the GPU replay buffer (include/agar_replay.h): mirrors src/model/replay_buffer.py's
ReplayBuffer / PrioritizedReplayBuffer for batches of transitions that stay on the GPU.  Randomness is injected
(uniforms in [0, 1)) exactly where the reference calls random.randint / random.random."""
import ctypes

import numpy as np

from . import env as _env

CheckpointError = _env.CheckpointError
ERR_STATE = 8  # AGAR_RP_ERR_STATE: a bank refused by agar_replay_load

REPLAY_CHECKPOINT_FORMAT = "agar_b200.replay.v1"
_REPLAY_KEYS = ("format", "capacity", "state_len", "action_len", "prioritized", "alpha", "beta", "bank", "sha256")


def write_replay_checkpoint(path, capacity, state_len, action_len, prioritized, alpha, beta, bank):
    """Write a replay-buffer checkpoint (.npz, no pickled objects).  bank: the uint8 host bytes of agar_replay_save."""
    _env.save_npz_checkpoint(path, REPLAY_CHECKPOINT_FORMAT, "bank", capacity=np.int64(capacity), state_len=np.int64(state_len),
                             action_len=np.int64(action_len), prioritized=np.bool_(prioritized), alpha=np.float64(alpha),
                             beta=np.float64(beta), bank=np.ravel(bank))


def read_replay_checkpoint(path):
    """Parse a replay checkpoint without a device: a dict of its fields.  Raises CheckpointError for a file that is not one of
    this format, whose bank is not 1-D uint8, or whose digest differs."""
    ck = _env.load_npz_checkpoint(path, REPLAY_CHECKPOINT_FORMAT, _REPLAY_KEYS, "replay")
    if ck["bank"].dtype != np.uint8 or ck["bank"].ndim != 1:
        raise CheckpointError("%s: bank of shape %s / %s is not 1-D uint8" % (path, ck["bank"].shape, ck["bank"].dtype))
    _env.check_npz_digest(path, ck, "bank")
    return ck


def check_replay_checkpoint(ck, capacity, state_len, action_len, prioritized, alpha, beta, state_bytes):
    """Raise CheckpointError naming the first field of a parsed replay checkpoint that differs from a buffer's
    (state_bytes: the buffer's bank size)."""
    for name, mine in (("capacity", capacity), ("state_len", state_len), ("action_len", action_len)):
        if int(ck[name]) != int(mine):
            raise CheckpointError("checkpoint %s is %d, the buffer's is %d" % (name, int(ck[name]), int(mine)))
    if bool(ck["prioritized"]) != bool(prioritized):
        raise CheckpointError("checkpoint prioritized is %s, the buffer's is %s" % (bool(ck["prioritized"]), bool(prioritized)))
    for name, mine in (("alpha", alpha), ("beta", beta)):  # compared bit for bit, as the device compares them
        if np.float64(ck[name]).tobytes() != np.float64(mine).tobytes():
            raise CheckpointError("checkpoint %s is %r, the buffer's is %r" % (name, float(ck[name]), float(mine)))
    if ck["bank"].size != int(state_bytes):
        raise CheckpointError("checkpoint bank has %d bytes, the buffer's has %d" % (ck["bank"].size, int(state_bytes)))


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
        self.alpha, self.beta = float(alpha), float(beta)
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
        """Sticky AGAR_RP_ERR_* bits (1 sampled a too-small buffer, 2 index out of range, 4 priority <= 0, 8 a state bank
        refused on restore)."""
        return int(self.lib.agar_replay_error_flags(self.h, self._stream()))

    def raise_on_error(self):
        """The reference raises / asserts in these cases (replay_buffer.py:66,116,203-204); call after a sync point."""
        f = self.error_flags
        if f:
            raise _env.AgarError("replay buffer error flags %d (1 = sampled from a buffer that is too small, 2 = index out of "
                                 "range, 4 = priority <= 0, 8 = a state bank refused on restore)" % f)

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

    # ---- state snapshots (agar_replay_save / agar_replay_load; bank layout in include/agar_replay.h)
    @property
    def state_bytes(self):
        """bytes of one bank of this buffer"""
        n = _env.bind_lazy(self.lib, "agar_replay_state_bytes", [ctypes.c_void_p], ctypes.c_int64)(self.h)
        if n < 0:
            self._check(int(n))
        return int(n)

    def _bank(self, bank):
        t = self.torch
        n = self.state_bytes
        if not (t.is_tensor(bank) and bank.dtype == t.uint8 and bank.device == self.device and bank.dim() == 1 and
                bank.numel() == n and bank.is_contiguous()):
            raise ValueError("a replay bank is a contiguous 1-D uint8 tensor of %d bytes on %s" % (n, self.device))
        return bank

    def snapshot(self, out=None):
        """The buffer's whole state (ring, next index, size, max priority, tree leaves) as a 1-D uint8 device tensor of
        state_bytes.  Canonical: two buffers with the same observable state give equal banks.  out: a bank to reuse."""
        out = self._bank(self.torch.empty(self.state_bytes, dtype=self.torch.uint8, device=self.device) if out is None else out)
        fn = _env.bind_lazy(self.lib, "agar_replay_save", [ctypes.c_void_p] * 3)
        self._check(fn(self.h, self._p(out), self._stream()))
        return out

    def restore(self, bank):
        """Install a bank of a buffer created with the same size, state_len, action_len, prioritized, alpha and beta; a clone is
        other.restore(buf.snapshot()).  The device checks the bank first: a refused one leaves this buffer unchanged and sets
        error flag 8.  No host synchronisation: a CUDA graph can capture it."""
        fn = _env.bind_lazy(self.lib, "agar_replay_load", [ctypes.c_void_p] * 3)
        self._check(fn(self.h, self._p(self._bank(bank)), self._stream()))

    def _fields(self):
        return (self.size_max, self.state_len, self.action_len, self.prioritized, self.alpha, self.beta)

    def save_checkpoint(self, path):
        """Write the buffer's bank with what a later load must match (size, state_len, action_len, prioritized, alpha, beta)."""
        write_replay_checkpoint(path, *self._fields(), bank=self.snapshot().cpu().numpy())

    def load_checkpoint(self, path):
        """Restore from a checkpoint of a buffer with the same parameters.  A file that differs in one of them, whose digest
        is wrong or whose bank the device refuses raises CheckpointError and leaves the buffer as it was."""
        ck = read_replay_checkpoint(path)
        check_replay_checkpoint(ck, *self._fields(), state_bytes=self.state_bytes)
        bank = self.torch.from_numpy(ck["bank"]).to(self.device)
        self.restore(bank)
        # banks are canonical, so an installed bank saves back unchanged; the sticky flag may have been set earlier
        if not self.torch.equal(self.snapshot(), bank):
            raise CheckpointError("%s: a bank that fails the device-side checks; nothing was loaded" % path)

    @classmethod
    def from_checkpoint(cls, path, device=0):
        """A new buffer with a checkpoint's parameters, loaded from it."""
        ck = read_replay_checkpoint(path)
        rp = cls(int(ck["capacity"]), int(ck["state_len"]), int(ck["action_len"]), bool(ck["prioritized"]), float(ck["alpha"]),
                 float(ck["beta"]), device=device)
        rp.load_checkpoint(path)
        return rp
