"""Host side of the batched agar.io env: a thin ctypes binding of include/agar_b200.h plus the mirror of the
reference's Model / Bot surface (src/model/model.py:90-120, src/model/bot.py:252-299,645).

PyTorch is used for device memory, streams and DLPack only.  There is NO CPU fallback: if libagar_b200.so is
missing or no CUDA device is present every constructor raises."""
import ctypes
import os

import numpy as np

from . import layout as lay

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.environ.get("AGAR_B200_LIB", os.path.join(_HERE, "libagar_b200.so"))  # override: A/B builds
_lib = None

EXPORTS = ["agar_layout_for_config", "agar_create", "agar_destroy", "agar_last_error", "agar_get_layout", "agar_num_envs",
           "agar_reset", "agar_reset_bots", "agar_observe", "agar_step", "agar_step_observe", "agar_get",
           "agar_debug_dump", "agar_debug_load", "agar_launch_count", "agar_step_host", "agar_rollout_random",
           "agar_set_tile_width", "agar_get_tile_width", "agar_state_ptr",
           "agar_step_host_begin", "agar_step_host_end"]


def load_library():
    """dlopen the in-tree CUDA library; fail loudly when it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(_LIB_PATH):
        raise ImportError("%s not found: build it with `python -m aigar_b200.build` (needs nvcc); "
                          "there is no CPU fallback" % _LIB_PATH)
    lib = ctypes.CDLL(_LIB_PATH)
    vp, i32, u64, u32 = ctypes.c_void_p, ctypes.c_int, ctypes.c_uint64, ctypes.c_uint32
    lib.agar_layout_for_config.argtypes = [ctypes.POINTER(lay.AgarConfig), ctypes.POINTER(lay.AgarLayout)]
    lib.agar_create.argtypes = [ctypes.POINTER(lay.AgarConfig), i32, i32, u64, u64, vp, ctypes.POINTER(vp)]
    lib.agar_destroy.argtypes = [vp]
    lib.agar_last_error.argtypes = [vp]
    lib.agar_last_error.restype = ctypes.c_char_p
    lib.agar_get_layout.argtypes = [vp, ctypes.POINTER(lay.AgarLayout)]
    lib.agar_num_envs.argtypes = [vp]
    lib.agar_reset.argtypes = [vp, vp, vp]
    lib.agar_reset_bots.argtypes = [vp, vp, vp]
    lib.agar_observe.argtypes = [vp, vp, vp]
    lib.agar_step.argtypes = [vp, vp, i32, vp]
    lib.agar_step_observe.argtypes = [vp, vp, i32, vp, vp]
    lib.agar_get.argtypes = [vp, i32, vp, vp]
    lib.agar_debug_dump.argtypes = [vp, i32, vp, ctypes.c_size_t, vp]
    lib.agar_debug_load.argtypes = [vp, i32, vp, ctypes.c_size_t, vp]
    lib.agar_launch_count.argtypes = [vp]
    lib.agar_launch_count.restype = ctypes.c_int64
    lib.agar_step_host.argtypes = [vp, vp, i32, vp, vp, vp, vp]
    lib.agar_step_host_begin.argtypes = [vp, vp, i32, vp, vp]
    lib.agar_step_host_end.argtypes = [vp, vp, vp, vp]
    lib.agar_rollout_random.argtypes = [vp, i32, i32, u32, vp, vp]
    lib.agar_set_tile_width.argtypes = [vp, i32]
    lib.agar_get_tile_width.argtypes = [vp]
    lib.agar_state_ptr.argtypes = [vp]
    lib.agar_state_ptr.restype = vp
    for name in EXPORTS:
        getattr(lib, name)
    _lib = lib
    return lib


class AgarError(RuntimeError):
    pass


_GET_DTYPES = {lay.GET_REWARD: "float32", lay.GET_DONE: "uint8", lay.GET_VALID: "uint8", lay.GET_NEED_ACTION: "uint8",
               lay.GET_MASS: "float32", lay.GET_FOV: "float32", lay.GET_NCELLS: "int32", lay.GET_ALIVE: "uint8",
               lay.GET_STATS: "float64", lay.GET_OVERFLOW: "uint32", lay.GET_EVENT_HASH: "uint64"}


class AgarBatch(object):
    """E lock-stepped agar.io envs on one GPU.  All device work is enqueued on torch's current stream."""

    def __init__(self, cfg, n_envs, device=0, seed=0, first_env_id=0, tile_width=None, stream=None):
        """stream: a torch.cuda.Stream every call of this handle is enqueued on (default: torch's current stream at call time).
        Several handles on their own streams step concurrently — the env groups of a host-side pipeline (step_host_begin / _end)."""
        import torch
        if not torch.cuda.is_available():
            raise AgarError("no CUDA device: the agar.io step has no CPU fallback")
        self.torch = torch
        self.lib = load_library()
        self.cfg = cfg
        self.n_envs = int(n_envs)
        self.device = torch.device("cuda", device)
        self.stream = stream
        self.h = ctypes.c_void_p()
        with torch.cuda.device(self.device):
            rc = self.lib.agar_create(ctypes.byref(cfg), self.n_envs, self.device.index, seed, first_env_id,
                                      self._stream(), ctypes.byref(self.h))
        if rc != 0:
            raise AgarError("agar_create failed (%d): %s" % (rc, self.lib.agar_last_error(None).decode()))
        self.layout = lay.AgarLayout()
        self.lib.agar_get_layout(self.h, ctypes.byref(self.layout))
        if tile_width:
            self._check(self.lib.agar_set_tile_width(self.h, int(tile_width)))
        a, L = self.layout.n_agents, self.layout.state_len
        # caller-owned I/O buffers: plain torch tensors (zero-copy for any torch consumer, DLPack for others)
        self.obs = torch.zeros((self.n_envs, max(a, 1), L), dtype=torch.float32, device=self.device)
        self.actions = torch.zeros((self.n_envs, max(a, 1), 4), dtype=torch.float32, device=self.device)

    # ---- plumbing
    def _stream(self):
        if self.stream is not None:
            return ctypes.c_void_p(self.stream.cuda_stream)
        return ctypes.c_void_p(self.torch.cuda.current_stream(self.device).cuda_stream)

    def _check(self, rc):
        if rc != 0:
            raise AgarError("agar call failed (%d): %s" % (rc, self.lib.agar_last_error(self.h).decode()))

    def close(self):
        if getattr(self, "h", None) and self.h.value:
            self.lib.agar_destroy(self.h)
            self.h = ctypes.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def tile_width(self):
        return self.lib.agar_get_tile_width(self.h)

    def set_tile_width(self, w):
        self._check(self.lib.agar_set_tile_width(self.h, int(w)))

    @property
    def launch_count(self):
        return int(self.lib.agar_launch_count(self.h))

    @property
    def observer_launch_count(self):
        """Launches whose decision observations observer warps encoded (not in EXPORTS: older builds load for A/B runs)."""
        fn = self.lib.agar_observer_launch_count
        fn.argtypes, fn.restype = [ctypes.c_void_p], ctypes.c_int64
        return int(fn(self.h))

    def _ptr(self, t):
        return ctypes.c_void_p(t.data_ptr()) if t is not None else ctypes.c_void_p()

    def _actions(self, actions):
        if actions is None:
            return self.actions
        t = self.torch.as_tensor(actions, dtype=self.torch.float32, device=self.device)
        t = t.reshape(self.n_envs, max(self.layout.n_agents, 1), 4).contiguous()
        return t

    # ---- the env surface
    def reset(self, mask=None):
        """Model.resetModel() (model.py:96-98) for all envs or those with mask != 0."""
        m = None if mask is None else self.torch.as_tensor(mask, dtype=self.torch.uint8, device=self.device).contiguous()
        self._check(self.lib.agar_reset(self.h, self._ptr(m), self._stream()))

    def reset_bots(self, mask=None):
        m = None if mask is None else self.torch.as_tensor(mask, dtype=self.torch.uint8, device=self.device).contiguous()
        self._check(self.lib.agar_reset_bots(self.h, self._ptr(m), self._stream()))

    def observe(self, out=None):
        """First half of every NN bot's turn; returns the [E, A, L] float32 observation tensor."""
        out = self.obs if out is None else out
        self._check(self.lib.agar_observe(self.h, self._ptr(out), self._stream()))
        return out

    def step(self, actions=None, n_frames=1):
        a = self._actions(actions)
        self._check(self.lib.agar_step(self.h, self._ptr(a), int(n_frames), self._stream()))

    def step_observe(self, actions=None, n_frames=1, out=None):
        a = self._actions(actions)
        out = self.obs if out is None else out
        self._check(self.lib.agar_step_observe(self.h, self._ptr(a), int(n_frames), self._ptr(out), self._stream()))
        return out

    def rollout_random(self, n_decisions, n_frames=None, decision_base=0, out=None, write_obs=True):
        n_frames = self.cfg.frame_skip + 1 if n_frames is None else n_frames
        out = (self.obs if out is None else out) if write_obs else None
        self._check(self.lib.agar_rollout_random(self.h, int(n_decisions), int(n_frames), int(decision_base),
                                                 self._ptr(out), self._stream()))
        return out

    def get(self, which):
        per_env = which in (lay.GET_OVERFLOW, lay.GET_EVENT_HASH)
        a = max(self.layout.n_agents, 1)
        shape = (self.n_envs,) if per_env else ((self.n_envs, a, 4) if which == lay.GET_STATS else (self.n_envs, a))
        if _GET_DTYPES[which] in ("uint32", "uint64"):  # torch lacks some unsigned dtypes on older builds
            dt = {"uint32": self.torch.int32, "uint64": self.torch.int64}[_GET_DTYPES[which]]
        else:
            dt = getattr(self.torch, _GET_DTYPES[which])
        out = self.torch.zeros(shape, dtype=dt, device=self.device)
        self._check(self.lib.agar_get(self.h, int(which), self._ptr(out), self._stream()))
        return out

    def obs_dlpack(self):
        """The observation buffer as a DLPack capsule (zero copy)."""
        return self.torch.utils.dlpack.to_dlpack(self.obs)

    def step_host(self, actions_np, n_frames, obs_out, reward_out, done_out):
        """Host-buffer path (agar_step_host): numpy in, numpy out, copies included."""
        a = np.ascontiguousarray(actions_np, dtype=np.float32)
        self._check(self.lib.agar_step_host(self.h, a.ctypes.data, int(n_frames), obs_out.ctypes.data,
                                            reward_out.ctypes.data, done_out.ctypes.data, self._stream()))

    def step_host_begin(self, actions_np, n_frames, obs_out):
        """First half of step_host: enqueue on torch's current stream and return (buffers must stay alive and unchanged
        until step_host_end)."""
        a = np.ascontiguousarray(actions_np, dtype=np.float32)
        self._pending = (a, obs_out)
        self._check(self.lib.agar_step_host_begin(self.h, a.ctypes.data, int(n_frames), obs_out.ctypes.data, self._stream()))

    def step_host_end(self, reward_out, done_out):
        self._check(self.lib.agar_step_host_end(self.h, reward_out.ctypes.data, done_out.ctypes.data, self._stream()))
        self._pending = None

    # the same two calls on raw host addresses (ints), for loops that reuse pinned buffers and do not want numpy's
    # ctypes conversion on every call; the caller keeps the buffers alive
    def step_host_begin_ptr(self, actions_addr, n_frames, obs_addr):
        rc = self.lib.agar_step_host_begin(self.h, actions_addr, n_frames, obs_addr,
                                           self.stream.cuda_stream if self.stream is not None else self._stream())
        if rc != 0:
            self._check(rc)

    def step_host_end_ptr(self, reward_addr, done_addr):
        rc = self.lib.agar_step_host_end(self.h, reward_addr, done_addr,
                                         self.stream.cuda_stream if self.stream is not None else self._stream())
        if rc != 0:
            self._check(rc)

    # ---- parity / debugging
    def dump(self, env_index):
        buf = np.zeros(int(self.layout.record_bytes), dtype=np.uint8)
        self._check(self.lib.agar_debug_dump(self.h, int(env_index), buf.ctypes.data, buf.nbytes, self._stream()))
        return lay.Record(self.layout, buf)

    def load(self, env_index, rec):
        buf = np.ascontiguousarray(rec.buf if isinstance(rec, lay.Record) else rec, dtype=np.uint8)
        self._check(self.lib.agar_debug_load(self.h, int(env_index), buf.ctypes.data, buf.nbytes, self._stream()))

    def state_tensor(self):
        """All env records as one uint8 tensor view [E, record_bytes] (zero copy, for checksums)."""
        n = self.n_envs * int(self.layout.record_bytes)
        ptr = self.lib.agar_state_ptr(self.h)

        class _Holder(object):
            pass

        h = _Holder()
        h.__cuda_array_interface__ = {"shape": (n,), "typestr": "|u1", "data": (ptr, False), "version": 2}
        return self.torch.as_tensor(h, device=self.device).view(self.n_envs, int(self.layout.record_bytes))


class BatchedModel(object):
    """Mirror of the reference's Model for E envs (src/model/model.py:90-120): same method names and call
    order — bots act on the pre-step world, then the world steps."""

    def __init__(self, parameters, n_envs, device=0, seed=0, first_env_id=0):
        self.parameters = parameters
        self.batch = AgarBatch(parameters, n_envs, device=device, seed=seed, first_env_id=first_env_id)

    def initialize(self):  # Model.initialize: done by agar_create
        return self

    def resetModel(self):
        self.batch.reset()

    def resetBots(self):
        self.batch.reset_bots()

    def getStateRepresentation(self):  # Bot.getStateRepresentation for every NN bot (bot.py:272-299)
        return self.batch.observe()

    def update(self, actions=None):  # Model.update (model.py:100-112): takeBotActions, then field.update
        self.batch.observe()
        self.batch.step(actions, 1)

    def getLastReward(self):  # Bot.getLastReward (bot.py:645)
        return self.batch.get(lay.GET_REWARD)

    def getIsAlive(self):  # Player.getIsAlive (player.py:180)
        return self.batch.get(lay.GET_ALIVE)

    def getTotalMass(self):  # Player.getTotalMass (player.py:129)
        return self.batch.get(lay.GET_MASS)
