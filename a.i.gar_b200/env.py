"""Host side of the batched agar.io env: a thin ctypes binding of include/agar_b200.h plus the mirror of the
reference's Model / Bot surface (src/model/model.py:90-120, src/model/bot.py:252-299,645).

PyTorch is used for device memory, streams and DLPack only.  There is NO CPU fallback: if libagar_b200.so is
missing or no CUDA device is present every constructor raises."""
import ctypes
import hashlib
import os
from collections import namedtuple

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


def bind_lazy(lib, name, argtypes, restype=ctypes.c_int):
    """A C function bound on first use (not in EXPORTS: older builds load for A/B runs)."""
    fn = getattr(lib, name)
    fn.argtypes, fn.restype = argtypes, restype
    return fn


class AgarError(RuntimeError):
    pass


class CheckpointError(AgarError):
    """A checkpoint file that does not match the handle it is loaded into (the message names the field)."""


CHECKPOINT_FORMAT = "agar_b200.records.v1"
_CHECKPOINT_KEYS = ("format", "abi_version", "config", "layout", "n_envs", "seed", "first_env_id", "records", "sha256")


def _struct_bytes(s):
    return np.frombuffer(bytes(s), dtype=np.uint8).copy()


def save_npz_checkpoint(path, fmt, payload, **fields):
    """Write a checkpoint .npz (no pickled objects): a format tag, the fields, and `payload` (a uint8 host array, stored under
    that name) with its SHA-256."""
    arr = np.ascontiguousarray(fields[payload], dtype=np.uint8)
    fields[payload] = arr
    with open(path, "wb") as f:  # a file object: numpy would otherwise append ".npz" to the name
        np.savez(f, format=np.array(fmt), sha256=np.array(hashlib.sha256(arr.tobytes()).hexdigest()), **fields)


def load_npz_checkpoint(path, fmt, keys, kind):
    """The fields `keys` of a checkpoint .npz, read without pickles.  Raises CheckpointError for a file that lacks one of
    them (naming it a `kind` checkpoint) or has another format tag."""
    with np.load(path, allow_pickle=False) as z:
        missing = [k for k in keys if k not in z.files]
        if missing:
            raise CheckpointError("%s: not a %s checkpoint (missing %s)" % (path, kind, ", ".join(missing)))
        ck = {k: z[k] for k in keys}
    if str(ck["format"]) != fmt:
        raise CheckpointError("%s: format %r, expected %r" % (path, str(ck["format"]), fmt))
    return ck


def check_npz_digest(path, ck, payload):
    if hashlib.sha256(np.ascontiguousarray(ck[payload]).tobytes()).hexdigest() != str(ck["sha256"]):
        raise CheckpointError("%s: sha256 of the %s does not match the stored digest" % (path, payload))


def write_checkpoint(path, cfg, layout, n_envs, seed, first_env_id, records):
    """Write a batch checkpoint (.npz, no pickled objects).  records: uint8 [n_envs, record_bytes] host array."""
    save_npz_checkpoint(path, CHECKPOINT_FORMAT, "records", abi_version=np.int64(lay.ABI_VERSION),
                        config=_struct_bytes(cfg), layout=_struct_bytes(layout), n_envs=np.int64(n_envs),
                        seed=np.uint64(seed), first_env_id=np.uint64(first_env_id), records=records)


def read_checkpoint(path):
    """Parse a checkpoint file without a device: a dict of its fields.  Raises CheckpointError for a file that is not a
    checkpoint of this format and ABI version, whose records are not [n_envs, record_bytes] uint8, or whose digest differs."""
    ck = load_npz_checkpoint(path, CHECKPOINT_FORMAT, _CHECKPOINT_KEYS, "records")
    if int(ck["abi_version"]) != lay.ABI_VERSION:
        raise CheckpointError("%s: abi_version %d, this library has %d" % (path, int(ck["abi_version"]), lay.ABI_VERSION))
    for name, struct in (("config", lay.AgarConfig), ("layout", lay.AgarLayout)):
        if ck[name].dtype != np.uint8 or ck[name].nbytes != ctypes.sizeof(struct):
            raise CheckpointError("%s: %s is not the bytes of an %s" % (path, name, struct.__name__))
    rec, rb = ck["records"], int(lay.AgarLayout.from_buffer_copy(ck["layout"].tobytes()).record_bytes)
    if rec.dtype != np.uint8 or rec.ndim != 2 or rec.shape != (int(ck["n_envs"]), rb):
        raise CheckpointError("%s: records of shape %s / %s do not match n_envs and the layout's record_bytes"
                              % (path, rec.shape, rec.dtype))
    check_npz_digest(path, ck, "records")
    return ck


def check_checkpoint(ck, cfg, layout, n_envs, seed, first_env_id):
    """Raise CheckpointError naming the first field of a parsed checkpoint that differs from a handle's."""
    want = (("config", _struct_bytes(cfg)), ("layout", _struct_bytes(layout)))
    for name, mine in want:
        if not np.array_equal(ck[name], mine):
            raise CheckpointError("checkpoint %s bytes differ from the handle's" % name)
    for name, mine in (("n_envs", n_envs), ("seed", seed), ("first_env_id", first_env_id)):
        if int(ck[name]) != int(mine):
            raise CheckpointError("checkpoint %s is %d, the handle's is %d" % (name, int(ck[name]), int(mine)))


TRAJECTORY_FIELDS = ("obs", "action", "reward", "done", "valid", "need_action")


class _CTrajectory(ctypes.Structure):
    """AgarTrajectory of include/agar_b200.h: one nullable device pointer per field"""
    _fields_ = [(f, ctypes.c_void_p) for f in TRAJECTORY_FIELDS]


class Trajectory(namedtuple("Trajectory", TRAJECTORY_FIELDS + ("n_frames", "frame_skip"))):
    """A recorded rollout (AgarBatch.rollout): device tensors, A = max(n_agents, 1), D decisions.

    obs [D+1, E, A, L] float32, action [D, E, A, 4] float32, reward [D+1, E, A] float32, done / valid / need_action
    [D+1, E, A] uint8.  Row d < D holds what decision d observed (and, for action, what it did); row D the trailing
    observation.  The turn fields are what agar_get returns right after that observation.  Observation rows of skipping or
    dead agents are not written: they keep what the tensor held (zeros in a fresh allocation).  A field that is None is not
    recorded.  n_frames: frames per decision of the rollout that filled it (None before one has); frame_skip: the config's."""
    __slots__ = ()

    @staticmethod
    def shapes(n_decisions, n_envs, n_agents, state_len):
        """{field: (shape, dtype name)} of a D-decision trajectory (no device needed)"""
        D, E, A, L = int(n_decisions), int(n_envs), max(int(n_agents), 1), int(state_len)
        turn = ((D + 1, E, A), "uint8")
        return {"obs": ((D + 1, E, A, L), "float32"), "action": ((D, E, A, 4), "float32"),
                "reward": ((D + 1, E, A), "float32"), "done": turn, "valid": turn, "need_action": turn}

    @classmethod
    def allocate(cls, batch, n_decisions, fields=TRAJECTORY_FIELDS):
        """Zeroed tensors for the named fields on the batch's device, None for the others: reusable through
        AgarBatch.rollout(out=...), for instance inside a CUDA graph."""
        unknown = set(fields) - set(TRAJECTORY_FIELDS)
        if unknown:
            raise ValueError("unknown trajectory fields %s (known: %s)" % (sorted(unknown), ", ".join(TRAJECTORY_FIELDS)))
        torch = batch.torch
        sh = cls.shapes(n_decisions, batch.n_envs, batch.layout.n_agents, batch.layout.state_len)
        t = {f: torch.zeros(sh[f][0], dtype=getattr(torch, sh[f][1]), device=batch.device) if f in fields else None
             for f in TRAJECTORY_FIELDS}
        return cls(n_frames=None, frame_skip=int(batch.cfg.frame_skip), **t)


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
        self.seed, self.first_env_id = int(seed), int(first_env_id)  # the Philox key of slot e: (seed, first_env_id + e)
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

    def _lazy(self, name, argtypes, restype=ctypes.c_int):
        return bind_lazy(self.lib, name, argtypes, restype)

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

    def rollout(self, n_decisions, n_frames=None, decision_base=0, actions=None, out=None):
        """agar_rollout: n_decisions x (observe -> act -> n_frames frames) and a trailing observation in one launch, every
        decision recorded.  actions: [D, E, A, 4] caller actions (decision d takes row d), or None for the random driver of
        rollout_random (whose actions are then recorded).  out: a Trajectory to fill (Trajectory.allocate; None fields are not
        recorded; out.action must be None with caller actions), or None for a new one.  Returns the Trajectory, whose
        action is the caller's tensor when actions are given.  The records end as after rollout_random(D, n_frames,
        decision_base) + observe."""
        n_frames = self.cfg.frame_skip + 1 if n_frames is None else int(n_frames)
        D = int(n_decisions)
        act = None
        if actions is not None:
            act = self.torch.as_tensor(actions, dtype=self.torch.float32, device=self.device)
            shape = (D, self.n_envs, max(self.layout.n_agents, 1), 4)
            act = (act if tuple(act.shape) == shape else act.reshape(shape)).contiguous()
        if out is None:
            out = Trajectory.allocate(self, D, [f for f in TRAJECTORY_FIELDS if not (f == "action" and act is not None)])
        sh = Trajectory.shapes(D, self.n_envs, self.layout.n_agents, self.layout.state_len)
        for f in TRAJECTORY_FIELDS:
            t = getattr(out, f)
            if t is not None and not (self.torch.is_tensor(t) and tuple(t.shape) == sh[f][0] and t.device == self.device
                                      and t.dtype == getattr(self.torch, sh[f][1]) and t.is_contiguous()):
                raise ValueError("out.%s must be a contiguous %s tensor %s on %s" % (f, sh[f][1], sh[f][0], self.device))
        c = _CTrajectory(*[getattr(out, f).data_ptr() if getattr(out, f) is not None else None for f in TRAJECTORY_FIELDS])
        fn = self._lazy("agar_rollout", [ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_uint32, ctypes.c_void_p,
                                         ctypes.POINTER(_CTrajectory), ctypes.c_void_p])
        self._check(fn(self.h, D, n_frames, int(decision_base), self._ptr(act), ctypes.byref(c), self._stream()))
        return out._replace(action=act if act is not None else out.action, n_frames=n_frames)

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

    # ---- state snapshots (agar_save_records / agar_load_records)
    def _index(self, idx, n):
        """a device tensor must already be int32 on this device (no copy, graph-capturable); anything else is converted"""
        if self.torch.is_tensor(idx):
            t = idx
        else:
            t = self.torch.as_tensor(np.asarray(idx, dtype=np.int32), device=self.device)
        if t.dtype != self.torch.int32 or t.device != self.device or t.dim() != 1 or (n is not None and t.numel() != n):
            raise ValueError("index must be a 1-D int32 tensor on %s%s" % (self.device, "" if n is None else " of %d entries" % n))
        return t.contiguous()

    def _bank(self, bank):
        rb = int(self.layout.record_bytes)
        if not (self.torch.is_tensor(bank) and bank.dtype == self.torch.uint8 and bank.device == self.device and
                bank.dim() == 2 and bank.shape[1] == rb and bank.is_contiguous()):
            raise ValueError("a bank is a contiguous uint8 tensor [n, %d] on %s" % (rb, self.device))
        return bank

    def snapshot(self, envs=None, out=None):
        """Records of all envs, or of envs[i] for row i (any order, repeats allowed), as a uint8 device tensor
        [n, record_bytes].  out: a bank to write into instead of a new tensor."""
        idx = None if envs is None else self._index(envs, None)
        n = self.n_envs if idx is None else idx.numel()
        if out is None:
            out = self.torch.empty((n, int(self.layout.record_bytes)), dtype=self.torch.uint8, device=self.device)
        out = self._bank(out)
        if out.shape[0] != n:
            raise ValueError("out has %d rows, %d are saved" % (out.shape[0], n))
        fn = self._lazy("agar_save_records", [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p])
        self._check(fn(self.h, self._ptr(out), self._ptr(idx), int(n), self._stream()))
        return out

    def restore(self, bank, index=None):
        """Overwrite env records from a bank: env e takes row index[e] (int32 [n_envs], -1 keeps env e); without an index
        row e.  A record restored into the slot it came from continues bit for bit; one restored into another slot (a
        clone: b.restore(b.snapshot(), index)) continues under that slot's Philox key.  Observation buffers are not
        part of a record.  Rows that fail the device-side checks are not installed (record_error_flags())."""
        bank = self._bank(bank)
        idx = None if index is None else self._index(index, self.n_envs)
        fn = self._lazy("agar_load_records", [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p])
        self._check(fn(self.h, self._ptr(bank), int(bank.shape[0]), self._ptr(idx), self._stream()))

    def record_error_flags(self):
        """Sticky AGAR_REC_ERR_* bits (1: an index out of range, 2: a record refused on load); synchronises the stream."""
        rc = self._lazy("agar_record_error_flags", [ctypes.c_void_p, ctypes.c_void_p])(self.h, self._stream())
        if rc < 0:
            self._check(rc)
        return int(rc)

    def _on_stream(self):
        """torch's copies in stream order with this handle's calls"""
        import contextlib
        return self.torch.cuda.stream(self.stream) if self.stream is not None else contextlib.nullcontext()

    def save_checkpoint(self, path):
        """Write every env record with what a later load must match (config, layout, n_envs, seed, first_env_id)."""
        with self._on_stream():
            records = self.snapshot().cpu().numpy()
        write_checkpoint(path, self.cfg, self.layout, self.n_envs, self.seed, self.first_env_id, records)

    def load_checkpoint(self, path):
        """Restore every env from a checkpoint of a handle with the same config, layout, n_envs, seed and first_env_id.
        A file that differs in any of them, whose digest is wrong, or one of whose records the device-side checks refuse is
        refused (CheckpointError) and the handle's state is left as it was."""
        ck = read_checkpoint(path)
        check_checkpoint(ck, self.cfg, self.layout, self.n_envs, self.seed, self.first_env_id)
        with self._on_stream():
            bank = self.torch.from_numpy(ck["records"]).to(self.device)
            backup = self.snapshot()
            self.restore(bank)
            # an identity load installs every row unless the checks refuse it: compare instead of reading the sticky flags,
            # which an earlier call may have set already
            if not self.torch.equal(self.state_tensor(), bank):
                self.restore(backup)
                raise CheckpointError("%s: records that fail the device-side checks (counts or indices out of range); "
                                      "nothing was loaded" % path)

    @classmethod
    def from_checkpoint(cls, path, device=0, tile_width=None, stream=None):
        """A new handle matching a checkpoint (config, n_envs, seed, first_env_id), loaded from it."""
        ck = read_checkpoint(path)
        cfg = lay.AgarConfig.from_buffer_copy(ck["config"].tobytes())
        b = cls(cfg, int(ck["n_envs"]), device=device, seed=int(ck["seed"]), first_env_id=int(ck["first_env_id"]),
                tile_width=tile_width, stream=stream)
        b.load_checkpoint(path)
        return b

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
