"""Recorded rollouts (agar_rollout, AgarBatch.rollout, GpuReplayBuffer.add_trajectory): every field of every decision equals
the per-decision path (observe + agar_get + a one-decision rollout_random) and the portable-math oracle, bit for bit, on
every kernel path; observation tensors are prefilled with NaN so that rows the call must leave untouched are checked too."""
import ctypes

import numpy as np
import pytest

import aigar_b200.layout as lay
from aigar_b200 import env as agar_env
from aigar_b200.replay import trajectory_transitions

gpu = pytest.mark.gpu

CFG_1V1 = dict(num_nn=1, num_greedy=1, virus=True, split=True, eject=True)
CFG_ARENA = dict(num_nn=4, num_greedy=4, virus=True, split=True, eject=True)
CFG_G42 = dict(grid=42, overrides={"use_fovsize": 0, "use_totalmass": 0})
TURN = ("reward", "done", "valid", "need_action")
GETS = {"reward": lay.GET_REWARD, "done": lay.GET_DONE, "valid": lay.GET_VALID, "need_action": lay.GET_NEED_ACTION}


@pytest.fixture(scope="module")
def torch_cuda():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("these tests need a GPU (the product has no CPU fallback; run with -m gpu on the B200 box)")
    return torch


def _batch(cfg, n, **kw):
    return agar_env.AgarBatch(cfg, n, **kw)


def _same(x, y):
    """bit equality (NaN sentinels included)"""
    import torch
    if x.dtype == torch.float32:
        x, y = x.view(torch.int32), y.view(torch.int32)
    return torch.equal(x, y)


def _nan_trajectory(b, D, fields=agar_env.TRAJECTORY_FIELDS):
    t = agar_env.Trajectory.allocate(b, D, fields)
    if t.obs is not None:
        t.obs.fill_(float("nan"))
    return t


def _per_decision(b, D, F, base, actions=None):
    """D x (observe into a NaN row buffer, the four agar_get fields, a one-decision step), then the trailing observe"""
    torch = b.torch
    rows, turn = [], {f: [] for f in TURN}
    buf = torch.empty_like(b.obs)
    for d in range(D + 1):
        buf.fill_(float("nan"))
        b.observe(out=buf)
        rows.append(buf.clone())
        for f in TURN:
            turn[f].append(b.get(GETS[f]))
        if d == D:
            break
        if actions is None:
            b.rollout_random(1, F, base + d, write_obs=False)
        else:
            b.step(actions[d], F)
    return torch.stack(rows), {f: torch.stack(v) for f, v in turn.items()}


def _philox_actions(seed, first, D, E, A, base):
    from oracle.philox import philox4x32
    out = np.zeros((D, E, A, 4), dtype=np.float32)
    for d in range(D):
        for e in range(E):
            for a in range(A):
                w = philox4x32((base + d) & 0xFFFFFFFF, 7, first + e, a, seed & 0xFFFFFFFF, seed >> 32)
                out[d, e, a] = [np.float32(x >> 8) * np.float32(1.0 / 16777216.0) for x in w]
    return out


# (name, config kwargs, envs, tile width, decisions, frames per decision, expect the observer launch)
PER_DECISION = [
    ("k_simple W=1", {}, 70, 1, 6, 8, False),
    ("k_simple W=2", {}, 70, 2, 6, 8, False),
    ("k_simple W=4 observers", {}, 70, 4, 6, 8, True),
    ("k_simple W=8 observers", {}, 70, 8, 6, 8, True),
    ("k_simple W=16", {}, 70, 16, 6, 8, False),
    ("k_simple W=32", {}, 70, 32, 6, 8, False),
    ("k_simple W=8 F=3 inline", {}, 70, 8, 9, 3, False),
    ("k_simple W=8 F=5 misaligned", {}, 70, 8, 7, 5, True),
    ("k_simple W=2 F=5 misaligned", {}, 40, 2, 7, 5, False),
    ("k_simple W=8 F=0", {}, 20, 8, 3, 0, False),
    ("1-vs-greedy", CFG_1V1, 16, None, 5, 8, False),
    ("1-vs-greedy F=3 misaligned", CFG_1V1, 16, None, 6, 3, False),
    ("1-vs-greedy F=0", CFG_1V1, 8, None, 3, 0, False),
    ("arena", CFG_ARENA, 6, None, 4, 4, False),
    ("G=42 general kernel", CFG_G42, 16, None, 5, 4, False),
]


@gpu
@pytest.mark.parametrize("name,kw,n,tile,D,F,observers", PER_DECISION, ids=[c[0] for c in PER_DECISION])
def test_rollout_equals_per_decision_path(torch_cuda, name, kw, n, tile, D, F, observers):
    torch = torch_cuda
    cfg = lay.derive_config(**kw)
    seed, first, base = 5, 40, 17
    a = _batch(cfg, n, seed=seed, first_env_id=first, tile_width=tile)
    c = _batch(cfg, n, seed=seed, first_env_id=first, tile_width=tile)
    for b in (a, c):
        b.rollout_random(3, 8, 0)
    n_obs, n_launch = a.observer_launch_count, a.launch_count
    traj = a.rollout(D, F, base, out=_nan_trajectory(a, D))
    assert a.launch_count == n_launch + 1
    assert (a.observer_launch_count > n_obs) == observers, name
    rows, turn = _per_decision(c, D, F, base)
    assert _same(traj.obs, rows), name
    for f in TURN:
        assert torch.equal(getattr(traj, f), turn[f]), "%s: %s" % (name, f)
    assert torch.equal(a.state_tensor(), c.state_tensor()), name
    A = max(a.layout.n_agents, 1)
    assert np.array_equal(traj.action.cpu().numpy(), _philox_actions(seed, first, D, n, A, base)), name
    assert traj.n_frames == F and traj.frame_skip == cfg.frame_skip


ORACLE = [("configs[1] W=8", {}, 70, 8), ("configs[1] W=1", {}, 70, 1), ("1-vs-greedy", CFG_1V1, 12, None)]


@gpu
@pytest.mark.parametrize("name,kw,n,tile", ORACLE, ids=[c[0] for c in ORACLE])
def test_rollout_equals_oracle(torch_cuda, name, kw, n, tile):
    from oracle import oracle as orc
    cfg = lay.derive_config(**kw)
    seed, first, base, D, F = 9, 300, 4, 12, 8
    b = _batch(cfg, n, seed=seed, first_env_id=first, tile_width=tile)
    traj = b.rollout(D, F, base, out=_nan_trajectory(b, D))
    obs = traj.obs.cpu().numpy()
    turn = {f: getattr(traj, f).cpu().numpy() for f in TURN}
    st = b.state_tensor().cpu().numpy()
    for e in range(n):
        ora = orc.OracleEnv(cfg, seed=seed, env_id=first + e, portable=True)
        for d in range(D + 1):
            t = ora.observe()
            for a, ta in enumerate(t):
                where = "%s env %d decision %d agent %d" % (name, e, d, a)
                if ta["need_action"]:
                    assert np.array_equal(obs[d, e, a], ta["obs32"]), where
                else:
                    assert np.isnan(obs[d, e, a]).all(), where
                assert turn["reward"][d, e, a] == np.float32(ta["reward"]), where
                assert (turn["done"][d, e, a], turn["valid"][d, e, a], turn["need_action"][d, e, a]) == \
                    (ta["done"], ta["valid"], ta["need_action"]), where
            if d < D:
                ora.rollout_random(1, F, base + d)
        diff = lay.compare_records(ora.record, lay.Record(b.layout, st[e].copy()), what="%s env %d " % (name, e))
        assert not diff, diff


REPLAY = [("k_simple W=8", {}, 64, 8), ("1-vs-greedy", CFG_1V1, 16, None)]


@gpu
@pytest.mark.parametrize("name,kw,n,tile", REPLAY, ids=[c[0] for c in REPLAY])
def test_recorded_actions_replay_the_run(torch_cuda, name, kw, n, tile):
    """snapshot, record a random-driver rollout, restore, roll out the recorded actions: the same trajectory and records,
    which also equal D x (observe, step) with those actions"""
    torch = torch_cuda
    cfg = lay.derive_config(**kw)
    D, F = 10, 8
    b = _batch(cfg, n, seed=3, first_env_id=11, tile_width=tile)
    c = _batch(cfg, n, seed=3, first_env_id=11, tile_width=tile)
    b.rollout_random(2, 8, 0)
    bank = b.snapshot()
    c.restore(bank)
    first = b.rollout(D, F, 50, out=_nan_trajectory(b, D))
    end = b.state_tensor().clone()
    b.restore(bank)
    n_launch = b.launch_count
    second = b.rollout(D, F, 0, actions=first.action, out=_nan_trajectory(b, D, [f for f in agar_env.TRAJECTORY_FIELDS
                                                                                 if f != "action"]))
    assert b.launch_count == n_launch + 1
    assert second.action is first.action
    assert _same(first.obs, second.obs)
    for f in TURN:
        assert torch.equal(getattr(first, f), getattr(second, f)), f
    assert torch.equal(b.state_tensor(), end)
    rows, turn = _per_decision(c, D, F, 0, actions=first.action)
    assert _same(second.obs, rows)
    for f in TURN:
        assert torch.equal(getattr(second, f), turn[f]), f
    assert torch.equal(c.state_tensor(), end)


@gpu
def test_bench_shape_on_observer_warps(torch_cuda):
    """4096 envs x 125 decisions x 8 frames at the default tile width (observer warps) == the same rollout at 2 lanes per
    env (inline encoder); the records == rollout_random + observe"""
    torch = torch_cuda
    cfg = lay.derive_config()
    a, c, r = (_batch(cfg, 4096, seed=2026, tile_width=w) for w in (None, 2, None))
    assert a.tile_width == 8
    ta = a.rollout(125, 8, 0, out=_nan_trajectory(a, 125))
    tc = c.rollout(125, 8, 0, out=_nan_trajectory(c, 125))
    assert a.observer_launch_count == 1 and c.observer_launch_count == 0
    for f in agar_env.TRAJECTORY_FIELDS:
        assert _same(getattr(ta, f), getattr(tc, f)), f
    r.rollout_random(125, 8, 0)
    r.observe()
    assert torch.equal(a.state_tensor(), r.state_tensor()) and torch.equal(c.state_tensor(), r.state_tensor())


@gpu
def test_trajectory_larger_than_4_gib(torch_cuda):
    torch = torch_cuda
    cfg = lay.derive_config()
    n, D, F = 65536, 140, 8
    a, c = _batch(cfg, n, seed=8), _batch(cfg, n, seed=8)
    traj = a.rollout(D, F, 0, out=_nan_trajectory(a, D, ("obs", "action", "reward", "need_action")))
    assert traj.obs.numel() * 4 > 2 ** 32
    sampled = {0, 1, 69, D - 1, D}
    buf = torch.empty_like(c.obs)
    for d in range(D + 1):
        if d in sampled:
            buf.fill_(float("nan"))
            c.observe(out=buf)
            assert _same(traj.obs[d], buf), d
            assert _same(traj.obs[d, n - 1], buf[n - 1]), d
            assert torch.equal(traj.reward[d], c.get(lay.GET_REWARD)), d
            assert torch.equal(traj.need_action[d], c.get(lay.GET_NEED_ACTION)), d
        if d < D:
            c.rollout_random(1, F, d, write_obs=False)
    c.observe()
    assert torch.equal(a.state_tensor(), c.state_tensor())
    last = _philox_actions(a.seed, a.first_env_id + n - 1, 1, 1, 1, D - 1)[0, 0, 0]
    assert np.array_equal(traj.action[D - 1, n - 1, 0].cpu().numpy(), last)


@gpu
def test_restore_and_rollout_in_a_cuda_graph(torch_cuda):
    torch = torch_cuda
    cfg = lay.derive_config()
    b = _batch(cfg, 512, seed=12)
    b.rollout_random(4, 8, 0)
    bank = b.snapshot()
    out = agar_env.Trajectory.allocate(b, 6)
    for _ in range(2):  # warm up outside the capture
        b.restore(bank)
        b.rollout(6, 8, 0, out=out)
    ref = [t.clone() for t in out[:6]]
    for t in out[:6]:
        t.zero_()
    graph = torch.cuda.CUDAGraph()
    n0 = b.launch_count
    with torch.cuda.graph(graph):
        b.restore(bank)
        b.rollout(6, 8, 0, out=out)
    assert b.launch_count == n0 + 2
    for _ in range(2):
        graph.replay()
        torch.cuda.synchronize()
        for x, y in zip(ref, out[:6]):
            assert torch.equal(x, y)


@gpu
def test_host_refusals(torch_cuda):
    torch = torch_cuda
    b = _batch(lay.derive_config(), 8, seed=1)
    fn = b._lazy("agar_rollout", [ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_uint32, ctypes.c_void_p,
                                  ctypes.POINTER(agar_env._CTrajectory), ctypes.c_void_p])
    t = agar_env.Trajectory.allocate(b, 2)
    act = torch.zeros((2, 8, 1, 4), device=b.device)
    raw = torch.zeros(4096, dtype=torch.uint8, device=b.device)

    def call(D, F, actions, traj):
        st = b.state_tensor().clone()
        n = b.launch_count
        rc = fn(b.h, D, F, 0, actions, traj, b._stream())
        torch.cuda.synchronize()
        assert b.launch_count == n and torch.equal(st, b.state_tensor())
        return rc, b.lib.agar_last_error(b.h).decode()

    def ctraj(**kw):
        return ctypes.byref(agar_env._CTrajectory(**kw))
    cases = [
        (2, 8, None, None, "out is NULL"),
        (-1, 8, None, ctraj(), "negative"),
        (2, -1, None, ctraj(), "negative"),
        (2, 8, act.data_ptr(), ctraj(action=t.action.data_ptr()), "caller actions"),
        (2, 8, None, ctraj(obs=raw.data_ptr() + 2), "aligned"),
        (2, 8, raw.data_ptr() + 1, ctraj(), "aligned"),
    ]
    for D, F, actions, traj, msg in cases:
        rc, err = call(D, F, actions, traj)
        assert rc == -1, (msg, rc)  # AGAR_E_INVALID
        assert msg in err, (msg, err)
    with pytest.raises(agar_env.AgarError, match="caller actions"):
        b.rollout(2, 8, 0, actions=act, out=t)
    with pytest.raises(ValueError, match="out.obs"):
        b.rollout(3, 8, 0, out=t)


@gpu
@pytest.mark.parametrize("prioritized", [False, True])
def test_add_trajectory_equals_add_batch_per_decision(torch_cuda, prioritized):
    torch = torch_cuda
    from aigar_b200.replay import GpuReplayBuffer
    b = _batch(lay.derive_config(), 64, seed=6)
    L = b.layout.state_len
    for size, D in ((5000, 6), (300, 9)):  # the second trajectory (576 transitions) wraps the 300-slot ring
        one = GpuReplayBuffer(size, L, 2, prioritized)
        many = GpuReplayBuffer(size, L, 2, prioritized)
        traj = b.rollout(D)
        one.add_trajectory(traj)
        for d in range(D):
            many.add_batch(traj.obs[d], traj.action[d], traj.reward[d + 1], traj.obs[d + 1], traj.done[d + 1],
                           traj.valid[d + 1])
        assert (len(one), one.next_idx) == (len(many), many.next_idx)
        idx = torch.arange(len(one), dtype=torch.int32, device=b.device)
        for x, y in zip(one.gather(idx), many.gather(idx)):
            assert torch.equal(x, y)
        g = torch.Generator(device=b.device).manual_seed(3)
        u = torch.rand(4096, dtype=torch.float64, device=b.device, generator=g)
        for x, y in zip(one.sample(u), many.sample(u)):  # the prioritized sample reads both segment trees
            assert torch.equal(x, y)
        assert one.error_flags == 0 == many.error_flags
    with pytest.raises(ValueError, match="one bot turn per decision"):
        one.add_trajectory(b.rollout(2, 3))


# ---- no device needed

def test_trajectory_shapes_and_transition_slices():
    import torch
    sh = agar_env.Trajectory.shapes(5, 7, 0, 123)
    assert sh == {"obs": ((6, 7, 1, 123), "float32"), "action": ((5, 7, 1, 4), "float32"), "reward": ((6, 7, 1), "float32"),
                  "done": ((6, 7, 1), "uint8"), "valid": ((6, 7, 1), "uint8"), "need_action": ((6, 7, 1), "uint8")}
    assert agar_env.Trajectory.shapes(2, 3, 4, 10)["obs"][0] == (3, 3, 4, 10)
    t = {f: torch.arange(int(np.prod(s)), dtype=getattr(torch, dt)).reshape(s) for f, (s, dt) in
         agar_env.Trajectory.shapes(4, 3, 2, 6).items()}
    traj = agar_env.Trajectory(n_frames=8, frame_skip=7, **t)
    o, a, r, o2, d, v = trajectory_transitions(traj)
    assert torch.equal(o, t["obs"][:4]) and torch.equal(o2, t["obs"][1:]) and a is t["action"]
    assert torch.equal(r, t["reward"][1:]) and torch.equal(d, t["done"][1:]) and torch.equal(v, t["valid"][1:])
    assert all(x.is_contiguous() for x in (o, a, r, o2, d, v))
    assert o.data_ptr() == t["obs"].data_ptr() and o2.data_ptr() == t["obs"][1].data_ptr()

    class StandIn(object):
        def add_batch(self, *args):
            self.args = args
    from aigar_b200.replay import GpuReplayBuffer
    s = StandIn()
    GpuReplayBuffer.add_trajectory(s, traj)
    assert all(x is y or torch.equal(x, y) for x, y in zip(s.args, (o, a, r, o2, d, v)))
    for bad in (traj._replace(n_frames=3), traj._replace(n_frames=None)):
        with pytest.raises(ValueError, match="one bot turn per decision"):
            trajectory_transitions(bad)
    with pytest.raises(ValueError, match="action"):
        trajectory_transitions(traj._replace(action=None))
