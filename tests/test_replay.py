"""GPU replay buffer (SURVEY §8f rank 1).  CPU: oracle/replay_oracle.py pinned against a recording of the reference's own
ReplayBuffer / PrioritizedReplayBuffer.  GPU: the CUDA buffer against the oracle."""
import numpy as np
import pytest

from oracle.replay_oracle import ReplayOracle


def _transitions(n, L, rng):
    return [(rng.random(L).astype(np.float32), rng.random(4).astype(np.float32), float(np.float32(rng.normal())),
             rng.random(L).astype(np.float32), bool(rng.random() < 0.1)) for _ in range(n)]


@pytest.mark.parametrize("prioritized", [False, True])
def test_oracle_equals_reference_replay_buffer(prioritized):
    """12 rounds of adds, samples from 8 injected uniforms and priority updates: length, next index, every sampled column,
    index and weight, the max priority and both segment trees bit for bit against the recording of the reference's ReplayBuffer /
    PrioritizedReplayBuffer on the same sequence (tests/golden/live/replay_*.npz, tools/gen_golden_live.py)."""
    import gen_golden_live as gl
    from golden_util import live
    z = live("replay_prioritized" if prioritized else "replay_uniform")
    got = gl.record_replay("oracle", prioritized)
    assert np.array_equal(z["states"], got["states"], equal_nan=True)
    assert np.array_equal(z["samples"], got["samples"])


@pytest.mark.gpu
@pytest.mark.parametrize("prioritized,size", [(False, 37), (True, 37), (True, 1000), (False, 64)])
def test_gpu_replay_equals_oracle(prioritized, size):
    import torch
    from aigar_b200.replay import GpuReplayBuffer
    rng = np.random.default_rng(11)
    L = 123
    gpu = GpuReplayBuffer(size, L, 4, prioritized, 0.6, 0.4)
    ora = ReplayOracle(size, prioritized, 0.6, 0.4)
    dev = gpu.device
    for rnd in range(14):
        n = int(rng.integers(5, 3 * size if rnd == 9 else 60))   # round 9 overflows the ring within one batch
        trs = _transitions(n, L, rng)
        valid = rng.random(n) < 0.7
        for tr, v in zip(trs, valid):
            if v:
                ora.add(*tr)
        gpu.add_batch(torch.tensor(np.stack([t[0] for t in trs]), device=dev), torch.tensor(np.stack([t[1] for t in trs]), device=dev),
                      torch.tensor(np.array([t[2] for t in trs], np.float32), device=dev),
                      torch.tensor(np.stack([t[3] for t in trs]), device=dev),
                      torch.tensor(np.array([t[4] for t in trs]), device=dev), torch.tensor(valid, device=dev))
        assert len(gpu) == len(ora) and gpu.next_idx == ora.next_idx
        if len(ora) < 4:
            continue
        u = rng.random(32)
        out_g = gpu.sample(u)
        out_o = ora.sample([float(x) for x in u])
        idx_g = out_g[-1].cpu().numpy()
        assert list(idx_g) == list(out_o[-1])                       # sampled indices: exact
        for a, b in zip(out_g[:5], out_o[:5]):
            assert np.array_equal(a.cpu().numpy().astype(np.asarray(b).dtype), np.asarray(b))
        if prioritized:
            np.testing.assert_allclose(out_g[5].cpu().numpy(), out_o[5], rtol=1e-12)   # pow(): portable vs libm
            pr = np.abs(rng.normal(size=32)) + 1e-4
            gpu.update_priorities(out_g[-1], pr)
            ora.update_priorities(out_o[-1], pr)
    assert gpu.launch_count > 0


@pytest.mark.gpu
def test_replay_fed_by_the_env():
    """Transition assembly on device: (s, a, R, s', done) straight from the env's buffers (bot.py:204-217)."""
    import torch
    import aigar_b200.layout as lay
    from aigar_b200.env import AgarBatch
    from aigar_b200.replay import GpuReplayBuffer
    cfg = lay.derive_config()
    E = 256
    b = AgarBatch(cfg, E, seed=4)
    rp = GpuReplayBuffer(4000, b.layout.state_len, 4)
    obs = b.observe().clone()
    g = torch.Generator(device=b.device).manual_seed(0)
    total = 0
    for t in range(20):
        act = torch.rand((E, 1, 4), device=b.device, generator=g)
        nxt = b.step_observe(act, 8)
        valid, done, rew = b.get(lay.GET_VALID), b.get(lay.GET_DONE), b.get(lay.GET_REWARD)
        rp.add_batch(obs, act, rew, nxt, done, valid)
        total += int(valid.sum().item())
        obs = nxt.clone()
    assert len(rp) == min(total, 4000) and total == 20 * E
    s = rp.sample(np.random.default_rng(0).random(64))
    assert torch.isfinite(s[0]).all() and s[0].shape == (64, b.layout.state_len)


@pytest.mark.gpu
@pytest.mark.parametrize("prioritized", [False, True])
def test_gpu_replay_guards_what_the_reference_raises_on(prioritized):
    """ADVICE r1: sampling an empty or one-element buffer (the reference raises: random.randint(0, -1), unbounded recursion in
    sum(0, len - 1)), indices outside [0, size) and priorities <= 0 (the reference asserts) must neither hang the GPU nor touch
    memory outside the buffer: the kernels return index 0 / weight 0, leave the trees alone and raise a sticky error flag."""
    import torch
    from aigar_b200.replay import GpuReplayBuffer
    L = 8
    rp = GpuReplayBuffer(64, L, 2, prioritized, 0.6, 0.4)
    dev = rp.device
    u = torch.rand(16, dtype=torch.float64, device=dev)
    out = rp.sample(u)                      # empty buffer
    torch.cuda.synchronize()
    assert rp.error_flags & 1 and int(out[-1].max()) == 0
    obs = torch.rand((1, L), device=dev)
    rp.add_batch(obs, torch.rand((1, 2), device=dev), torch.ones(1, device=dev), obs, torch.zeros(1, dtype=torch.uint8, device=dev))
    out = rp.sample(u)                      # one element: fine for the uniform buffer, too small for the prioritized one
    torch.cuda.synchronize()
    assert len(rp) == 1 and int(out[-1].max()) == 0
    for _ in range(5):
        rp.add_batch(obs, torch.rand((1, 2), device=dev), torch.ones(1, device=dev), obs, torch.zeros(1, dtype=torch.uint8, device=dev))
    rp2 = GpuReplayBuffer(64, L, 2, prioritized, 0.6, 0.4)
    for _ in range(6):
        rp2.add_batch(obs, torch.rand((1, 2), device=dev), torch.ones(1, device=dev), obs, torch.zeros(1, dtype=torch.uint8, device=dev))
    assert rp2.error_flags == 0
    rp2.gather(torch.tensor([0, 5, 6, -1, 1000], dtype=torch.int32, device=dev))   # 6, -1, 1000 are outside [0, 6)
    torch.cuda.synchronize()
    assert rp2.error_flags & 2
    if prioritized:
        rp3 = GpuReplayBuffer(64, L, 2, True, 0.6, 0.4)
        for _ in range(6):
            rp3.add_batch(obs, torch.rand((1, 2), device=dev), torch.ones(1, device=dev), obs, torch.zeros(1, dtype=torch.uint8, device=dev))
        s0 = rp3.sample(u)
        rp3.update_priorities(torch.tensor([0, 1, 2], dtype=torch.int32, device=dev), torch.tensor([0.5, 0.0, -1.0], dtype=torch.float64, device=dev))
        torch.cuda.synchronize()
        assert rp3.error_flags & 4
        w = rp3.sample(u)[-2]
        assert bool(torch.isfinite(w).all())    # the trees were not poisoned by the bad priorities
        with pytest.raises(Exception):
            rp3.raise_on_error()
