"""Rollouts whose decision observations k_simple hands off to observer warps (agar_rollout_random at 4 and 8 lanes per env,
>= 8 frames per decision): every row a decision stores equals the portable-math oracle's, and the rollout equals the one
whose observations are encoded inline (2 lanes per env)."""
import numpy as np
import pytest

import aigar_b200.layout as lay

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def torch_cuda():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("these tests need a GPU (the product has no CPU fallback; run with -m gpu on the B200 box)")
    return torch


@pytest.mark.parametrize("tile", [8, 4])
def test_every_decision_row_equals_oracle(torch_cuda, tile):
    """One launch per decision, so that each decision's row is visible; 70 envs leave a partly filled CTA.  Then one
    multi-decision launch (both snapshot buffers reused) and every record."""
    from aigar_b200.env import AgarBatch
    from oracle import oracle as orc
    cfg = lay.derive_config()
    n, seed, first = 70, 31, 500
    b = AgarBatch(cfg, n, seed=seed, first_env_id=first, tile_width=tile)
    oras = [orc.OracleEnv(cfg, seed=seed, env_id=first + i, portable=True) for i in range(n)]
    n_obs = b.observer_launch_count
    for d in range(125):
        obs = b.rollout_random(1, 8, d).cpu().numpy()
        for i, e in enumerate(oras):
            e.rollout_random(1, 8, d)
            assert np.array_equal(e.obs[0], obs[i, 0]), "tile %d decision %d env %d" % (tile, d, i)
    obs = b.rollout_random(7, 8, 125).cpu().numpy()
    assert b.observer_launch_count == n_obs + 126  # every launch above ran the observer warps
    st = b.state_tensor().cpu().numpy()
    for i, e in enumerate(oras):
        e.rollout_random(7, 8, 125)
        assert np.array_equal(e.obs[0], obs[i, 0]), "tile %d env %d after the 7-decision launch" % (tile, i)
        diff = lay.compare_records(e.record, lay.Record(b.layout, st[i].copy()), what="env %d " % i)
        assert not diff, diff


@pytest.mark.parametrize("frames", [8, 4])
def test_bench_size_equals_inline_encoder(torch_cuda, frames):
    """4096 envs x 1000 frames, an observation every `frames` frames, at the default tile width (observer warps) == the same
    rollout at 2 lanes per env."""
    torch = torch_cuda
    from aigar_b200.env import AgarBatch
    cfg = lay.derive_config()
    a = AgarBatch(cfg, 4096, seed=2026)
    c = AgarBatch(cfg, 4096, seed=2026, tile_width=2)
    assert a.tile_width == 8
    oa = a.rollout_random(1000 // frames, frames, 0)
    oc = c.rollout_random(1000 // frames, frames, 0)
    assert (a.observer_launch_count, c.observer_launch_count) == (1, 0)
    assert torch.equal(a.state_tensor(), c.state_tensor())
    assert torch.equal(oa, oc)


def test_observers_only_where_the_waves_allow(torch_cuda):
    """On 148 SMs an observer CTA holds at most 28 envs (W = 8) and an SM one such CTA, the inline shape two CTAs of 16 envs:
    4096 envs take one wave either way (observer warps), 4608 would take two instead of one (inline encoder)."""
    from aigar_b200.env import AgarBatch
    if torch_cuda.cuda.get_device_properties(0).multi_processor_count != 148:
        pytest.skip("the wave counts below are those of a 148-SM B200")
    cfg = lay.derive_config()
    for n, expect in ((4096, 1), (4608, 0)):
        b = AgarBatch(cfg, n, seed=3)
        assert b.tile_width == 8
        b.rollout_random(2, 8, 0)
        assert b.observer_launch_count == expect, n
        b.close()
