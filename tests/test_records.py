"""State snapshots (agar_save_records / agar_load_records, AgarBatch.snapshot / restore / save_checkpoint / load_checkpoint):
a restore is a replay bit for bit, a clone steps like the oracle under its slot's key, loads refuse records that could make
a kernel index out of bounds, and checkpoint files are checked field by field."""
import ctypes

import numpy as np
import pytest

import aigar_b200.layout as lay
from aigar_b200 import env as agar_env

gpu = pytest.mark.gpu

CFG_1V1 = dict(num_nn=1, num_greedy=1, virus=True, split=True, eject=True)
CFG_ARENA = dict(num_nn=8, num_greedy=8, virus=True, split=True, eject=True)


@pytest.fixture(scope="module")
def torch_cuda():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("these tests need a GPU (the product has no CPU fallback; run with -m gpu on the B200 box)")
    return torch


def _batch(cfg, n, **kw):
    from aigar_b200.env import AgarBatch
    return AgarBatch(cfg, n, **kw)


def _continue(torch, b, frames):
    """step_observe with seeded actions, then rollout_random at a fixed decision_base: every record, observation and
    agar_get field along the way."""
    g = torch.Generator(device=b.device).manual_seed(11)
    out = []
    for _ in range(3):
        act = torch.rand(b.actions.shape, device=b.device, generator=g)
        out += [b.step_observe(act, frames).clone(), b.state_tensor().clone()]
    out += [b.rollout_random(4, frames, 100).clone(), b.state_tensor().clone()]
    for which in range(lay.GET_EVENT_HASH + 1):
        out.append(b.get(which))
    return out


# (config, n_envs, tile width, frames per decision, expected record bytes or None)
ROUND_TRIP = [
    ("k_simple W=8", dict(), 64, 8, 8, None),
    ("k_simple W=1", dict(), 64, 1, 8, None),
    ("observer warps", dict(), 4096, None, 8, None),
    ("1-vs-greedy", CFG_1V1, 32, None, 8, 8960),
    ("arena", CFG_ARENA, 6, None, 4, 60672),
    ("G=42", dict(grid=42, overrides={"use_fovsize": 0, "use_totalmass": 0}), 16, None, 4, None),
]


@gpu
@pytest.mark.parametrize("name,kw,n,tile,frames,rb", ROUND_TRIP, ids=[c[0] for c in ROUND_TRIP])
def test_round_trip_is_a_replay(torch_cuda, name, kw, n, tile, frames, rb):
    torch = torch_cuda
    b = _batch(lay.derive_config(**kw), n, seed=21, first_env_id=300, tile_width=tile)
    if rb is not None:
        assert int(b.layout.record_bytes) == rb
    b.rollout_random(3, frames, 0)
    bank, obs0 = b.snapshot(), b.obs.clone()
    n_obs = b.observer_launch_count if name == "observer warps" else 0
    first = _continue(torch, b, frames)
    if name == "observer warps":
        assert b.tile_width == 8 and b.observer_launch_count > n_obs
    b.restore(bank)
    b.obs.copy_(obs0)
    assert torch.equal(b.state_tensor(), bank)
    second = _continue(torch, b, frames)
    for i, (x, y) in enumerate(zip(first, second)):
        assert torch.equal(x, y), "%s: output %d differs after the restore" % (name, i)


@gpu
def test_partial_restore_changes_only_indexed_envs(torch_cuda):
    torch = torch_cuda
    cfg = lay.derive_config(**CFG_1V1)
    a, c = _batch(cfg, 16, seed=4, first_env_id=7), _batch(cfg, 16, seed=4, first_env_id=7)
    for b in (a, c):
        b.rollout_random(5, 8, 0)
    bank = a.snapshot()
    for b in (a, c):
        b.rollout_random(5, 8, 5)
    assert not torch.equal(a.state_tensor(), bank)
    idx = torch.full((16,), -1, dtype=torch.int32, device=a.device)
    idx[[1, 6, 7, 12]] = torch.tensor([1, 6, 3, 15], dtype=torch.int32, device=a.device)
    a.restore(bank, idx)
    st, ref = a.state_tensor(), c.state_tensor()
    keep = (idx < 0).nonzero().flatten()
    assert torch.equal(st[keep], ref[keep])
    for e in (1, 6, 7, 12):
        assert torch.equal(st[e], bank[int(idx[e])])
    for b in (a, c):
        b.rollout_random(4, 8, 10)
    assert torch.equal(a.state_tensor()[keep], c.state_tensor()[keep])
    assert a.record_error_flags() == 0


@gpu
def test_clone_equals_oracle_under_the_slot_key(torch_cuda):
    torch = torch_cuda
    from oracle import oracle as orc
    cfg = lay.derive_config(event_cap=64, **CFG_1V1)
    seed, first, s, d = 7, 20, 1, 4
    b = _batch(cfg, 6, seed=seed, first_env_id=first)
    b.rollout_random(6, 8, 0)
    bank = b.snapshot()
    src = bank[s].cpu().numpy()
    idx = torch.full((6,), -1, dtype=torch.int32, device=b.device)
    idx[d] = s
    b.restore(bank, idx)                          # the documented clone recipe: save, then load with an index
    assert torch.equal(b.state_tensor()[d], bank[s])
    ora = orc.OracleEnv(cfg, seed=seed, env_id=first + d, portable=True)
    ora.load_record(src)
    ora.set_key(seed, first + d)
    other = _batch(cfg, 2, seed=seed, first_env_id=first + d)   # slot 0 has d's global id
    other.restore(bank[s:s + 1].clone(), torch.tensor([0, -1], dtype=torch.int32, device=b.device))
    b.rollout_random(5, 8, 6)
    ora.rollout_random(5, 8, 6)
    other.rollout_random(5, 8, 6)
    st = b.state_tensor().cpu().numpy()
    diff = lay.compare_records(ora.record, lay.Record(b.layout, st[d].copy()), check_events=True)
    assert not diff, diff
    assert torch.equal(other.state_tensor()[0], b.state_tensor()[d])


@gpu
def test_snapshot_gathers_rows(torch_cuda):
    torch = torch_cuda
    b = _batch(lay.derive_config(**CFG_1V1), 10, seed=2)
    b.rollout_random(3, 8, 0)
    st = b.state_tensor()
    for envs in ([3, 3, 0, 9, 5], [9, 8, 7, 6, 5, 4, 3, 2, 1, 0, 0, 1, 2], [4]):
        idx = torch.tensor(envs, dtype=torch.int32, device=b.device)
        assert torch.equal(b.snapshot(idx), st[idx.long()])
    out = torch.zeros((3, int(b.layout.record_bytes)), dtype=torch.uint8, device=b.device)
    assert b.snapshot(torch.tensor([2, 2, 7], dtype=torch.int32, device=b.device), out=out) is out
    assert torch.equal(out, st[[2, 2, 7]])
    assert torch.equal(b.snapshot(), st)
    assert b.record_error_flags() == 0


def _rewrite(src, dst, **changes):
    with np.load(src, allow_pickle=False) as z:
        d = {k: z[k] for k in z.files}
    d.update(changes)
    with open(dst, "wb") as f:
        np.savez(f, **d)
    return dst


def _mismatched_files(tmp_path, good, cfg, layout, n_envs, seed, first, records):
    """(file, word its refusal must name) for each field a load checks"""
    out = []
    cfg2 = lay.AgarConfig.from_buffer_copy(bytes(cfg))
    cfg2.reward_scale += 1.0
    lay2 = lay.AgarLayout.from_buffer_copy(bytes(layout))
    lay2.max_pellets += 1.0
    for name, args in (("config", (cfg2, layout, n_envs, seed, first, records)),
                       ("layout", (cfg, lay2, n_envs, seed, first, records)),
                       ("n_envs", (cfg, layout, n_envs - 1, seed, first, records[:-1])),
                       ("seed", (cfg, layout, n_envs, seed + 1, first, records)),
                       ("first_env_id", (cfg, layout, n_envs, seed, first + 1, records))):
        p = str(tmp_path / ("bad_%s.npz" % name))
        agar_env.write_checkpoint(p, *args)
        out.append((p, name))
    out.append((_rewrite(good, str(tmp_path / "bad_format.npz"), format=np.array("something.else")), "format"))
    out.append((_rewrite(good, str(tmp_path / "bad_abi.npz"), abi_version=np.int64(lay.ABI_VERSION + 1)), "abi_version"))
    tampered = records.copy()
    tampered[-1, 17] ^= 1
    out.append((_rewrite(good, str(tmp_path / "bad_digest.npz"), records=tampered), "sha256"))
    return out


def test_checkpoint_file_checks_without_a_device(tmp_path):
    """Parsing and matching a checkpoint needs no GPU: a stand-in writes the files."""
    cfg = lay.derive_config(**CFG_1V1)
    layout = lay.layout_for_config(cfg)
    n, seed, first = 5, 3, 2 ** 63 + 11
    records = np.random.default_rng(0).integers(0, 256, (n, int(layout.record_bytes)), dtype=np.uint8)
    good = str(tmp_path / "ck")                   # no .npz suffix: the file is written under exactly this name
    agar_env.write_checkpoint(good, cfg, layout, n, seed, first, records)
    ck = agar_env.read_checkpoint(good)
    agar_env.check_checkpoint(ck, cfg, layout, n, seed, first)
    assert np.array_equal(ck["records"], records)
    assert bytes(lay.AgarConfig.from_buffer_copy(ck["config"].tobytes())) == bytes(cfg)
    for path, word in _mismatched_files(tmp_path, good, cfg, layout, n, seed, first, records):
        with pytest.raises(agar_env.CheckpointError, match=word):
            agar_env.check_checkpoint(agar_env.read_checkpoint(path), cfg, layout, n, seed, first)
    nodigest = str(tmp_path / "nodigest.npz")
    with np.load(good, allow_pickle=False) as z:
        np.savez(nodigest, **{k: z[k] for k in z.files if k != "sha256"})
    with pytest.raises(agar_env.CheckpointError, match="missing sha256"):
        agar_env.read_checkpoint(nodigest)


def test_abi_version_matches_the_header():
    import os
    import re
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    src = open(os.path.join(root, "include", "agar_b200.h")).read()
    assert int(re.search(r"#define AGAR_ABI_VERSION (\d+)", src).group(1)) == lay.ABI_VERSION
    assert int(re.search(r"AGAR_REC_ERR_INDEX = (\d+)", src).group(1)) == lay.REC_ERR_INDEX
    assert int(re.search(r"AGAR_REC_ERR_RECORD = (\d+)", src).group(1)) == lay.REC_ERR_RECORD


@gpu
def test_checkpoint_round_trip_and_refusals(torch_cuda, tmp_path):
    torch = torch_cuda
    from aigar_b200.env import AgarBatch, CheckpointError
    cfg = lay.derive_config(**CFG_1V1)
    a = _batch(cfg, 16, seed=9, first_env_id=40)
    a.rollout_random(4, 8, 0)
    path = str(tmp_path / "batch.npz")
    a.save_checkpoint(path)
    b = AgarBatch.from_checkpoint(path, tile_width=8)
    assert (b.tile_width, a.tile_width) == (8, 32)
    assert (b.n_envs, b.seed, b.first_env_id) == (16, 9, 40)
    assert torch.equal(a.state_tensor(), b.state_tensor())
    a.rollout_random(5, 8, 4)
    b.rollout_random(5, 8, 4)
    assert torch.equal(a.state_tensor(), b.state_tensor())
    records = a.snapshot().cpu().numpy()
    a.save_checkpoint(path)
    before = b.state_tensor().clone()
    b.rollout_random(1, 8, 9)
    changed = b.state_tensor().clone()
    assert not torch.equal(changed, before)
    for p, word in _mismatched_files(tmp_path, path, cfg, b.layout, 16, 9, 40, records):
        with pytest.raises(CheckpointError, match=word):
            b.load_checkpoint(p)
        assert torch.equal(b.state_tensor(), changed), word
    b.load_checkpoint(path)
    assert torch.equal(b.state_tensor(), before)
    assert b.record_error_flags() == 0
    # a file with a valid digest but a record the device-side checks refuse: nothing is loaded, also once the sticky
    # refusal bit is already set
    corrupt = records.copy()
    lay.Record(b.layout, corrupt[5]).header["n_blobs"][0] = b.layout.blob_cap + 1
    bad = str(tmp_path / "bad_record.npz")
    agar_env.write_checkpoint(bad, cfg, b.layout, 16, 9, 40, corrupt)
    b.rollout_random(1, 8, 9)
    changed = b.state_tensor().clone()
    for _ in range(2):
        with pytest.raises(CheckpointError, match="device-side"):
            b.load_checkpoint(bad)
        assert torch.equal(b.state_tensor(), changed)
    assert b.record_error_flags() == lay.REC_ERR_RECORD


def _corrupt_rows(layout, bank_h):
    """one row per listed field, each set one past its capacity (or below 0); returns the corrupted row numbers"""
    L = layout
    K = L.n_players
    cases = [("n_viruses", L.virus_cap + 1), ("n_blobs", L.blob_cap + 1), ("n_fat", L.fat_cap + 1),
             ("n_pellets", L.pellet_cap + 1), ("n_dead", K + 1), ("n_viruses", -1), ("n_cells", L.cell_cap + 1),
             ("n_cells", -1), ("dead_order", K), ("dead_twice", 0), ("pellet_x", L.field_size), ("pellet_y", L.field_size)]
    rows = []
    for r, (field, v) in enumerate(cases):
        rec = lay.Record(L, bank_h[r])
        if field == "n_cells":
            rec.players["n_cells"][K - 1] = v
        elif field == "dead_order":
            rec.header["n_dead"][0] = 1
            rec.header["dead_order"][0][0] = v
        elif field == "dead_twice":
            rec.header["n_dead"][0] = 2
            rec.header["dead_order"][0][:2] = [1, 1]
        elif field.startswith("pellet_"):
            rec.pellets[3] = lay.pack_pellet(v, 5, 1) if field == "pellet_x" else lay.pack_pellet(5, v, 1)
        else:
            rec.header[field][0] = v
        rows.append(r)
    return rows


@gpu
def test_validation_refuses_bad_rows_and_indices(torch_cuda):
    torch = torch_cuda
    cfg = lay.derive_config(**CFG_1V1)
    n = 16
    src = _batch(cfg, n, seed=5)
    src.rollout_random(4, 8, 0)
    bank_h = src.snapshot().cpu().numpy()
    bad = _corrupt_rows(src.layout, bank_h)
    assert len(bad) < n
    bank = torch.from_numpy(bank_h).to(src.device)
    dst = _batch(cfg, n, seed=5)
    before = dst.state_tensor().clone()
    dst.restore(bank)
    st = dst.state_tensor()
    good = [e for e in range(n) if e not in bad]
    assert torch.equal(st[bad], before[bad])
    assert torch.equal(st[good], bank[good])
    assert dst.record_error_flags() == lay.REC_ERR_RECORD
    dst.rollout_random(3, 8, 4)                   # only valid records were installed
    torch.cuda.synchronize()

    # indices out of range: those envs / rows stay untouched, the rest is copied
    dst2 = _batch(cfg, n, seed=5)
    before = dst2.state_tensor().clone()
    idx = torch.arange(n, dtype=torch.int32, device=src.device).flip(0)
    idx[2], idx[5], idx[9] = n, -2, -1
    good_bank = src.snapshot()
    dst2.restore(good_bank, idx)
    st = dst2.state_tensor()
    for e in range(n):
        want = before[e] if e in (2, 5, 9) else good_bank[int(idx[e])]
        assert torch.equal(st[e], want), e
    assert dst2.record_error_flags() == lay.REC_ERR_INDEX
    out = torch.full((4, int(src.layout.record_bytes)), 0xAB, dtype=torch.uint8, device=src.device)
    src.snapshot(torch.tensor([1, n, -1, 0], dtype=torch.int32, device=src.device), out=out)
    st = src.state_tensor()
    assert torch.equal(out[0], st[1]) and torch.equal(out[3], st[0])
    assert bool((out[1:3] == 0xAB).all())
    assert src.record_error_flags() == lay.REC_ERR_INDEX


@gpu
@pytest.mark.parametrize("kw,n,decisions", [(CFG_1V1, 64, 125), (CFG_ARENA, 8, 100)], ids=["1-vs-greedy", "arena"])
def test_simulated_records_pass_validation(torch_cuda, kw, n, decisions):
    """After a long rollout every record the simulator produced loads: the checks refuse nothing it makes."""
    torch = torch_cuda
    cfg = lay.derive_config(**kw)
    b = _batch(cfg, n, seed=13)
    b.rollout_random(decisions, 8, 0)
    bank = b.snapshot()
    c = _batch(cfg, n, seed=13)
    c.restore(bank)
    b.restore(bank.clone())
    assert b.record_error_flags() == 0 and c.record_error_flags() == 0
    assert torch.equal(c.state_tensor(), bank)


@gpu
def test_host_refusals(torch_cuda):
    torch = torch_cuda
    b = _batch(lay.derive_config(), 8)
    rb = int(b.layout.record_bytes)
    vp, i32 = ctypes.c_void_p, ctypes.c_int
    save = b._lazy("agar_save_records", [vp, vp, vp, i32, vp])
    load = b._lazy("agar_load_records", [vp, vp, i32, vp, vp])
    bank = torch.zeros((9, rb), dtype=torch.uint8, device=b.device)
    before = b.state_tensor().clone()
    n0 = b.launch_count
    state = b.lib.agar_state_ptr(b.h)
    p, s = bank.data_ptr(), b._stream()
    one_t, idx8_t = torch.zeros(1, dtype=torch.int32, device=b.device), torch.zeros(8, dtype=torch.int32, device=b.device)
    one, idx8 = vp(one_t.data_ptr()), vp(idx8_t.data_ptr())
    cases = [
        save(b.h, None, None, 8, s), load(b.h, None, 8, None, s),                       # NULL bank
        save(b.h, vp(p + 8), None, 8, s), load(b.h, vp(p + 1), 8, None, s),            # not 16-byte aligned
        # overlapping the records: every address named lies inside the handle's own allocation, so a regression of the
        # check could not touch memory the test does not own
        save(b.h, vp(state + 7 * rb), one, 1, s), load(b.h, vp(state), 8, None, s),
        load(b.h, vp(state + 3 * rb), 5, idx8, s),
        save(b.h, vp(p), None, 0, s), load(b.h, vp(p), 0, None, s),                     # no rows
        save(b.h, vp(p), None, 9, s), load(b.h, vp(p), 7, None, s),                     # NULL index, row count != n_envs
    ]
    assert cases == [-1] * len(cases)
    assert b.lib.agar_last_error(b.h).decode().startswith("agar_")
    assert b.launch_count == n0
    assert torch.equal(b.state_tensor(), before) and b.record_error_flags() == 0
    with pytest.raises(ValueError):
        b.restore(bank[:, :-1])
    with pytest.raises(ValueError):
        b.restore(bank[:8], torch.zeros(8, dtype=torch.int64, device=b.device))


@gpu
def test_restore_in_a_cuda_graph(torch_cuda):
    torch = torch_cuda
    cfg = lay.derive_config()
    a, c = _batch(cfg, 512, seed=12), _batch(cfg, 512, seed=12)
    for b in (a, c):
        b.rollout_random(4, 8, 0)
    bank = a.snapshot()
    for b in (a, c):
        b.rollout_random(2, 8, 4)
    g = torch.Generator(device=a.device).manual_seed(1)
    idx = torch.randint(-1, 512, (512,), device=a.device, generator=g).to(torch.int32)
    act = torch.rand(a.actions.shape, device=a.device, generator=g)
    for _ in range(2):
        a.restore(bank, idx)
        a.step_observe(act, 8)
    graph = torch.cuda.CUDAGraph()
    n0 = c.launch_count
    with torch.cuda.graph(graph):
        c.restore(bank, idx)
        c.step_observe(act, 8)
    assert c.launch_count == n0 + 2
    for _ in range(2):
        graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(a.state_tensor(), c.state_tensor()) and torch.equal(a.obs, c.obs)
    assert c.record_error_flags() == 0
