"""k_simple (the register-resident single-cell kernel) against the portable-math oracle over the configs and launch shapes it
admits: every tile width, grid size, observation mode, extras set, pellet cap at the edges of the candidate-mask words,
an empty pool, every frame_skip / frames-per-decision pairing, the reward variants and the event-ring sizes.  Three paths
per case: observe + one frame, step_observe over several frames, and rollout_random (one launch per decision, then multi-decision
launches).  Then the launch shapes of the observer-warp rollout, and configs without a pellet grid (general kernel).

Everything is compared exactly (rtol = 0): every observation row, reward and turn flag, and every record with its events."""
import numpy as np
import pytest

import aigar_b200.layout as lay
import gpu_check

pytestmark = pytest.mark.gpu

REF, CANON = lay.OBS_REFERENCE, lay.OBS_CANONICAL
MASS = {"mass_as_reward": True}


def case(name, W, G, obs, fov, mass, cap, fs, nf, ev, spawn=True, reward=None):
    """One admitted config.  cap: pellet_cap override (None: the layout's own, 85 with spawning, 0 without); nf: frames per
    rollout decision, chosen against fs so that decisions align with turns (nf a multiple of fs + 1) or not."""
    return dict(name=name, W=W, G=G, obs=obs, fov=fov, mass=mass, cap=cap, fs=fs, nf=nf, ev=ev, spawn=spawn,
                reward=reward or {})


CASES = [
    case("w1_g1", 1, 1, REF, 1, 1, 85, 7, 8, 64),
    case("w1_g15_bits", 1, 15, REF, 1, 0, 128, 0, 1, 64),
    case("w1_g16_nobits", 1, 16, REF, 0, 0, 85, 3, 5, 2),
    case("w1_g5_canon", 1, 5, CANON, 0, 1, 128, 9, 9, 0, reward=MASS),
    case("w2_g15_bits", 2, 15, REF, 1, 1, 128, 1, 3, 64),
    case("w2_g16_nobits", 2, 16, REF, 1, 1, 129, 7, 9, 2),
    case("w2_g2_canon", 2, 2, CANON, 1, 0, 256, 3, 4, 64, reward={"reward_scale": 0.5, "reward_term": 0.25}),
    case("w2_g3_empty", 2, 3, REF, 1, 1, None, 7, 8, 64, spawn=False),
    case("w4_g7", 4, 7, REF, 1, 1, 128, 7, 5, 64),
    case("w4_g11_canon", 4, 11, CANON, 1, 0, 129, 3, 4, 64),
    case("w4_g13", 4, 13, REF, 0, 1, 256, 9, 5, 2, reward=MASS),
    case("w4_g16_canon", 4, 16, CANON, 0, 0, 85, 1, 3, 0),
    case("w8_g11", 8, 11, REF, 1, 1, 256, 7, 8, 64),
    case("w8_g16_canon", 8, 16, CANON, 1, 1, 257, 7, 9, 64),
    case("w8_g15", 8, 15, REF, 0, 0, 512, 3, 4, 0),
    case("w8_g1_canon", 8, 1, CANON, 1, 1, 85, 0, 1, 2, reward={"reward_scale": 3.0, "reward_term": -0.5}),
    case("w8_g5_empty", 8, 5, REF, 1, 1, None, 9, 9, 64, spawn=False),
    case("w16_g13_canon", 16, 13, CANON, 1, 1, 85, 9, 5, 64, reward={"reward_scale": 1.0, "reward_term": 0.125}),
    case("w16_g3", 16, 3, REF, 1, 0, 300, 1, 4, 2),
    case("w32_g16", 32, 16, REF, 1, 1, 200, 7, 8, 2),
    case("w32_g7_canon", 32, 7, CANON, 0, 1, 85, 0, 1, 64, reward=MASS),
]
IDS = [c["name"] for c in CASES]

# the axes every case list must cover (a later edit must not drop one silently)
AXIS_W = {1, 2, 4, 8, 16, 32}
AXIS_G = {1, 2, 3, 5, 7, 11, 13, 15, 16}
CAP_EDGES = {1: {85, 128}, 2: {128, 129, 256}, 4: {128, 129, 256}, 8: {256, 257, 512}}
CAP_LIMIT = {W: (128 if W <= 2 else 64) * W for W in AXIS_W}  # two candidate-mask words per lane (SMask<W>)
OBS_LANES, OBS_WARPS, OBS_MIN_FRAMES = 4, 4, 4  # observer warps: SIMPLE_OBS_LANES, SIMPLE_OBS_WARPS, SIMPLE_OBS_MIN_FRAMES
OBS_MAX_THREADS = {4: 256, 8: 352}  # simple_max_threads


def case_kw(c):
    ov = {"use_fovsize": c["fov"], "use_totalmass": c["mass"]}
    if c["cap"] is not None:
        ov["pellet_cap"] = c["cap"]
    return dict(grid=c["G"], obs_mode=c["obs"], frame_skip=c["fs"], pellet_spawn=c["spawn"], overrides=ov, **c["reward"])


def observers_expected(c, layout):
    return c["W"] in (4, 8) and c["nf"] >= OBS_MIN_FRAMES and layout.pellet_cap <= 64 * OBS_LANES


@pytest.fixture(scope="module")
def torch_cuda():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("these tests need a GPU (the product has no CPU fallback; run with -m gpu on the B200 box)")
    return torch


def spread_pellets(batch, oras):
    """Move each env's live pellets from the lowest slots (where spawning puts them) to slots spread over the whole pool, the
    last slot included, in the oracle and on the GPU alike: otherwise the second candidate-mask word never holds a pellet."""
    for i, e in enumerate(oras):
        rec = lay.Record(e.layout, e.record.buf.copy())
        live = rec.pellets[rec.pellets != 0].copy()
        cap = len(rec.pellets)
        if len(live) < 2 or len(live) == cap:
            continue
        slots = np.round(np.linspace(cap - 1, 0, len(live))).astype(np.int64)
        assert len(set(slots.tolist())) == len(live)
        rec.pellets[:] = 0
        rec.pellets[slots] = live
        e.load_record(rec)
        batch.load(i, rec)


def make(cfg, n_envs, W, seed, first, spread=True):
    from aigar_b200.env import AgarBatch
    from oracle import oracle as orc
    b = AgarBatch(cfg, n_envs, seed=seed, first_env_id=first, tile_width=W)
    assert W is None or b.tile_width == W
    oras = [orc.OracleEnv(cfg, seed=seed, env_id=first + i, portable=True) for i in range(n_envs)]
    if spread:
        spread_pellets(b, oras)
    return b, oras


def assert_equal_to_oracle(b, oras, obs, tag, envs=None):
    """Rows of the observation buffer, reward and turn flags of agar_get, and the records (events included) of `envs`."""
    envs = range(b.n_envs) if envs is None else envs
    obs = obs.cpu().numpy()
    st = b.state_tensor().cpu().numpy()
    get = {k: b.get(k).cpu().numpy() for k in (lay.GET_REWARD, lay.GET_NEED_ACTION, lay.GET_VALID, lay.GET_DONE)}
    for i in envs:
        e = oras[i]
        where = "%s env %d" % (tag, i)
        neq = obs[i] != e.obs
        if neq.any():
            j = tuple(np.argwhere(neq)[0])
            pytest.fail("%s obs%r: gpu %r oracle %r (%d differ)" % (where, list(j), obs[i][j], e.obs[j], int(neq.sum())))
        t = e.turn()[0]
        got = (bool(get[lay.GET_NEED_ACTION][i, 0]), bool(get[lay.GET_VALID][i, 0]), bool(get[lay.GET_DONE][i, 0]))
        assert got == (t["need_action"], t["valid"], t["done"]), where + " turn flags"
        assert get[lay.GET_REWARD][i, 0] == np.float32(t["reward"]), where + " reward"
        diff = lay.compare_records(e.record, lay.Record(b.layout, st[i].copy()), what=where + " ", check_events=True)
        assert not diff, "\n".join(diff[:6])


# ---------------------------------------------------------------- (a) the admission domain
def test_case_list_covers_the_domain():
    assert {c["W"] for c in CASES} == AXIS_W
    assert {c["G"] for c in CASES} >= AXIS_G
    for W in (1, 2):  # use_bits: on at G = 15, off at G = 16 (reference binning only)
        assert {c["G"] for c in CASES if c["W"] == W and c["obs"] == REF} >= {15, 16}, W
    for W in AXIS_W:
        assert {c["obs"] for c in CASES if c["W"] == W} == {REF, CANON}, W
    assert {(c["fov"], c["mass"]) for c in CASES} == {(1, 1), (1, 0), (0, 1), (0, 0)}
    for W, caps in CAP_EDGES.items():
        assert {c["cap"] for c in CASES if c["W"] == W} >= caps, W
    assert any(not c["spawn"] for c in CASES)
    assert {c["fs"] for c in CASES} >= {0, 1, 3, 7, 9}
    assert any(c["reward"].get("mass_as_reward") for c in CASES)
    assert any("reward_scale" in c["reward"] and "reward_term" in c["reward"] for c in CASES)
    assert {c["ev"] for c in CASES} == {0, 2, 64}
    assert {c["nf"] for c in CASES} == {1, 3, 4, 5, 8, 9}
    assert any(c["nf"] % (c["fs"] + 1) == 0 for c in CASES) and any(c["nf"] % (c["fs"] + 1) for c in CASES)
    # observer rollouts whose decisions do and do not all observe, and the observer pool's second mask word (cap > 128)
    obs_cases = [c for c in CASES if c["W"] in (4, 8) and c["nf"] >= OBS_MIN_FRAMES and (c["cap"] or 0) <= 256]
    assert any(c["nf"] % (c["fs"] + 1) for c in obs_cases) and any(c["nf"] % (c["fs"] + 1) == 0 for c in obs_cases)
    assert any((c["cap"] or 0) > 128 for c in obs_cases)
    assert len(set(IDS)) == len(IDS)


@pytest.mark.parametrize("c", CASES, ids=IDS)
def test_case_admitted(torch_cuda, c):
    cfg = lay.derive_config(event_cap=c["ev"], **case_kw(c))
    L = lay.layout_for_config(cfg)
    assert L.pellet_cap == (c["cap"] if c["cap"] is not None else 0)
    assert L.state_len == c["G"] ** 2 + c["fov"] + c["mass"]
    b, _ = make(cfg, 2, c["W"], seed=1, first=0, spread=False)
    assert b.tile_width == c["W"]


@pytest.mark.parametrize("W", sorted(AXIS_W))
def test_pellet_cap_limit(torch_cuda, W):
    """The largest pool a tile width holds is admitted; one slot more is refused."""
    from aigar_b200.env import AgarBatch, AgarError
    cap = CAP_LIMIT[W]
    b = AgarBatch(lay.derive_config(overrides={"pellet_cap": cap}), 2, tile_width=W)
    assert b.tile_width == W
    with pytest.raises(AgarError):
        AgarBatch(lay.derive_config(overrides={"pellet_cap": cap + 1}), 2, tile_width=W)


def test_grid_17_refuses_k_simple(torch_cuda):
    """k_simple bins a pellet into at most two squares per axis, which needs G <= 16: G = 17 runs the general kernel only."""
    from aigar_b200.env import AgarBatch, AgarError
    cfg = lay.derive_config(grid=17)
    assert AgarBatch(cfg, 2).tile_width == 32
    with pytest.raises(AgarError):
        AgarBatch(cfg, 2, tile_width=8)


# ---------------------------------------------------------------- (b) three paths per case
@pytest.mark.parametrize("c", CASES, ids=IDS)
def test_per_frame(torch_cuda, c):
    def setup(b, oras):
        assert b.tile_width == c["W"]
        spread_pellets(b, oras)

    assert gpu_check.check(case_kw(c), n_envs=8, frames=100, seed=11, first_env=40, tile_width=c["W"], event_cap=c["ev"],
                           verbose=False, setup=setup)


@pytest.mark.parametrize("c", CASES, ids=IDS)
def test_step_observe(torch_cuda, c):
    """step_observe(acts, n) == oracle step(act, n) + observe: the trailing observation follows n frames."""
    cfg = lay.derive_config(event_cap=c["ev"], **case_kw(c))
    b, oras = make(cfg, 7, c["W"], seed=12, first=300)
    rng = np.random.default_rng(12)
    for k, n in enumerate([1, 3, 8] * 7):
        act = rng.random((b.n_envs, 1, 4)).astype(np.float32)
        obs = b.step_observe(act, n)
        for i, e in enumerate(oras):
            e.step(act[i], n)
            e.observe()
        assert_equal_to_oracle(b, oras, obs, "call %d (%d frames)" % (k, n))


def run_rollout(cfg, W, nf, n_envs, seed, first, frames=100):
    """rollout_random one decision per launch (each decision's row visible), then launches of 2, 3 and 7 decisions.  Returns
    (batch, launches)."""
    b, oras = make(cfg, n_envs, W, seed, first)
    d = 0
    launches = 0
    for _ in range(max(6, frames // nf)):
        obs = b.rollout_random(1, nf, d)
        for e in oras:
            e.rollout_random(1, nf, d)
        assert_equal_to_oracle(b, oras, obs, "decision %d (%d frames)" % (d, nf))
        d += 1
        launches += 1
    for n_dec in (2, 3, 7):
        obs = b.rollout_random(n_dec, nf, d)
        for e in oras:
            e.rollout_random(n_dec, nf, d)
        assert_equal_to_oracle(b, oras, obs, "%d-decision launch from decision %d (%d frames)" % (n_dec, d, nf))
        d += n_dec
        launches += 1
    return b, launches


@pytest.mark.parametrize("c", CASES, ids=IDS)
def test_rollout_random(torch_cuda, c):
    cfg = lay.derive_config(event_cap=c["ev"], **case_kw(c))
    b, launches = run_rollout(cfg, c["W"], c["nf"], 6, seed=13, first=700)
    assert b.tile_width == c["W"]
    assert b.observer_launch_count == (launches if observers_expected(c, b.layout) else 0)


# ---------------------------------------------------------------- (c) observer launch shapes
SHAPE_CFGS = {"default": (dict(), 8),
              "g16_canon_cap256_fs3": (dict(grid=16, obs_mode=CANON, frame_skip=3, overrides={"pellet_cap": 256}), 4)}


def rollout_both(b, oras, nf, dec0, n_dec):
    obs = b.rollout_random(n_dec, nf, dec0)
    for e in oras:
        e.rollout_random(n_dec, nf, dec0)
    return obs


@pytest.mark.parametrize("W", [4, 8])
@pytest.mark.parametrize("which", sorted(SHAPE_CFGS))
def test_observer_small_batches(torch_cuda, which, W):
    """Batches up to one env past a CTA (27 / 28 / 29, 33) and past one CTA per SM (147 / 148 / 149): every env against the
    oracle, after a one-decision and a three-decision launch."""
    kw, nf = SHAPE_CFGS[which]
    cfg = lay.derive_config(event_cap=64, **kw)
    for n in (1, 2, 27, 28, 29, 33, 147, 148, 149):
        b, oras = make(cfg, n, W, seed=21, first=1000)
        assert b.tile_width == W
        assert_equal_to_oracle(b, oras, rollout_both(b, oras, nf, 0, 1), "%d envs, decision 0" % n)
        assert_equal_to_oracle(b, oras, rollout_both(b, oras, nf, 1, 3), "%d envs, decisions 1-3" % n)
        assert b.observer_launch_count == 2, n
        b.close()


def uses_observers(cfg, n, W, nf):
    from aigar_b200.env import AgarBatch
    b = AgarBatch(cfg, n, seed=1, tile_width=W)
    b.rollout_random(1, nf, 0)
    used = b.observer_launch_count == 1
    b.close()
    return used


def one_wave_edge(cfg, W, nf, sms):
    """(last env count one observer wave holds, the next one).  plan_observers gives a CTA at most `full` envs and the
    device fits `occ` such CTAs per SM: the wave holds sms * occ * full envs.  occ is what the occupancy query inside the
    library reports, read back as the smallest k at which sms * k * full + 1 envs leave the observer launch."""
    full = (OBS_MAX_THREADS[W] // 32 - OBS_WARPS) * (32 // W)
    for occ in (1, 2, 3, 4):
        n = sms * occ * full
        if not uses_observers(cfg, n + 1, W, nf):
            return n, n + 1
    pytest.fail("observer launches at every probed wave edge (W = %d)" % W)


def cdiv(a, b):
    return -(-a // b)


def envs_per_cta(n, W, sms, observers):
    """plan_observers' CTA size, or the inline launch's (128 threads)."""
    if not observers:
        return 128 // W
    per_warp = 32 // W
    warps = min(cdiv(cdiv(n, sms), per_warp), OBS_MAX_THREADS[W] // 32 - OBS_WARPS)
    return warps * per_warp


@pytest.mark.parametrize("W", [4, 8])
@pytest.mark.parametrize("which", sorted(SHAPE_CFGS))
def test_observer_wave_edge(torch_cuda, which, W):
    """The last env count one observer wave holds and the first past it: state and observations bit for bit against the same
    rollout at W = 2 (inline encoder), and env 0, the first env of the last CTA and the last env against the oracle."""
    torch = torch_cuda
    from oracle import oracle as orc
    from aigar_b200.env import AgarBatch
    kw, nf = SHAPE_CFGS[which]
    cfg = lay.derive_config(event_cap=64, **kw)
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    pair = one_wave_edge(cfg, W, nf, sms)
    if sms == 148 and W == 8:
        assert pair == (4144, 4145)  # 28 envs per CTA, one CTA per SM
    seed, first, n_dec = 5, 20000, 6
    for n, expect in zip(pair, (True, False)):
        a = AgarBatch(cfg, n, seed=seed, first_env_id=first, tile_width=W)
        c = AgarBatch(cfg, n, seed=seed, first_env_id=first, tile_width=2)
        oa = a.rollout_random(n_dec, nf, 0)
        oc = c.rollout_random(n_dec, nf, 0)
        used = a.observer_launch_count == 1
        if sms == 148:
            assert used == expect, n
        assert c.observer_launch_count == 0
        assert torch.equal(a.state_tensor(), c.state_tensor()), n
        assert torch.equal(oa, oc), n
        per = envs_per_cta(n, W, sms, used)
        envs = [0, (n - 1) // per * per, n - 1]
        oras = {i: orc.OracleEnv(cfg, seed=seed, env_id=first + i, portable=True) for i in envs}
        for e in oras.values():
            e.rollout_random(n_dec, nf, 0)
        assert_equal_to_oracle(a, oras, oa, "%d envs" % n, envs=envs)
        a.close()
        c.close()


# ---------------------------------------------------------------- (d) configs without a pellet grid
NO_GRID = {"both": dict(use_fovsize=1, use_totalmass=1), "fov": dict(use_fovsize=1, use_totalmass=0),
           "none": dict(use_fovsize=0, use_totalmass=0)}


@pytest.mark.parametrize("extras", sorted(NO_GRID))
def test_no_pellet_grid_runs_general_kernel(torch_cuda, extras):
    """A single-cell config without a pellet grid is not k_simple's (its encoder always writes the G x G grid): the general
    kernel runs it, rows of state_len = number of extras (0 included) equal the oracle's."""
    from aigar_b200.env import AgarError
    kw = dict(overrides=dict(pellet_grid=0, **NO_GRID[extras]))
    cfg = lay.derive_config(event_cap=64, **kw)
    b, oras = make(cfg, 8, None, seed=17, first=60)
    assert b.layout.state_len == sum(NO_GRID[extras].values())
    assert b.tile_width == 32
    with pytest.raises(AgarError):
        b.set_tile_width(1)
    assert b.tile_width == 32
    assert gpu_check.check(kw, n_envs=8, frames=80, seed=17, first_env=60, verbose=False)
    b, launches = run_rollout(cfg, None, 8, 8, seed=18, first=90, frames=80)
    assert b.observer_launch_count == 0
