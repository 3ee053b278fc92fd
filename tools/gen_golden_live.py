"""Record tests/golden/live/*.npz: what tests/test_oracle_vs_reference.py, tests/test_replay.py and tests/test_results.py compare
against, on exactly the inputs those tests drive, so that they run without the reference's sources.

python tools/gen_golden_live.py [--source reference|oracle] [NAME ...]

--source reference (the default) executes the unmodified reference (NILOIDE/A.I.gar, AGAR_REF_SRC) through
oracle/ref_harness.py.  --source oracle records the repository's restatements instead (oracle/agar_oracle.c libm build,
oracle/replay_oracle.py, aigar_b200.results): the committed files were recorded that way at the commit where the live
comparison of these restatements with the reference passed on these same inputs (VERDICT.md, round 2).  Every file carries its
source.  Env cases hold the actions, the env record (with its event log) every few frames, the event hash, event count and
event list of every frame, every agent's turn flags every frame and every float32 observation."""
import argparse
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import numpy as np  # noqa: E402

import aigar_b200.layout as lay  # noqa: E402

OUT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden", "live")
KWS = {"1": dict(), "3": dict(num_nn=1, num_greedy=1, virus=True, split=True, eject=True),
       "4": dict(num_nn=8, num_greedy=8, virus=True, split=True, eject=True),
       "r": dict(num_nn=1, num_greedy=1, num_random=1, virus=True, split=True, eject=True),
       "4nv": dict(num_nn=8, num_greedy=8, virus=False, split=True, eject=True)}
ORACLE_CASES = [("1", 400, 11), ("1", 250, 12), ("3", 500, 13), ("r", 300, 14), ("4", 40, 15), ("4nv", 30, 16)]
VARIATIONS = [
    dict(mass_as_reward=True),
    dict(frame_skip=3, reward_scale=1.0, reward_term=0.5),
    dict(grid=7),
    dict(grid=13, num_nn=1, num_greedy=1),
    dict(num_nn=2, num_random=1, split=True),                      # two agents, a random bot, split without eject
    dict(num_nn=1, num_greedy=2, virus=True),                      # viruses without split: explosions only
    dict(num_nn=1, num_greedy=1, virus=True, split=True, eject=True, death_term=-10.0, death_factor=0.5),
    dict(num_nn=3, num_greedy=1, split=True, eject=True, obs_mode=1),
    dict(overrides={"use_second_last_action": 1, "self_grid_slf": 1, "enemy_grid_slf": 1}, num_nn=1, num_greedy=1,
         virus=True, split=True, eject=True),
    dict(grid=42, overrides={"use_fovsize": 0, "use_totalmass": 0}),   # the handcraft-CNN grid (bot.py:103-111), §8f rank 3
    dict(grid=42, num_nn=1, num_greedy=1, virus=True, split=True, eject=True),
    dict(grid=63),
    dict(grid=84, overrides={"use_fovsize": 0, "use_totalmass": 0}),   # CNN_INPUT_DIM_2
    # ALL_PLAYER_GRID (networkParameters.py:88-91): one "biggest cell of any player" channel instead of self / enemy
    dict(num_nn=1, num_greedy=1, virus=True, split=True, eject=True, overrides={"all_player_grid": 1, "self_grid": 0, "enemy_grid": 0, "self_grid_lf": 0, "enemy_grid_lf": 0}),
    dict(overrides={"all_player_grid": 1}),
    # NORMALIZE_GRID_BY_MAX_MASS in the run's parameters (bot.py:365,412,422,430): cell channels relative to the biggest cell in view
    dict(num_nn=2, num_greedy=1, virus=True, split=True, eject=True, overrides={"normalize_grid_by_max_mass": 1}),
    dict(num_nn=1, num_greedy=1, split=True, overrides={"normalize_grid_by_max_mass": 1, "all_player_grid": 1, "self_grid": 0, "enemy_grid": 0,
                                                        "self_grid_lf": 0, "enemy_grid_lf": 0}),
    # GRID_VIEW_ENABLED = False (networkParameters.py:119): Bot.getSimpleStateRepresentation, bot.py:511-548
    dict(grid_view=False),
    dict(num_nn=1, num_greedy=1, virus=True, split=True, eject=True, grid_view=False),
    dict(num_nn=2, num_greedy=3, split=True, eject=True, grid_view=False, frame_skip=2),
]
FUZZ_N, FUZZ_SEED = 6, 23


def variation_frames(kw):
    frames = 160 if kw.get("num_nn", 1) + kw.get("num_greedy", 0) + kw.get("num_random", 0) <= 2 else 90
    return 48 if kw.get("grid", 11) >= 42 else frames  # the reference's encoder is O(G^2) Python per observation


class _Driver(object):
    """One env of either source behind the interface the recorder needs: frame(actions) -> turn, record, reset()."""

    def __init__(self, source, cfg, seed, env_id):
        if source == "reference":
            from oracle import ref_harness as rh
            self.env, self.ref = rh.RefEnv(cfg, seed=seed, env_id=env_id), True
        else:
            from oracle import oracle as orc
            self.env, self.ref = orc.OracleEnv(cfg, seed=seed, env_id=env_id), False
        self.turn = None

    def frame(self, actions):
        if self.ref:
            self.turn = self.env.step(actions)
            return [dict(t, obs32=None if t["obs"] is None else t["obs"].astype(np.float32)) for t in self.turn]
        return self.env.frame(actions)

    def record(self):
        return self.env.to_record(self.turn) if self.ref else lay.Record(self.env.layout, self.env.record.buf.copy())

    def reset(self):
        self.env.reset()
        self.env.reset_bots()
        self.turn = None


def record_rollout(source, kw, frames, seed, env_id=0, n_records=40):
    """The rollout of tools/compare_oracle_ref.run (event_cap 512, actions from default_rng(seed * 1000 + env_id))."""
    cfg = lay.derive_config(event_cap=512, **kw)
    drv = _Driver(source, cfg, seed, env_id)
    L = lay.layout_for_config(cfg)
    A = max(L.n_agents, 1)
    rng = np.random.default_rng(seed * 1000 + env_id)
    every = max(1, frames // n_records)
    recs, rec_frames = [drv.record().buf.copy()], [-1]
    actions, flags, hashes, n_events, events, obs, obs_idx = [], np.zeros((frames, A), np.uint8), [], [], [], [], []
    for t in range(frames):
        act = rng.random((A, 4)).astype(np.float32)
        actions.append(act)
        turn = drv.frame(act)
        rec = drv.record()
        for a in range(L.n_agents):
            flags[t, a] = (int(turn[a]["observed"]) | int(turn[a]["valid"]) << 1 | int(turn[a]["done"]) << 2 |
                           int(turn[a]["need_action"]) << 3 | int(turn[a]["obs32"] is not None) << 4)
            if turn[a]["obs32"] is not None:
                obs.append(turn[a]["obs32"])
                obs_idx.append((t, a))
        hashes.append(int(rec.header["event_hash"][0]))
        n_events.append(int(rec.header["n_events"][0]))
        events.extend(rec.event_list())
        if (t + 1) % every == 0 or t == frames - 1:
            recs.append(rec.buf.copy())
            rec_frames.append(t)
    return dict(kw=np.array(repr(kw)), seed=seed, env_id=env_id, event_cap=512, actions=np.stack(actions), flags=flags,
                records=np.stack(recs), record_frames=np.array(rec_frames, np.int32), event_hash=np.array(hashes, np.uint64),
                n_events=np.array(n_events, np.int32), events=np.array(events, np.int64).reshape(-1, 5),
                obs=np.stack(obs) if obs else np.zeros((0, L.state_len), np.float32),
                obs_index=np.array(obs_idx, np.int32).reshape(-1, 2))


def record_reset(source):
    """test_reset_matches_reference: 120 frames, reset + reset_bots, 60 frames."""
    cfg = lay.derive_config(num_nn=1, num_greedy=1, virus=True, split=True, eject=True, event_cap=256)
    drv = _Driver(source, cfg, 5, 1)
    rng = np.random.default_rng(0)
    for t in range(120):
        drv.frame(rng.random((1, 4)).astype(np.float32))
    drv.reset()
    after_reset = drv.record().buf.copy()
    for t in range(60):
        drv.frame(rng.random((1, 4)).astype(np.float32))
    return dict(after_reset=after_reset, after_reset_60=drv.record().buf.copy())


def record_views(source):
    """test_views_show_what_the_reference_objects_show: the View getters after 150 frames of the 1-vs-greedy config."""
    from aigar_b200.views import FieldView
    cfg = lay.derive_config(num_nn=1, num_greedy=1, virus=True, split=True, eject=True)
    drv = _Driver(source, cfg, 9, 2)
    rng = np.random.default_rng(1)
    for t in range(150):
        drv.frame(rng.random((1, 4)).astype(np.float32))
    f = drv.env.field if drv.ref else FieldView(drv.env.record)
    out = dict(size=np.array([f.getWidth(), f.getHeight()], np.float64))
    for name in ("Pellets", "Viruses", "Blobs", "PlayerCells"):
        out[name] = view_cells(getattr(f, "get" + name)())
    players, cells = [], []
    for k, p in enumerate(f.getPlayers()):
        players.append((float(p.getIsAlive()), float(len(p.getCells())), p.getTotalMass()))
        cells.extend([k] + list(c.getPos()) + [c.getMass(), c.getRadius()] for c in p.getCells())
    out["players"], out["player_cells"] = np.array(players, np.float64), np.array(cells, np.float64).reshape(-1, 5)
    p0 = f.getPlayers()[0]
    if p0.getIsAlive():
        pos, size = p0.getFovPos(), p0.getFovSize()
        out["fov"] = np.array(list(pos) + [size], np.float64)
        out["PelletsInFov"] = view_cells(f.getPelletsInFov(pos, size))
    return out


def view_cells(cells):
    """(x, y, mass, radius) rounded to 9 decimals, sorted: the key the views test compares."""
    return np.array(sorted((round(c.getX(), 9), round(c.getY(), 9), round(c.getMass(), 9), round(c.getRadius(), 9)) for c in cells),
                    np.float64).reshape(-1, 4)


def replay_transitions(n, L, rng):
    return [(rng.random(L).astype(np.float32), rng.random(4).astype(np.float32), float(np.float32(rng.normal())),
             rng.random(L).astype(np.float32), bool(rng.random() < 0.1)) for _ in range(n)]


def record_replay(source, prioritized):
    """test_oracle_equals_reference_replay_buffer: 12 rounds of adds, 8 injected uniforms per sample, priority updates.  states:
    per round length and next index, and for the prioritized buffer the max priority and both segment trees after the adds and
    again after the update; samples: per sampling round the 8 rows of (obs, action, reward, next obs, done, index[, weight])."""
    size, L = 37, 6
    if source == "reference":
        import importlib
        from oracle import ref_harness as rh
        sys.path.insert(0, rh.REF_SRC)
        rb = importlib.import_module("model.replay_buffer")
        feed = []

        class _R(object):  # the injected stdlib random
            @staticmethod
            def randint(a, b):
                return min(a + int(feed.pop(0) * (b - a + 1)), b)

            @staticmethod
            def random():
                return feed.pop(0)

        rb.random = _R
        buf = rb.PrioritizedReplayBuffer(size, 0.6, 0.4) if prioritized else rb.ReplayBuffer(size)

        def sample(u):
            feed[:] = list(u)
            return buf.sample(8)
        state = lambda: (len(buf), buf._next_idx) + ((buf._max_priority,) + tuple(buf._it_sum._value) + tuple(buf._it_min._value)
                                                    if prioritized else ())
    else:
        from oracle.replay_oracle import ReplayOracle
        buf = ReplayOracle(size, prioritized, 0.6, 0.4)
        sample = buf.sample
        state = lambda: (len(buf), buf.next_idx) + ((buf.max_priority,) + tuple(buf.sum) + tuple(buf.min) if prioritized else ())
    rng = np.random.default_rng(3)
    states, samples = [], []
    for rnd in range(12):
        for tr in replay_transitions(int(rng.integers(3, 15)), L, rng):
            buf.add(*tr)
        states.append(state())
        if states[-1][0] < 4:
            continue
        out = sample([float(x) for x in rng.random(8)])
        idxes = list(out[6] if prioritized else out[5])
        row = [np.asarray(out[0], np.float64).reshape(8, -1), np.asarray(out[1], np.float64).reshape(8, -1),
               np.asarray(out[2], np.float64).reshape(8, 1), np.asarray(out[3], np.float64).reshape(8, -1),
               np.asarray(out[4], np.float64).reshape(8, 1), np.array(idxes, np.float64).reshape(8, 1)]
        if prioritized:
            row.append(np.asarray(out[5], np.float64).reshape(8, 1))
            buf.update_priorities(idxes, np.abs(rng.normal(size=8)) + 1e-4)
            states[-1] = states[-1] + state()[2:]
        samples.append(np.concatenate(row, axis=1))
    n = max(len(s) for s in states)
    return dict(states=np.array([list(s) + [np.nan] * (n - len(s)) for s in states], np.float64), samples=np.stack(samples))


EXPORT_VALUES = [123.456, 99.0, 1e-3, 250.12345678901234]


def record_export(source):
    """test_against_the_reference_functions: the file exportResults writes for EXPORT_VALUES under the name "m"."""
    import tempfile
    if source == "reference":
        from oracle import ref_harness as rh
        src = open(os.path.join(rh.REF_SRC, "aigar.py")).read()
        ns = {}
        exec(src[src.index("def exportResults(results, path, name):"):
                 src.index("# Plot test result and export plot to file with given name")], ns)
        fn = ns["exportResults"]
    else:
        from aigar_b200 import results as res
        fn = res.export_results
    with tempfile.TemporaryDirectory() as tmp:
        fn(EXPORT_VALUES, tmp + os.sep, "m")
        return open(os.path.join(tmp, "m.txt")).read()


def targets():
    from fuzz_oracle_ref import cases
    out = {"oracle_%s_%d" % (w, s): (lambda src, w=w, f=f, s=s: record_rollout(src, KWS[w], f, s)) for w, f, s in ORACLE_CASES}
    for i, kw in enumerate(VARIATIONS):
        out["variation_%d" % i] = lambda src, kw=kw: record_rollout(src, kw, variation_frames(kw), 31)
    for case, kw, frames, seed in cases(FUZZ_N, FUZZ_SEED):
        out["fuzz_%d" % case] = lambda src, kw=kw, f=frames, s=seed: record_rollout(src, kw, f, s)
    out["reset"] = record_reset
    out["views"] = record_views
    out["replay_uniform"] = lambda src: record_replay(src, False)
    out["replay_prioritized"] = lambda src: record_replay(src, True)
    out["export_results"] = lambda src: dict(values=np.array(EXPORT_VALUES), text=np.array(record_export(src)))
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--source", choices=("reference", "oracle"), default="reference")
    ap.add_argument("names", nargs="*")
    args = ap.parse_args()
    os.makedirs(OUT, exist_ok=True)
    for name, fn in targets().items():
        if args.names and name not in args.names:
            continue
        path = os.path.join(OUT, name + ".npz")
        np.savez_compressed(path, source=np.array(args.source), **fn(args.source))
        print(name, os.path.getsize(path), "bytes")


if __name__ == "__main__":
    main()
