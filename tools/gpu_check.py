"""GPU vs portable-math oracle, record by record (run on a GPU box).  Prints the first divergence."""
import os, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch
import aigar_b200.layout as lay
from aigar_b200.env import AgarBatch
from oracle import oracle as orc

KWS = {"1": dict(), "3": dict(num_nn=1, num_greedy=1, virus=True, split=True, eject=True),
       "4": dict(num_nn=8, num_greedy=8, virus=True, split=True, eject=True),
       "r": dict(num_nn=1, num_greedy=1, num_random=1, virus=True, split=True, eject=True),
       "4nv": dict(num_nn=8, num_greedy=8, virus=False, split=True, eject=True),
       # AGAR_OBS_CANONICAL: robust observation binning (exact floors, always G columns)
       "1c": dict(obs_mode=1), "3c": dict(num_nn=1, num_greedy=1, virus=True, split=True, eject=True, obs_mode=1),
       "4c": dict(num_nn=8, num_greedy=8, virus=True, split=True, eject=True, obs_mode=1)}


def records(batch):
    st = batch.state_tensor().cpu().numpy()
    return [lay.Record(batch.layout, st[i].copy()) for i in range(batch.n_envs)]


def check(which="1", n_envs=32, frames=200, seed=3, first_env=5, tile_width=None, every=1, event_cap=64, verbose=True, tally=None,
          setup=None):
    """tally: dict that receives the event-type counts of the ORACLE's per-frame event logs (all envs, all frames).
    setup: setup(batch, oracles) runs once before the first comparison, e.g. to load the same records into both."""
    cfg = lay.derive_config(event_cap=event_cap, **(which if isinstance(which, dict) else KWS[which]))
    batch = AgarBatch(cfg, n_envs, seed=seed, first_env_id=first_env, tile_width=tile_width)
    L = batch.layout
    oras = [orc.OracleEnv(cfg, seed=seed, env_id=first_env + i, portable=True) for i in range(n_envs)]
    A = max(L.n_agents, 1)
    rng = np.random.default_rng(seed)
    bad = []
    if setup is not None:
        setup(batch, oras)

    def cmp(tag):
        recs = records(batch)
        for i in range(n_envs):
            d = lay.compare_records(oras[i].record, recs[i], what="%s env %d " % (tag, i), check_events=True)
            if d:
                bad.extend(d[:6])
                bad.append("oracle events: %r" % (oras[i].record.event_list()[:12],))
                bad.append("gpu    events: %r" % (recs[i].event_list()[:12],))
                return False
        return True

    if not cmp("init"):
        print("\n".join(bad)); return False
    for t in range(frames):
        act = rng.random((n_envs, A, 4)).astype(np.float32)
        obs = batch.observe().cpu().numpy()
        need = batch.get(lay.GET_NEED_ACTION).cpu().numpy()
        valid = batch.get(lay.GET_VALID).cpu().numpy()
        done = batch.get(lay.GET_DONE).cpu().numpy()
        rew = batch.get(lay.GET_REWARD).cpu().numpy()
        for i in range(n_envs):
            tr = oras[i].observe()
            for a in range(L.n_agents):
                if (bool(need[i, a]), bool(valid[i, a]), bool(done[i, a])) != (tr[a]["need_action"], tr[a]["valid"], tr[a]["done"]):
                    bad.append("frame %d env %d agent %d turn flags differ: gpu %r oracle %r" % (
                        t, i, a, (need[i, a], valid[i, a], done[i, a]), (tr[a]["need_action"], tr[a]["valid"], tr[a]["done"])))
                if rew[i, a] != np.float32(tr[a]["reward"]):
                    bad.append("frame %d env %d agent %d reward %r != %r" % (t, i, a, rew[i, a], tr[a]["reward"]))
                if tr[a]["obs32"] is not None:
                    neq = obs[i, a] != tr[a]["obs32"]
                    if neq.any():
                        j = int(np.argwhere(neq)[0][0])
                        bad.append("frame %d env %d agent %d obs[%d]: gpu %r oracle %r (%d bad)" % (
                            t, i, a, j, obs[i, a, j], tr[a]["obs32"][j], int(neq.sum())))
            oras[i].step(act[i], 1)
            if tally is not None:
                rec = oras[i].record
                n = min(int(rec.header["n_events"][0]), L.event_cap)
                if n:
                    for typ, cnt in zip(*np.unique(rec.events["type"][:n], return_counts=True)):
                        tally[lay.EV_NAMES[int(typ)]] = tally.get(lay.EV_NAMES[int(typ)], 0) + int(cnt)
        batch.step(act, 1)
        if bad or ((t + 1) % every == 0 and not cmp("frame %d" % t)):
            print("\n".join(bad[:30])); return False
    if not cmp("final"):
        print("\n".join(bad[:30])); return False
    if verbose:
        print("OK config %s: %d envs x %d frames bit-exact (W=%d)" % (which if not isinstance(which, dict) else "custom", n_envs, frames, batch.tile_width))
    return True


if __name__ == "__main__":
    which = sys.argv[1] if len(sys.argv) > 1 else "1"
    n_envs = int(sys.argv[2]) if len(sys.argv) > 2 else 32
    frames = int(sys.argv[3]) if len(sys.argv) > 3 else 200
    tw = int(sys.argv[4]) if len(sys.argv) > 4 else None
    t0 = time.time()
    ok = check(which, n_envs, frames, tile_width=tw, every=int(os.environ.get("EVERY", "1")))
    print("elapsed %.1fs" % (time.time() - t0))
    sys.exit(0 if ok else 1)
