"""Throughput sweep of the pellet-collection config over env counts and tile widths (run on a GPU box)."""
import os, sys, json
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import aigar_b200.layout as lay
from aigar_b200.env import AgarBatch

KWS = {"1": dict(), "3": dict(num_nn=1, num_greedy=1, virus=True, split=True, eject=True),
       "4": dict(num_nn=8, num_greedy=8, virus=True, split=True, eject=True)}


def measure(E, W, decisions=25, reps=3, write_obs=True, which="1"):
    cfg = lay.derive_config(**KWS[which])
    b = AgarBatch(cfg, E, seed=1, tile_width=W)
    b.rollout_random(decisions, 8, 0, write_obs=write_obs)
    torch.cuda.synchronize()
    best = 1e9
    for i in range(reps):
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record(); b.rollout_random(decisions, 8, (i + 1) * decisions, write_obs=write_obs); e.record(); torch.cuda.synchronize()
        best = min(best, s.elapsed_time(e))
    b.close()
    return E * decisions * 8 / (best * 1e-3), best

if __name__ == "__main__":
    Es = [int(x) for x in (sys.argv[1] if len(sys.argv) > 1 else "4096,65536,1048576").split(",")]
    Ws = [int(x) for x in (sys.argv[2] if len(sys.argv) > 2 else "1,4,8,32").split(",")]
    which = sys.argv[3] if len(sys.argv) > 3 else "1"
    for E in Es:
        for W in Ws:
            dec = (125 if E <= 16384 else 25) if which == "1" else 12
            v, ms = measure(E, W, decisions=dec, which=which)
            print(json.dumps({"config": which, "envs": E, "tile": W, "env_steps_per_s": v, "ms": ms, "frames": dec * 8}), flush=True)
