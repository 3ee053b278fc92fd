"""Cost of recording rollouts (agar_rollout through AgarBatch.rollout) at the BASELINE.json bench shapes, on one GPU, with CUDA
events; every timed call is warmed up first and the card's name, power limit and max SM clock are read in the same run.

Per shape (configs[1]: 4096 envs, configs[2]: 16 384, configs[3]: 8192; 125 decisions x 8 frames):
  - rollout: agar_rollout recording every field, against agar_rollout_random writing each decision's observation into one
    [E, A, L] buffer (`random_obs`) and without observations (`random_no_obs`);
  - replay fill: random transitions into a prioritized GpuReplayBuffer, one D-decision rollout + add_trajectory against
    D x (rollout_random(1) + observe + three agar_get + add_batch), in env-steps/s, median and spread over the rounds.
configs[3]'s trajectory is about 224 MB per decision; its rows use fewer decisions (`decisions` says how many).

    python tools/bench_trajectory.py [--out profiles/r05_bench_trajectory.json]
"""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import torch  # noqa: E402

import aigar_b200.layout as lay  # noqa: E402
from aigar_b200.env import AgarBatch, Trajectory  # noqa: E402
from aigar_b200.replay import GpuReplayBuffer  # noqa: E402

# (name, derive_config arguments, envs, decisions)
SHAPES = [("configs[1]", dict(), 4096, 125),
          ("configs[2]", dict(num_nn=1, num_greedy=1, virus=True, split=True, eject=True), 16384, 125),
          ("configs[3]", dict(num_nn=8, num_greedy=8, virus=True, split=True, eject=True), 8192, 25)]
FRAMES = 8
ROUNDS = 7


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    name, power, clock = [s.strip() for s in q.stdout.strip().splitlines()[0].split(",")]
    return {"gpu": name, "power_limit": power, "max_sm_clock": clock}


def times(fn, rounds=ROUNDS):
    """seconds per call over `rounds` timed calls, after two warm-up calls"""
    for _ in range(2):
        fn()
    torch.cuda.synchronize()
    out = []
    for _ in range(rounds):
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0.record()
        fn()
        t1.record()
        t1.synchronize()
        out.append(t0.elapsed_time(t1) / 1e3)
    return sorted(out)


def stats(ts, steps):
    med = ts[len(ts) // 2]
    return {"median_s": round(med, 6), "min_s": round(ts[0], 6), "max_s": round(ts[-1], 6),
            "env_steps_per_s": float("%.4g" % (steps / med)), "spread": round((ts[-1] - ts[0]) / med, 4)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "profiles",
                                                  "r05_bench_trajectory.json"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_trajectory needs a CUDA device")
    info = card()
    rows = [dict(info, what="card")]
    print(json.dumps(rows[-1]), flush=True)
    for name, kw, n, D in SHAPES:
        cfg = lay.derive_config(**kw)
        b = AgarBatch(cfg, n, seed=1)
        b.rollout_random(4, FRAMES, 0)
        bank = b.snapshot()
        A, L = max(b.layout.n_agents, 1), b.layout.state_len
        steps = n * D * FRAMES
        traj = Trajectory.allocate(b, D)

        def run(fn):  # every timed call starts from the same records
            def go():
                b.restore(bank)
                fn()
            return go
        t = {"rollout": times(run(lambda: b.rollout(D, FRAMES, 0, out=traj))),
             "random_obs": times(run(lambda: b.rollout_random(D, FRAMES, 0))),
             "random_no_obs": times(run(lambda: b.rollout_random(D, FRAMES, 0, write_obs=False))),
             "restore": times(lambda: b.restore(bank))}
        row = {"what": "rollout", "config": name, "n_envs": n, "decisions": D, "frames": FRAMES,
               "trajectory_mb": round(sum(x.numel() * x.element_size() for x in traj[:6]) / 1e6, 1),
               "gpu": info["gpu"], "power_limit": info["power_limit"],
               "note": "each timed call is restore + the call; restore_s is the restore alone"}
        for k, v in t.items():
            row[k] = stats(v, steps)
        rest = t["restore"][len(t["restore"]) // 2]
        for k in ("random_obs", "random_no_obs"):
            row["rollout_vs_" + k] = round((row["rollout"]["median_s"] - rest) / (row[k]["median_s"] - rest), 4)
        print(json.dumps(row), flush=True)
        rows.append(row)
        del traj

        # replay fill: one bot turn per decision (frame_skip + 1 frames), as the per-tick training loops step
        F = cfg.frame_skip + 1
        Dr = min(D, 25)
        rb = GpuReplayBuffer(2 * n * A * Dr, L, 4, prioritized=True, device=b.device.index)
        tr = Trajectory.allocate(b, Dr, ("obs", "action", "reward", "done", "valid"))
        prev = torch.empty_like(b.obs)

        def fused():
            rb.add_trajectory(b.rollout(Dr, F, 0, out=tr))

        def per_tick():
            b.observe()
            for d in range(Dr):
                prev.copy_(b.obs)
                b.rollout_random(1, F, d, write_obs=False)
                b.observe()
                rb.add_batch(prev, b.actions, b.get(lay.GET_REWARD), b.obs, b.get(lay.GET_DONE), b.get(lay.GET_VALID))
        r = {"fused": times(run(fused)), "per_tick": times(run(per_tick))}
        row = {"what": "replay_fill", "config": name, "n_envs": n, "decisions": Dr, "frames": F,
               "transitions_per_call": n * A * Dr, "gpu": info["gpu"], "power_limit": info["power_limit"],
               "note": "per_tick stores b.actions (zeros) as its action column: the random actions are not exposed there"}
        for k, v in r.items():
            row[k] = stats(v, n * Dr * F)
        row["fused_speedup"] = round(row["per_tick"]["median_s"] / row["fused"]["median_s"], 3)
        print(json.dumps(row), flush=True)
        rows.append(row)
        rb.close()
        del b, bank, tr, rb
        torch.cuda.empty_cache()
    with open(args.out, "w") as f:
        for row in rows:
            f.write(json.dumps(row) + "\n")


if __name__ == "__main__":
    main()
