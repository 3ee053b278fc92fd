"""Bandwidth of the replay-buffer state snapshots (agar_replay_save / agar_replay_load through GpuReplayBuffer.snapshot /
restore) against torch's device-to-device copy_ of the same bytes, for full prioritized buffers on one GPU.  CUDA events,
median of 7 rounds, every timed call warmed up first.  Bytes moved = 2 x state_bytes (one read, one write); the card's name,
power limit and max SM clock are read in the same run.

A restore is a validation pass, the install copy and the rebuild of both trees; `restore_refused` times the same call on a
bank the device refuses (validation, an install that copies nothing, the rebuild), i.e. the part of a restore that is not the
copy.  The 2^20 x 123 (the example's buffer) and 2^20 x 854 (the 1-vs-greedy state length) banks do not fit the 126 MB L2; the
2^14 x 123 bank does and is reported as it is.

    python tools/bench_replay_state.py > profiles/r06_bench_replay_state.json
"""
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import torch  # noqa: E402

from aigar_b200.replay import GpuReplayBuffer  # noqa: E402

SHAPES = [(1 << 14, 123), (1 << 20, 123), (1 << 20, 854)]  # (capacity, state_len); action_len 1 as examples/train_dqn.py


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    name, power, clock = [s.strip() for s in q.stdout.strip().splitlines()[0].split(",")]
    return {"gpu": name, "power_limit": power, "max_sm_clock": clock}


def time_call(fn, reps, rounds=7):
    """median over `rounds` of the mean time of `reps` back-to-back calls, in seconds"""
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    times = []
    for _ in range(rounds):
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0.record()
        for _ in range(reps):
            fn()
        t1.record()
        t1.synchronize()
        times.append(t0.elapsed_time(t1) / 1e3 / reps)
    return sorted(times)[rounds // 2]


def filled(cap, L):
    rp = GpuReplayBuffer(cap, L, 1, prioritized=True, alpha=0.6, beta=0.4)
    g = torch.Generator(device="cuda").manual_seed(0)
    chunk = min(cap, 1 << 16)
    obs = torch.rand((chunk, L), device="cuda", generator=g)
    for k in range(cap // chunk):
        rp.add_batch(obs + k, torch.rand((chunk, 1), device="cuda", generator=g), torch.rand(chunk, device="cuda", generator=g),
                     obs - k, torch.zeros(chunk, dtype=torch.uint8, device="cuda"))
        idx = torch.randint(0, len(rp), (2048,), device="cuda", generator=g).to(torch.int32)
        rp.update_priorities(idx, torch.rand(2048, dtype=torch.float64, device="cuda", generator=g) + 1e-4)
    assert len(rp) == cap
    return rp


def main():
    if not torch.cuda.is_available():
        sys.exit("bench_replay_state needs a CUDA device")
    info = card()
    print(json.dumps(dict(info, what="card")), flush=True)
    for cap, L in SHAPES:
        rp = filled(cap, L)
        n = rp.state_bytes
        moved = 2 * n
        reps = max(10, int(2e10 / moved))
        bank, out = rp.snapshot(), torch.empty(n, dtype=torch.uint8, device="cuda")
        refused = bank.clone()
        refused[56:64] = 0xFF  # header size = -1
        src, dst = bank.clone(), torch.empty_like(bank)
        t = {"snapshot": time_call(lambda: rp.snapshot(out=out), reps),
             "restore": time_call(lambda: rp.restore(bank), reps),
             "copy_": time_call(lambda: dst.copy_(src), reps)}
        assert rp.error_flags == 0 and torch.equal(out, bank)
        t["restore_refused"] = time_call(lambda: rp.restore(refused), reps)
        assert torch.equal(rp.snapshot(), bank)
        row = {"what": "replay_state", "capacity": cap, "state_len": L, "bank_mb": round(n / 1e6, 1), "reps": reps,
               "gpu": info["gpu"], "power_limit": info["power_limit"]}
        for k, v in t.items():
            row[k + "_us"] = round(v * 1e6, 2)
            row[k + "_gbps"] = round(moved / v / 1e9, 1)
        for k in ("snapshot", "restore"):
            row[k + "_vs_copy"] = round(t["copy_"] / t[k], 3)
        print(json.dumps(row), flush=True)
        del rp, bank, out, refused, src, dst
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
