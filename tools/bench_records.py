"""Bandwidth of the state-snapshot calls (agar_load_records / agar_save_records through AgarBatch.restore / snapshot) against
torch's device-to-device copy_ of the same bytes, on one GPU.  CUDA events; every timed call is warmed up first.  Bytes
moved = 2 x n_envs x record_bytes (one read, one write); the card's name and power limit are read in the same run.

The pellet config's banks (3.7 MB at 4096 envs, 59 MB at 65 536) fit the 126 MB L2 and are reported as they are; the
1-vs-greedy (147 MB) and arena (497 MB) banks do not.

    python tools/bench_records.py [--reps-bytes 2e10] > profiles/r04_bench_records.json
"""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import torch  # noqa: E402

import aigar_b200.layout as lay  # noqa: E402
from aigar_b200.env import AgarBatch  # noqa: E402

SHAPES = [("pellet", dict(), 4096), ("pellet", dict(), 65536),
          ("1-vs-greedy", dict(num_nn=1, num_greedy=1, virus=True, split=True, eject=True), 16384),
          ("arena", dict(num_nn=8, num_greedy=8, virus=True, split=True, eject=True), 8192)]


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    name, power, clock = [s.strip() for s in q.stdout.strip().splitlines()[0].split(",")]
    return {"gpu": name, "power_limit": power, "max_sm_clock": clock}


def time_call(fn, reps, rounds=5):
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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps-bytes", type=float, default=2e10, help="bytes each timed round moves per measurement")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_records needs a CUDA device")
    info = card()
    print(json.dumps(dict(info, what="card")))
    for name, kw, n in SHAPES:
        b = AgarBatch(lay.derive_config(**kw), n, seed=1)
        rb = int(b.layout.record_bytes)
        moved = 2 * n * rb
        reps = max(10, int(args.reps_bytes / moved))
        bank = b.snapshot()
        out = torch.empty_like(bank)
        perm = torch.randperm(n, device=b.device).to(torch.int32)
        src, dst = bank.clone(), torch.empty_like(bank)
        t = {"restore": time_call(lambda: b.restore(bank), reps),
             "restore_permuted": time_call(lambda: b.restore(bank, perm), reps),
             "snapshot": time_call(lambda: b.snapshot(out=out), reps),
             "copy_": time_call(lambda: dst.copy_(src), reps)}
        assert b.record_error_flags() == 0
        row = {"what": "records", "config": name, "n_envs": n, "record_bytes": rb, "bank_mb": round(n * rb / 1e6, 1),
               "reps": reps, "gpu": info["gpu"], "power_limit": info["power_limit"]}
        for k, v in t.items():
            row[k + "_us"] = round(v * 1e6, 2)
            row[k + "_gbps"] = round(moved / v / 1e9, 1)
        for k in ("restore", "restore_permuted", "snapshot"):
            row[k + "_vs_copy"] = round(t["copy_"] / t[k], 3)
        print(json.dumps(row), flush=True)
        del b, bank, out, src, dst
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
