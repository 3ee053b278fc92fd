"""What the observation encoder costs the bench rollout: AgarBatch.rollout_random(125, 8) at 4096 envs (--envs) with write_obs=True and
write_obs=False (the kernel still advances the fov caches, it only skips the binning and the row stores), at W = 8 and W = 4;
--fpd 1,2,4,8 times 1000-frame rollouts with an observation every 1 / 2 / 4 / 8 frames instead.
L2 flushed (256 MiB write) before every timed launch, CUDA events, the two arms alternated launch by launch.

Several builds of the library can be compared in the same call: every run is a fresh process with AGAR_B200_LIB pointing at
one of them, and the builds take turns run by run.  Build each with `python a.i.gar_b200/build.py --force` (staleness is
decided by mtime).  Run on a GPU box:

    python tools/ab_rollout_obs.py [--lib NAME=PATH ...] [--runs N] [--reps R] [--fpd F,F,...] [--envs E]"""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

CHILD = r'''
import json, sys, torch
sys.path.insert(0, %r)
import aigar_b200.layout as lay
from aigar_b200.env import AgarBatch
E, REPS, FPDS = %d, %d, %r
flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device="cuda")
out = {}
for W, FPD in [(W, F) for W in (8, 4) for F in FPDS]:
    DEC = 1000 // FPD
    b = AgarBatch(lay.derive_config(), E, seed=2026, tile_width=W)
    for i in range(4):
        b.rollout_random(DEC, FPD, i * DEC, write_obs=bool(i & 1))
    torch.cuda.synchronize()
    ms = {"obs": [], "no_obs": []}
    for i in range(2 * REPS):
        wo = (i & 1) == 0
        flush.fill_(i & 0xff)
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        b.rollout_random(DEC, FPD, (4 + i) * DEC, write_obs=wo)
        e.record()
        torch.cuda.synchronize()
        ms["obs" if wo else "no_obs"].append(s.elapsed_time(e))
    out["W=%%d F=%%d" %% (W, FPD)] = ms
    b.close()
info = {"gpu": torch.cuda.get_device_name(0)}
try:
    import pynvml
    pynvml.nvmlInit()
    h = pynvml.nvmlDeviceGetHandleByIndex(torch.cuda.current_device())
    b = AgarBatch(lay.derive_config(), E, seed=2026)
    b.rollout_random(125, 8, 0)  # the SM clock under this load, read while the launch runs
    info["sm_mhz"] = pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM)
    torch.cuda.synchronize()
    b.close()
    info["power_limit_w"] = pynvml.nvmlDeviceGetPowerManagementLimit(h) / 1000.0
    info["sm_max_mhz"] = pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM)
except Exception as ex:
    info["nvml"] = str(ex)[:100]
print(json.dumps({"ms": out, "info": info}))
'''


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--lib", action="append", default=[], metavar="NAME=PATH",
                    help="a build of libagar_b200.so to time (repeatable; default: the in-tree build)")
    ap.add_argument("--runs", type=int, default=3, help="processes per build, alternated between the builds")
    ap.add_argument("--reps", type=int, default=5, help="timed launches per arm and tile width in each process")
    ap.add_argument("--fpd", default="8", help="frames per decision (comma-separated); 1000 // F decisions per rollout")
    ap.add_argument("--envs", type=int, default=4096)
    args = ap.parse_args()
    libs = [tuple(s.split("=", 1)) for s in args.lib] or [("tree", os.path.join(ROOT, "a.i.gar_b200", "libagar_b200.so"))]
    res, info = {}, {}
    for run in range(args.runs):
        for name, path in libs:
            env = dict(os.environ, AGAR_B200_LIB=os.path.abspath(path))
            child = CHILD % (ROOT, args.envs, args.reps, [int(f) for f in args.fpd.split(",")])
            p = subprocess.run([sys.executable, "-c", child], env=env, capture_output=True, text=True)
            if p.returncode != 0:
                sys.stderr.write(p.stderr)
                raise SystemExit("run %d of %s failed" % (run, name))
            r = json.loads(p.stdout.strip().splitlines()[-1])
            info.setdefault(name, []).append(r["info"])
            for w, arms in r["ms"].items():
                for arm, v in arms.items():
                    res.setdefault(name, {}).setdefault(w, {}).setdefault(arm, []).extend(v)
    summary = {}
    for name, ws in res.items():
        i0 = info[name][0]
        print("%s: %s, power limit %s W, SM clock %s MHz (max %s)" % (name, i0.get("gpu"), i0.get("power_limit_w"),
                                                                     [i.get("sm_mhz") for i in info[name]], i0.get("sm_max_mhz")))
        for w, arms in ws.items():
            med = {a: statistics.median(v) for a, v in arms.items()}
            summary.setdefault(name, {})[w] = {a: {"median_ms": med[a], "min_ms": min(v), "max_ms": max(v), "n": len(v)}
                                               for a, v in arms.items()}
            summary[name][w]["obs_share"] = 1.0 - med["no_obs"] / med["obs"]
            print("  %d envs %s  obs %.3f ms [%.3f, %.3f]   no obs %.3f ms [%.3f, %.3f]   obs share %.1f %%" % (
                args.envs, w, med["obs"], min(arms["obs"]), max(arms["obs"]), med["no_obs"], min(arms["no_obs"]), max(arms["no_obs"]),
                100.0 * summary[name][w]["obs_share"]))
    print(json.dumps({"summary": summary, "info": info}))


if __name__ == "__main__":
    main()
