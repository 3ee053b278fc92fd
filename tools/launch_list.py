"""Every kernel launch the library makes over a fixed matrix of configs, env counts, tile widths and entry points, from a
torch.profiler trace with CUDA activities: one JSON line per launch (case, kernel, grid, block, shared memory as the trace
reports it) and one line per case with agar_launch_count and agar_observer_launch_count.  Two builds whose launch planning
agrees print the same lines, so the library is chosen with AGAR_B200_LIB:

    AGAR_B200_LIB=/path/to/other/libagar_b200.so python tools/launch_list.py > other.jsonl
    python tools/launch_list.py > this.jsonl
    diff other.jsonl this.jsonl

The matrix reaches every instantiation the planner can select: configs[1] at every k_simple tile width, env counts on both
sides of the observer-warp wave rule, the default widths at 65 536 and 1 048 576 envs, configs[2] and a three-player variant
at the CTA sizes of k_main<32, true, 1024 / 768> (the wave cost model keeping and shrinking the CTA), configs[2] at 4, 8 and
16 lanes, configs[3], the G = 42 single-cell config and AGAR_GENERAL_KERNEL=1 (k_main<32, false>).  Each case creates its
handle (k_init) and runs observe, step, step_observe and rollout_random at 1, 3, 4 and 8 frames, with and without an
observation buffer, step_host with pinned and with pageable buffers, reset, reset_bots, snapshot and restore.  Then a second
handle of each case (case name + " | agar_rollout", so that the lines above stay comparable with builds that lack the call)
runs agar_rollout with the random driver and with caller actions at the same frame counts.  The trace goes to a temporary
directory."""
import json
import os
import re
import sys
import tempfile

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import numpy as np  # noqa: E402
import torch  # noqa: E402

import aigar_b200.layout as lay  # noqa: E402
from aigar_b200.env import AgarBatch, Trajectory  # noqa: E402

C2 = dict(num_nn=1, num_greedy=1, virus=True, split=True, eject=True)
C3 = dict(num_nn=8, num_greedy=8, virus=True, split=True, eject=True)
FRAMES = (1, 3, 4, 8)

# (case, derive_config arguments, envs, tile width (None: the library's default), AGAR_GENERAL_KERNEL set)
CASES = ([("configs[1] W=%d" % w, {}, 4096, w, False) for w in (1, 2, 4, 8, 16, 32)] +
         [("configs[1] %d envs W=%d" % (n, w), {}, n, w, False)
          for n, w in ((4144, 8), (4145, 8), (4608, 8), (8192, 4), (8192, 8))] +
         [("configs[1] %d envs" % n, {}, n, None, False) for n in (65536, 1048576)] +
         [("configs[2] %d envs" % n, C2, n, None, False) for n in (16384, 4736)] +
         [("configs[2] W=%d" % w, C2, 2048, w, False) for w in (4, 8, 16)] +
         [("1 NN + 2 greedy 16384 envs", dict(C2, num_greedy=2), 16384, None, False),
          ("configs[3] 8192 envs", C3, 8192, None, False),
          ("G=42 single cell", dict(grid=42), 4096, None, False),
          ("configs[1] AGAR_GENERAL_KERNEL=1", {}, 4096, None, True)])

KERNEL = re.compile(r"^(?:void )?k_\w+")


def run_ops(b):
    for nf in FRAMES:
        b.observe()
        b.step(None, nf)
        b.step_observe(None, nf)
        b.rollout_random(2, nf, 0)
        b.rollout_random(2, nf, 0, write_obs=False)
    A, L = max(b.layout.n_agents, 1), b.layout.state_len
    for pinned in (True, False):
        def buf(shape, dt):
            t = torch.zeros(shape, dtype=dt)
            return (t.pin_memory() if pinned else t).numpy()
        b.step_host(buf((b.n_envs, A, 4), torch.float32), 8, buf((b.n_envs, A, L), torch.float32),
                    buf((b.n_envs, A), torch.float32), buf((b.n_envs, A), torch.uint8))
    b.reset()
    b.reset_bots()
    b.restore(b.snapshot())


def run_rollout_ops(b):
    for nf in FRAMES:
        b.rollout(2, nf, 0, out=Trajectory.allocate(b, 2))
        traj = Trajectory.allocate(b, 2, [f for f in Trajectory._fields[:6] if f != "action"])
        b.rollout(2, nf, 0, actions=torch.zeros((2,) + tuple(b.actions.shape), device=b.device), out=traj)


def kernel_launches(prof, tmp):
    path = os.path.join(tmp, "trace.json")
    prof.export_chrome_trace(path)
    with open(path) as f:
        events = json.load(f)["traceEvents"]
    ks = sorted((e for e in events if e.get("cat") == "kernel" and KERNEL.match(e.get("name", ""))), key=lambda e: e["ts"])
    return [{"kernel": e["name"], "grid": e["args"].get("grid"), "block": e["args"].get("block"),
             "shared_memory": e["args"].get("shared memory")} for e in ks]


def main():
    if not torch.cuda.is_available():
        raise SystemExit("launch_list.py lists GPU kernel launches: it needs a CUDA device")
    with tempfile.TemporaryDirectory() as tmp:
        for case, kw, n, w, general in CASES:
            for name, ops in ((case, run_ops), (case + " | agar_rollout", run_rollout_ops)):
                if general:
                    os.environ["AGAR_GENERAL_KERNEL"] = "1"
                try:
                    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
                        b = AgarBatch(lay.derive_config(**kw), n, seed=1, tile_width=w)
                        ops(b)
                        torch.cuda.synchronize()
                finally:
                    os.environ.pop("AGAR_GENERAL_KERNEL", None)
                for k in kernel_launches(prof, tmp):
                    print(json.dumps(dict(case=name, **k)))
                print(json.dumps({"case": name, "tile_width": b.tile_width, "agar_launch_count": b.launch_count,
                                  "agar_observer_launch_count": b.observer_launch_count}))
                b.close()
                del b
                torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
