#!/usr/bin/env python
"""bench.py — batched agar.io env-steps/s on B200 (BASELINE.json metric), one JSON line on stdout.

Workload (config.workload): BASELINE.json configs[1] — pellet collection, 1 RL agent, no opponents or viruses,
grid-vision obs; 4096 envs per GPU, random-action driver, 1000-frame rollouts.  One "step" = one 1000-frame
rollout of every env (125 decisions x (observe -> random action -> 8 frames)), which agar_rollout_random runs
as ONE persistent launch.  value = env-steps (frames x envs) per second with all state resident in HBM;
e2e = the same rollout driven through agar_step_host (host action buffers in, host obs/reward/done out, copies
inside the timed region).  Weak scaling: every rank runs its own 4096 envs, no collective on the step path
(one NCCL all-reduce of episode statistics after the timed region).

python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--envs E] [--frames F] [--tile W] [--dump-outputs DIR]
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "env_steps_per_sec"
UNIT = "env-steps/s"
FRAME_SKIP = 7
PERIOD = FRAME_SKIP + 1


def algorithmic_bytes_per_env_step(p_live=85.0, c_live=1.0, vb_live=0.0, k=1, state_len=123, obs_per_frame=1.0 / PERIOD):
    """SURVEY.md §8(d): 12*P + 64*C + 48*(V+B) + 96*K + 4*L*n_obs."""
    return 12.0 * p_live + 64.0 * c_live + 48.0 * vb_live + 96.0 * k + 4.0 * state_len * obs_per_frame


def measured_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


def profiled_kernel_facts(envs, frames):
    """What ncu measured for the bench kernel at this launch shape (profiles/traffic.json, written from the committed ncu
    summary of the same command): DRAM bytes per launch, issue-slot utilisation, warp instructions per env-step."""
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            t = json.load(f)
        if int(t.get("envs", -1)) == envs and int(t.get("frames", -1)) == frames:
            return t
    except Exception:
        pass
    return {}


class ClockSampler(object):
    """SM clock / throttle reasons DURING the timed region (B200_PROFILING.md recipe).  NVML is read from a thread of this
    process every 2 ms (nvidia_ml_py: the library nvidia-smi itself reads) — a spawned `nvidia-smi -lms 5` needs 0.1-0.3 s to
    start, and the whole timed region is ~0.13 s: it delivered between 1 and 20 samples per run.  nvidia-smi remains the fallback."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")
    REASON_BITS = {"sw_power_cap": 0x4, "hw_slowdown": 0x8, "sw_thermal_slowdown": 0x20, "hw_thermal_slowdown": 0x40}

    def __init__(self, index):
        self.index = index
        self.proc = None
        self.path = None
        self.thread = None
        self.samples = []
        self.stop_flag = False

    def _nvml_handle(self):
        import pynvml
        pynvml.nvmlInit()
        try:  # the CUDA ordinal is not the NVML index when CUDA_VISIBLE_DEVICES reorders devices: go through the UUID
            import torch
            uuid = str(torch.cuda.get_device_properties(self.index).uuid)
            return pynvml, pynvml.nvmlDeviceGetHandleByUUID(("GPU-" + uuid) if not uuid.startswith("GPU-") else uuid)
        except Exception:
            return pynvml, pynvml.nvmlDeviceGetHandleByIndex(self.index)

    def _poll(self, nv, h):
        reasons_fn = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or nv.nvmlDeviceGetCurrentClocksThrottleReasons
        mx = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
        while not self.stop_flag:
            try:
                self.samples.append((nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM), mx, int(reasons_fn(h))))
            except Exception:
                pass
            time.sleep(0.002)

    def start(self):
        try:
            import threading
            nv, h = self._nvml_handle()
            nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)
            self.thread = threading.Thread(target=self._poll, args=(nv, h), daemon=True)
            self.thread.start()
            return
        except Exception:
            self.thread = None
        try:
            fd, self.path = tempfile.mkstemp(suffix=".csv")
            os.close(fd)
            self.out = open(self.path, "w")
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "5"], stdout=self.out,
                                         stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        res = {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        if self.thread is not None:
            self.stop_flag = True
            self.thread.join(timeout=2)
            if self.samples:
                sm = sorted(s[0] for s in self.samples)
                bits = 0
                for s in self.samples:
                    bits |= s[2]
                res = {"sm_mhz": float(sm[len(sm) // 2]), "sm_max_mhz": float(max(s[1] for s in self.samples)),
                       "reasons": sorted(n for n, b in self.REASON_BITS.items() if bits & b), "samples": len(sm),
                       "source": "NVML, 2 ms"}
            return res
        if self.proc is None:
            return res
        try:
            self.proc.terminate()
            self.proc.wait(timeout=5)
            self.out.close()
            sm, mx, reasons = [], [], set()
            names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
            with open(self.path) as f:
                for line in f:
                    parts = [p.strip() for p in line.split(",")]
                    if len(parts) < 9:
                        continue
                    try:
                        sm.append(float(parts[1]))
                        mx.append(float(parts[2]))
                    except ValueError:
                        continue
                    for n, v in zip(names, parts[5:9]):
                        if v.lower().startswith("active"):
                            reasons.add(n)
            os.unlink(self.path)
            if sm:
                sm.sort()
                res = {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": max(mx), "reasons": sorted(reasons), "samples": len(sm),
                       "source": "nvidia-smi -lms 5"}
        except Exception:
            pass
        return res


CONFIGS = {
    # BASELINE.json configs[1..3]; bytes = SURVEY §8d's worked algorithmic bytes per env-step (obs every 8th frame)
    "configs[1]": dict(kw=dict(), envs=4096, bytes=None,
                       name="pellet collection, 1 RL agent, no opponents/viruses, grid-vision obs"),
    "configs[2]": dict(kw=dict(num_nn=1, num_greedy=1, virus=True, split=True, eject=True), envs=16384, bytes=2950.0,
                       name="1 agent vs 1 greedy bot, viruses, splitting and ejection"),
    "configs[3]": dict(kw=dict(num_nn=8, num_greedy=8, virus=True, split=True, eject=True), envs=8192, bytes=22900.0,
                       name="multi-agent arena: 8 agents + 8 greedy bots, 1350 pellets, split / merge heavy"),
}


def cpu_port_throughput(n_threads, kw=None, target_s=10.0, frames=1000, max_envs=4096):
    """The C oracle (oracle/agar_oracle.c, libm build: bit-exact against the Python reference) on the host cores: the CPU
    baseline / reference arm.  Returns (env-steps/s, description of the bounded sample)."""
    import aigar_b200.layout as lay
    from oracle import oracle as orc
    cfg = lay.derive_config(**(kw or {}))
    decisions = frames // PERIOD
    t0 = time.perf_counter()
    steps, _ = orc.rollout_batch(cfg, n_threads, 11, 0, 10, n_threads)  # probe: 80 frames per thread
    probe = max(time.perf_counter() - t0, 1e-4)
    rate = steps / probe
    envs = int(max(n_threads, min(max_envs, rate * target_s / (decisions * PERIOD))))
    envs = max(n_threads, envs // n_threads * n_threads)
    t0 = time.perf_counter()
    steps, _ = orc.rollout_batch(cfg, envs, 11, 0, decisions, n_threads)
    dt = time.perf_counter() - t0
    return steps / dt, "sample of %d envs x %d frames of the same workload on %d threads (%.1f s)" % (
        envs, decisions * PERIOD, n_threads, dt)


def python_reference_numbers():
    """The unpatched Python reference timed in the build container (tools/time_reference.py -> profiles/): it cannot travel to
    the GPU box, so its numbers are cited, with the machine they were taken on, next to the C port timed here."""
    try:
        with open(os.path.join(ROOT, "profiles", "r02_python_reference.json")) as f:
            d = json.load(f)
        out = {"source": "profiles/r02_python_reference.json (tools/time_reference.py, build container)",
               "cpu_model": d["cpu_model"], "cores": d["cores"], "unit": "frames/s"}
        for k, v in d["configs"].items():
            out[k] = {"model_update_1core": round(v["model_update_frames_per_s_1core"], 1),
                      "model_update_pool": round(v["model_update_frames_per_s_pool"], 1),
                      "field_update_only_1core": round(v["field_update_only_frames_per_s_1core"], 1),
                      "get_state_representation_1core": round(v["get_state_representation_obs_per_s_1core"], 1)}
        return out
    except Exception:
        return None


def workload_name(envs, frames, key="configs[1]"):
    return ("%s: %s; %d envs per GPU, random-action driver, %d-frame rollouts (frame-skip 7, obs every 8th frame; "
            "observations in the reference's own binning, AGAR_OBS_REFERENCE)" % (key, CONFIGS[key]["name"], envs, frames))


def base_config(E, frames, world):
    """`config` of the JSON line — the SAME dict in the GPU arm and in the reference (CPU) arm, so that the driver can see that
    both ran one workload; launch-shape details of the GPU arm live under `launch`."""
    return {"workload": workload_name(E, frames), "envs_per_gpu": E, "frames_per_step": frames,
            "l2": "GPU arm: flushed between timed steps (256 MiB write); CPU arm: not applicable",
            "parallelism": "env-sharded x%d, no collective on the step path" % world}


def run_reference(args):
    """--impl reference: the reference's CPU implementation of the path.  The reference is pure Python and cannot travel
    to the GPU box, so this times its C restatement (oracle/, bit-exact against it) on all host threads, each step a
    bounded sample of the same workload."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    import aigar_b200.layout as lay
    from oracle import oracle as orc
    cfg = lay.derive_config()
    cores = os.cpu_count() or 1
    frames = args.frames
    decisions = frames // PERIOD
    frames = decisions * PERIOD
    # size one step to ~2 s
    t0 = time.perf_counter()
    steps, _ = orc.rollout_batch(cfg, cores, 11, 0, 10, cores)
    rate = steps / max(time.perf_counter() - t0, 1e-4)
    envs = int(max(cores, min(args.envs, rate * 2.0 / (decisions * PERIOD))))
    envs = max(cores, envs // cores * cores)
    for _ in range(args.warmup):
        orc.rollout_batch(cfg, envs, 11, 0, max(decisions // 8, 1), cores)
    t0 = time.perf_counter()
    total = 0
    for i in range(args.steps):
        s, _ = orc.rollout_batch(cfg, envs, 11, 1000 * (i + 1), decisions, cores)
        total += s
    dt = time.perf_counter() - t0
    v = total / dt
    sample = "sample of %d envs x %d frames per step (of the %d-env workload) on %d threads" % (envs, frames, args.envs, cores)
    conf = base_config(args.envs, frames, max(args.gpus, 1))
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": conf,
            "sample": {"envs": envs, "frames": frames, "of_envs": args.envs, "threads": cores, "text": sample},
            "cpu_baseline": {"value": v, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample,
                             "python_reference": python_reference_numbers()},
            "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))
    return 0


def device_rollouts(batch, decisions, steps, warmup, flush, dist=None, world=1):
    """W untimed + K timed persistent rollouts (one launch each), L2 flushed between timed steps, CUDA events on the launching
    stream, max over ranks.  Returns total ms of the K steps."""
    import torch
    for i in range(warmup):
        batch.rollout_random(decisions, PERIOD, decision_base=i * decisions)
    if dist is not None:
        dist.barrier()
    torch.cuda.synchronize()
    evs = []
    for i in range(steps):
        if flush is not None:
            flush.fill_(i & 0xff)  # evict L2 between timed steps (126 MB L2 < 256 MiB)
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        batch.rollout_random(decisions, PERIOD, decision_base=(warmup + i) * decisions)
        e.record()
        evs.append((s, e))
    if dist is not None:
        dist.barrier()
    torch.cuda.synchronize()
    total_ms = float(sum(s.elapsed_time(e) for s, e in evs))
    if dist is not None:
        t = torch.tensor([total_ms], dtype=torch.float64, device=batch.device)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        total_ms = float(t.item())
    return total_ms


DUMP_LIMIT_BYTES = 64 * 1000 * 1000  # all files together, .npy headers included
NPY_HEADER_BYTES = 128
DUMP_GETTERS = ("reward", "done", "valid", "need_action", "mass", "fov", "ncells", "alive", "stats", "overflow")  # lay.GET_<NAME>


def dump_outputs(batch, out_dir, limit=DUMP_LIMIT_BYTES):
    """--dump-outputs: what the last timed rollout hands its caller, written as out_dir/<name>.npy so that two builds run with
    the same arguments (same seed, env ids and decision indices, hence the same inputs) can be compared output for output.
    obs is the [E, A, L] observation tensor the rollout returns; the others are the env's getters after it ([E, A], stats
    [E, A, 4], overflow [E]); event_hash [E, 2] holds the high and low 32-bit halves of the per-env hash of every event.
    Values are float32, or float64 where float32 would round them.  Above `limit` bytes a fixed, seeded sample of envs is
    written and env_index.npy lists them."""
    import numpy as np
    import aigar_b200.layout as lay
    out = {"obs": batch.obs.cpu().numpy()}
    for name in DUMP_GETTERS:
        out[name] = batch.get(getattr(lay, "GET_" + name.upper())).cpu().numpy()
    out["overflow"] = out["overflow"].view(np.uint32).astype(np.float64)
    h = batch.get(lay.GET_EVENT_HASH).cpu().numpy().view(np.uint64)
    out["event_hash"] = np.stack([h >> np.uint64(32), h & np.uint64(0xFFFFFFFF)], axis=-1).astype(np.float64)
    out = {k: v if v.dtype == np.float64 else v.astype(np.float32) for k, v in out.items()}
    E = batch.n_envs
    per_env = sum(v.nbytes for v in out.values()) / E
    room = limit - NPY_HEADER_BYTES * (len(out) + 1)  # + env_index.npy
    if per_env * E > limit - NPY_HEADER_BYTES * len(out):
        idx = np.sort(np.random.default_rng(0).choice(E, int(room // (per_env + 8)), replace=False))
        out = {k: v[idx] for k, v in out.items()}
        out["env_index"] = idx.astype(np.float64)
    os.makedirs(out_dir, exist_ok=True)
    for k, v in out.items():
        np.save(os.path.join(out_dir, k + ".npy"), v)


def scaling_sweep(cfg, local, rank, world, dist, flush):
    """BASELINE configs[4]: 65 536 / 262 144 / 1 048 576 TOTAL envs sharded evenly over the ranks (shard_envs: contiguous global
    env ids, Philox key = global id), observations handed to a torch DQN (MLP 123-100-100-25) through DLPack, arg-max -> the
    reference's 5x5 action table -> 8 frames; one tick = MLP + our step kernel captured in a CUDA graph.  Timed with CUDA
    events per rank, max over ranks."""
    import torch
    from aigar_b200.dqn import DQNDriver
    from aigar_b200.env import AgarBatch
    from aigar_b200.sharding import shard_envs
    peak, _ = measured_peak()
    out = {}
    for total in (65536, 262144, 1048576):
        try:
            first, n = shard_envs(total, world, rank)
            b = AgarBatch(cfg, n, device=local, seed=2026, first_env_id=10 ** 7 + first)
            drv = DQNDriver(b, seed=0)
            ticks = 12
            drv.run(4, use_graph=True)
            if dist is not None:
                dist.barrier()
            torch.cuda.synchronize()
            flush.fill_(1)
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record()
            for _ in range(ticks):
                drv._graph.replay()
            e.record()
            torch.cuda.synchronize()
            ms = s.elapsed_time(e)
            # the env path alone at the same size (persistent random-action rollout)
            d2 = 12
            for i in range(2):
                b.rollout_random(d2, PERIOD, decision_base=i * d2)
            torch.cuda.synchronize()
            flush.fill_(2)
            s.record()
            b.rollout_random(d2, PERIOD, decision_base=2 * d2)
            e.record()
            torch.cuda.synchronize()
            ms_env = s.elapsed_time(e)
            t = torch.tensor([ms, ms_env], dtype=torch.float64, device=b.device)
            if dist is not None:
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms, ms_env = float(t[0].item()), float(t[1].item())
            v = total * ticks * PERIOD / (ms * 1e-3)
            v_env = total * d2 * PERIOD / (ms_env * 1e-3)
            out["envs_%d" % total] = {
                "total_envs": total, "envs_per_gpu": n, "n_gpus": world, "value_dqn_loop": v, "value_env_only": v_env,
                "unit": UNIT, "ms_per_tick": ms / ticks, "tile_width": b.tile_width,
                "state_bytes_per_gpu": int(n * b.layout.record_bytes),
                "roofline_frac_per_gpu_dqn_loop": v / world * algorithmic_bytes_per_env_step() / 1e9 / peak,
                "roofline_frac_per_gpu_env_only": v_env / world * algorithmic_bytes_per_env_step() / 1e9 / peak}
            b.close()
            del drv
        except Exception as ex:  # never lose the headline line to a side measurement
            out["envs_%d" % total] = {"error": str(ex)[:200]}
    return out


def other_config(key, local, flush, steps=5, warmup=2, with_cpu=True, e2e_steps=2, groups=2):
    """BASELINE configs[2] / [3] to the same contract as the headline: full 1000-frame rollouts at the named env count, L2 flush,
    >= 5 timed steps, their own e2e (host buffers through the C ABI) and CPU baseline (the C port on the host cores)."""
    import torch
    import aigar_b200.layout as lay
    from aigar_b200.env import AgarBatch
    spec = CONFIGS[key]
    cfg = lay.derive_config(**spec["kw"])
    E, decisions = spec["envs"], 1000 // PERIOD
    frames = decisions * PERIOD
    peak, _ = measured_peak()
    b = AgarBatch(cfg, E, device=local, seed=2026, first_env_id=3 * 10 ** 6)
    n0 = b.launch_count
    ms = device_rollouts(b, decisions, steps, warmup, flush)
    v = E * frames * steps / (ms * 1e-3)
    res = {"workload": workload_name(E, frames, key), "value": v, "unit": UNIT, "steps": steps, "warmup": warmup,
           "ms_per_step": ms / steps, "frames_per_step": frames, "envs": E, "gpu_launches": int(b.launch_count - n0 - warmup),
           "bytes_per_env_step": spec["bytes"], "roofline_frac": v * spec["bytes"] / 1e9 / peak,
           "players": int(b.layout.n_players), "state_len": int(b.layout.state_len), "tile_width": b.tile_width,
           "record_bytes": int(b.layout.record_bytes), "l2": "flushed between timed steps"}
    b.close()
    try:
        res["e2e"] = run_e2e(cfg, E, decisions, e2e_steps, local, 0, 1, None, torch.cuda.synchronize, groups)
    except Exception as ex:
        res["e2e"] = {"error": str(ex)[:200]}
    if with_cpu:
        cores = os.cpu_count() or 1
        cv, sample = cpu_port_throughput(cores, spec["kw"], target_s=6.0)
        res["cpu_baseline"] = {"value": cv, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample}
    return res


def run_e2e(cfg, E, decisions, e2e_steps, local, rank, world, dist, barrier, groups, seed=2026):
    """The same rollout driven from the HOST through the public C ABI: every decision the caller's pinned action buffer goes
    in and its pinned observation / reward / done buffers come back (agar_step_host_begin / _end, include/agar_b200.h).
    The envs are split into `groups` handles on their own streams, exactly as a CPU policy would pipeline them: while one
    group steps on the GPU the host already holds the previous group's observations.  Every group still receives the
    observation of decision d before its action of decision d + 1 is submitted.  Copies are inside the timed region: the
    step kernel reads the actions in place over PCIe and its CTAs store their rows into the caller's buffers."""
    import torch
    import aigar_b200.layout as lay
    from aigar_b200.env import AgarBatch
    G = max(1, min(groups, E))
    Eg = E // G
    assert Eg * G == E, "--groups must divide --envs"
    device = torch.device("cuda", local)
    streams = [torch.cuda.Stream(device=device) for _ in range(G)]
    hs = [AgarBatch(cfg, Eg, device=local, seed=seed, first_env_id=rank * E + g * Eg, stream=streams[g]) for g in range(G)]
    L = hs[0].layout
    A = max(L.n_agents, 1)
    acts = torch.rand((decisions, E, A, 4), dtype=torch.float32).pin_memory()
    obs_h = torch.empty((E, A, L.state_len), dtype=torch.float32).pin_memory()
    rew_h = torch.empty((E, A), dtype=torch.float32).pin_memory()
    done_h = torch.empty((E, A), dtype=torch.uint8).pin_memory()
    # raw addresses of every (decision, group) slice: no per-call numpy / ctypes conversion inside the timed loop
    a_ptr = [[acts[d, g * Eg:(g + 1) * Eg].data_ptr() for g in range(G)] for d in range(decisions)]
    o_ptr = [obs_h[g * Eg:(g + 1) * Eg].data_ptr() for g in range(G)]
    r_ptr = [rew_h[g * Eg:(g + 1) * Eg].data_ptr() for g in range(G)]
    d_ptr = [done_h[g * Eg:(g + 1) * Eg].data_ptr() for g in range(G)]

    clock = time.perf_counter
    last_launch = [0.0]

    def begin(g, d, spacing):
        # pacing: consecutive launches at least `spacing` apart, so that the groups run out of phase — one group's PCIe export
        # overlaps the other's frames (groups launched together finish together and the GPU idles while the rows leave)
        if spacing > 0.0:
            while clock() - last_launch[0] < spacing:
                pass
        hs[g].step_host_begin_ptr(a_ptr[d][g], PERIOD, o_ptr[g])
        last_launch[0] = clock()

    def rollout(spacing, n_dec=decisions):
        for g in range(G):
            begin(g, 0, spacing)
        for d in range(1, n_dec):
            for g in range(G):
                hs[g].step_host_end_ptr(r_ptr[g], d_ptr[g])      # observation / reward / done of decision d - 1 are on the host
                begin(g, d, spacing)
        for g in range(G):
            hs[g].step_host_end_ptr(r_ptr[g], d_ptr[g])

    for g in range(G):
        hs[g].observe()
    rollout(0.0)  # warm-up: one full rollout
    spacing = 0.0
    if G > 1:  # pick the launch spacing in the warm-up: fractions of the unpaced per-decision time
        n_try = min(decisions, 40)
        torch.cuda.synchronize()
        t0 = clock()
        rollout(0.0, n_try)
        base = (clock() - t0) / n_try
        best = base
        for frac in (0.15, 0.25, 0.35, 0.45, 0.55):
            cand = base * frac * 2.0 / G
            t0 = clock()
            rollout(cand, n_try)
            t = (clock() - t0) / n_try
            if t < best:
                best, spacing = t, cand
    barrier()
    t0 = time.perf_counter()
    for i in range(e2e_steps):
        rollout(spacing)
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    tt = torch.tensor([dt], dtype=torch.float64, device=device)
    if dist is not None:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    dt = float(tt.item())
    launches = sum(h.launch_count for h in hs)
    for h in hs:
        h.close()
    frames = decisions * PERIOD
    return {"value": world * E * frames * e2e_steps / dt, "unit": UNIT,
            "h2d_bytes_per_step": int(decisions * acts[0].numel() * 4),
            "d2h_bytes_per_step": int(decisions * (obs_h.numel() * 4 + rew_h.numel() * 4 + done_h.numel())),
            "steps": e2e_steps, "calls_per_step": decisions * G, "groups": G, "launch_spacing_us": spacing * 1e6,
            "ms_per_step": dt / e2e_steps * 1e3,
            "api": "agar_step_host_begin / agar_step_host_end (C ABI, pinned host buffers; %d env groups of %d on their own "
                   "streams: actions read in place by the step kernel, its CTAs store obs / reward / done over PCIe and raise "
                   "a flag the host polls; one launch per call)" % (G, Eg)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--envs", type=int, default=4096)
    ap.add_argument("--frames", type=int, default=1000)
    ap.add_argument("--tile", type=int, default=0)
    ap.add_argument("--groups", type=int, default=4, help="env groups in flight on the host-buffer (e2e) path")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-extra", action="store_true")
    ap.add_argument("--no-sweep", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one computed (rank 0's envs) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the GPU path's outputs; the reference arm reports throughput only")
    args.warmup = max(args.warmup, 3) if args.impl != "reference" else args.warmup
    if args.impl == "reference":
        return run_reference(args)

    import torch
    import aigar_b200.layout as lay
    from aigar_b200.env import AgarBatch

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (there is no CPU fallback; use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    try:  # opt-in (AGAR_BENCH_AFFINITY=1): one core set per rank.  Measured on the 8-GPU box (32 vCPUs, one NUMA node): e2e 2.30e9 with
        # the ranks pinned, 2.40e9 without — the scheduler spreads eight polling threads well enough, so the default is off
        ncpu = os.cpu_count() or 1
        if world > 1 and ncpu >= 2 * world and os.environ.get("AGAR_BENCH_AFFINITY", "0") == "1":
            per = ncpu // world
            os.sched_setaffinity(0, set(range(local * per, (local + 1) * per)))
    except Exception:
        pass

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    E, frames = args.envs, args.frames
    decisions = frames // PERIOD
    frames = decisions * PERIOD
    cfg = lay.derive_config()
    batch = AgarBatch(cfg, E, device=local, seed=2026, first_env_id=rank * E, tile_width=args.tile or None)
    L = batch.layout
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=batch.device)

    sampler = ClockSampler(local)  # samples from the warm-up on: the same load, more samples than the timed region alone
    sampler.start()
    launches0 = batch.launch_count
    total_ms = device_rollouts(batch, decisions, args.steps, args.warmup, flush, dist, world)
    launches = batch.launch_count - launches0 - args.warmup
    clocks = sampler.stop()
    value = world * E * frames * args.steps / (total_ms * 1e-3)
    if args.dump_outputs and rank == 0:
        dump_outputs(batch, args.dump_outputs)

    # ---- e2e: host buffers through the C ABI's host-buffer step (actions H2D, obs/reward/done D2H every decision)
    e2e = None
    if not args.no_e2e:
        e2e = run_e2e(cfg, E, decisions, min(args.steps, 5), local, rank, world, dist, barrier, args.groups)

    # ---- episode statistics: the one optional collective (SURVEY §8e), outside the timed region
    stats = batch.get(lay.GET_STATS).sum(dim=(0, 1))
    ovf = (batch.get(lay.GET_OVERFLOW) != 0).sum().to(torch.float64)
    if dist is not None:
        dist.all_reduce(stats)
        dist.all_reduce(ovf)
    mean_mass = float(stats[0].item() / max(stats[2].item(), 1.0))

    extra = {}
    # ---- BASELINE configs[4]: the env-count sweep sharded over ALL ranks with the DQN consumer (every N)
    if not args.no_extra and not args.no_sweep:
        extra["sweep"] = scaling_sweep(cfg, local, rank, world, dist, flush)
    if not args.no_extra and rank == 0 and world == 1:
        try:  # SURVEY §8d: the same workload with an observation EVERY frame (FRAME_SKIP_RATE = 0 -> 1672 B per env-step)
            cfg0 = lay.derive_config(frame_skip=0)
            b0 = AgarBatch(cfg0, E, device=local, seed=2026, first_env_id=5 * 10 ** 6)
            for i in range(3):
                b0.rollout_random(frames, 1, decision_base=i * frames)
            ts = []
            for i in range(5):
                flush.fill_(i)
                s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                s.record()
                b0.rollout_random(frames, 1, decision_base=(3 + i) * frames)
                e.record()
                torch.cuda.synchronize()
                ts.append(s.elapsed_time(e))
            ms = sum(ts) / len(ts)
            v0 = E * frames / (ms * 1e-3)
            peak, _ = measured_peak()
            extra["obs_every_frame"] = {"value": v0, "unit": UNIT, "ms_per_launch": ms, "bytes_per_env_step": algorithmic_bytes_per_env_step(obs_per_frame=1.0),
                                        "roofline_frac": v0 * algorithmic_bytes_per_env_step(obs_per_frame=1.0) / 1e9 / peak,
                                        "tile_width": b0.tile_width}
            b0.close()
        except Exception as ex:
            extra["obs_every_frame"] = {"error": str(ex)[:200]}
        # BASELINE configs[2] / [3] to the same contract (full rollouts, flush, e2e, CPU arm)
        for key in ("configs[2]", "configs[3]"):
            try:
                extra[key] = other_config(key, local, flush, with_cpu=not args.no_cpu, groups=2)
            except Exception as ex:
                extra[key] = {"error": str(ex)[:200]}
        try:  # SURVEY §8f rank 1: transitions from the env's buffers into the GPU replay ring, prioritized sampling
            from aigar_b200.replay import GpuReplayBuffer
            E4 = 65536
            b4 = AgarBatch(cfg, E4, device=local, seed=7, first_env_id=3 * 10 ** 6)
            rp = GpuReplayBuffer(1 << 20, L.state_len, 4, prioritized=True)
            o0 = b4.observe().clone()
            a4 = torch.rand((E4, 1, 4), device=batch.device)
            o1 = b4.step_observe(a4, PERIOD)
            v4, d4, r4 = b4.get(lay.GET_VALID), b4.get(lay.GET_DONE), b4.get(lay.GET_REWARD)
            for _ in range(3):
                rp.add_batch(o0, a4, r4, o1, d4, v4)
            u = torch.rand(4096, dtype=torch.float64, device=batch.device)
            rp.sample(u)
            torch.cuda.synchronize()
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record()
            for _ in range(10):
                rp.add_batch(o0, a4, r4, o1, d4, v4)
            e.record()
            torch.cuda.synchronize()
            add_ms = s.elapsed_time(e) / 10
            s.record()
            for _ in range(10):
                rp.sample(u)
            e.record()
            torch.cuda.synchronize()
            smp_ms = s.elapsed_time(e) / 10
            bytes_tr = (2 * L.state_len + 4 + 1) * 4 + 1
            extra["replay"] = {"add_transitions_per_s": E4 / (add_ms * 1e-3), "add_gbs": 2 * E4 * bytes_tr / (add_ms * 1e-3) / 1e9,
                               "per_sample_4096_ms": smp_ms, "capacity": 1 << 20, "prioritized": True,
                               "note": "add = block scan + one warp per transition + tree repair (20 level launches at this batch size); GB/s counts read + write"}
            b4.close(), rp.close()
        except Exception as ex:
            extra["replay"] = {"error": str(ex)[:200]}

    if dist is not None:
        dist.barrier()
    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return 0

    peak, peak_src = measured_peak()
    bytes_per = algorithmic_bytes_per_env_step()
    launch_ms = total_ms / args.steps
    achieved = E * frames * bytes_per / (launch_ms * 1e-3) / 1e9
    prof = profiled_kernel_facts(E, frames)
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": prof.get("dram_bytes_per_launch"), "kernel": ("k_simple<%d>" if batch.tile_width <= 16 else "k_main<%d,false>") % batch.tile_width, "peak_source": peak_src,
                "bytes_per_env_step": bytes_per, "env_steps_per_launch": E * frames, "launch_ms": launch_ms,
                # the persistent launch keeps an env on chip for the whole rollout: real DRAM traffic is ~0.1 % of the algorithmic
                # bytes and the kernel is issue / latency bound — the numbers that say how busy the SMs are (ncu, profiles/):
                "real_dram_bytes_per_env_step": prof.get("dram_bytes_per_env_step"),
                "issue_slots_busy_pct": prof.get("issue_active_pct"), "warp_instructions_per_env_step": prof.get("warp_inst_per_env_step"),
                "profile": prof.get("source")}
    cpu = None
    if world == 1 and not args.no_cpu:
        cores = os.cpu_count() or 1
        v, sample = cpu_port_throughput(cores)
        cpu = {"value": v, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample,
               "python_reference": python_reference_numbers()}
    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": launch_ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
            "data": "synthetic", "config": base_config(E, frames, world),
            "launch": {"tile_width": batch.tile_width, "record_bytes": int(L.record_bytes), "kernel": roofline["kernel"]},
            "clocks": clocks, "e2e": e2e, "gpu_launches": int(launches), "roofline": roofline, "cpu_baseline": cpu,
            "episode_stats": {"mean_mass": mean_mass, "envs_with_pool_overflow": int(ovf.item())}, "extra": extra}
    print(json.dumps(line))
    if dist is not None:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
