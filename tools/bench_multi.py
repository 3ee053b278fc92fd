"""Full 1000-frame rollouts of the multi-agent configs (steady state, not the first frames after a reset):
python tools/bench_multi.py CONFIG ENVS [steps] [tile width]   (run on a GPU box)"""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import aigar_b200.layout as lay
from aigar_b200.env import AgarBatch
from sweep import KWS
which, E = sys.argv[1], int(sys.argv[2])
steps = int(sys.argv[3]) if len(sys.argv) > 3 else 2
tile = int(sys.argv[4]) if len(sys.argv) > 4 else None
b = AgarBatch(lay.derive_config(**KWS[which]), E, seed=2026, first_env_id=3 * 10 ** 6, **({"tile_width": tile} if tile else {}))
b.rollout_random(125, 8, 0)
torch.cuda.synchronize()
ts = []
for i in range(steps):
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record(); b.rollout_random(125, 8, (i + 1) * 125); e.record(); torch.cuda.synchronize()
    ts.append(s.elapsed_time(e))
ms = sum(ts) / len(ts)
print("config %s, %d envs: %.3e env-steps/s (%.1f ms per 1000-frame rollout, tile %d)" % (
    which, E, E * 1000 / (ms * 1e-3), ms, b.tile_width))
