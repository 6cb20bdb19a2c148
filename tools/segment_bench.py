"""Whole-life ensemble (100 000 worlds of 64x64, greedy) under the notebook's stopping rule: device time per experiment for
segment lengths / trimmed vs checkpointed segments. python tools/segment_bench.py [B]"""
import os, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch
from therldaisyworld_b200 import RLDaisyWorld
from therldaisyworld_b200.ensemble import DeviceShard, simulate_lifespan
B = int(sys.argv[1]) if len(sys.argv) > 1 else 100000
np.random.seed(0)
env = RLDaisyWorld(grid_dimension=64)
env.batch_size = B
for label, segment, envs in (("auto (trimmed)", None, {}), ("segment 64 trimmed", 64, {}), ("segment 32 trimmed", 32, {}),
                             ("segment 16 trimmed", 16, {}), ("segment 64 checkpoint+replay", 64, {"DW_NO_TRIM": "1"})):
    os.environ.pop("DW_NO_TRIM", None)
    os.environ.update(envs)
    best = None
    for rep in range(3):
        env.reset_on_device(seed=13)
        env.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        r = simulate_lifespan(DeviceShard(env), policy="greedy", seed=7, device="cuda", segment=segment)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        best = ms if best is None else min(best, ms)
    print(f"{label:32s}: {r['steps']} steps, best of 3 {best:8.2f} ms -> {B * 4096 * r['steps'] / best / 1e-3:.3e} cell-updates/s "
          f"(lifespan {r['biosphere_lifespan_mean']:.3f}, agents {r['agent_lifespan_mean']:.3f})", flush=True)
