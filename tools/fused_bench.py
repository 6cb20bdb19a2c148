"""Time the fused path in isolation: B worlds of 64x64, T steps from a post-first-step checkpoint.
python tools/fused_bench.py [quick | mlp]. `quick` is the short set the kernel tuning in DESIGN.md section 4 was measured on;
run it once per build (DW_LIB=<path to the .so>) to compare two builds."""
import sys, os, time, ctypes as C
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
from therldaisyworld_b200 import RLDaisyWorld
from therldaisyworld_b200._lib import DwProfile

def bench(B, n_agents, policy, T=383, reps=3, N=64):
    np.random.seed(13)
    env = RLDaisyWorld(grid_dimension=N, n_agents=n_agents); env.batch_size = B; env.reset()
    if policy == "mlp":
        env.set_mlp(np.random.RandomState(0).randn(1808))
    env.run(1, policy=policy)                      # literal first step -> lattice
    lib, h = env._lib, env._h
    lib.dw_checkpoint_save(h)
    best = 1e9
    for r in range(reps):
        lib.dw_checkpoint_restore(h); env._pull_clock(); lib.dw_synchronize(h)
        lib.dw_set_profiling(h, 1)
        t = time.perf_counter(); env.run(T, policy=policy); lib.dw_synchronize(h); dt = time.perf_counter() - t
        p = DwProfile(); lib.dw_get_profile(h, C.byref(p))
        best = min(best, p.fused_ms if policy != "mlp" else dt * 1e3)
    print(f"N={N} B={B:6d} n={n_agents} {policy:7s}: fused {best:8.3f} ms for {T} steps -> {B*N*N*T/best/1e-3:.3e} cell-updates/s "
          f"(wall {dt*1e3:.2f} ms, {p.fused_launches} launches)", flush=True)

if __name__ == "__main__":
    if len(sys.argv) > 1 and sys.argv[1] == "quick":
        print("lib:", os.environ.get("DW_LIB", "default"))
        bench(1000, 4, "greedy"); bench(4736, 4, "greedy"); bench(4736, 0, "none")
        sys.exit(0)
    if len(sys.argv) > 1 and sys.argv[1] == "mlp":     # wall time is the measure (DW_MLP_UNFUSED=1: policy between one-step launches,
                                                       # the reference path the tests compare the in-kernel policy with)
        for B in (1000, 10000, 100000):
            bench(B, 4, "mlp", T=128 if B > 20000 else 383)
        sys.exit(0)
    for B in (1000, 1184, 4736):
        bench(B, 4, "greedy")
        bench(B, 4, "none")
        bench(B, 0, "none")
