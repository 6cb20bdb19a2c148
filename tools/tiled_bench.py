"""Time the giant-grid path in isolation on one GPU: N x N torus, n agents, K steps after the literal first step.

--series: the cost of series mode (BandedDaisyWorld.run_series): the same K steps with series mode off and on, the two arms
alternating, five repetitions each (optional argument: N, default 16384)."""
import sys, os, subprocess, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch
from therldaisyworld_b200.banded import BandedDaisyWorld

def bench(N, n, policy, K=64, reps=3):
    w = BandedDaisyWorld(N, n)
    w.reset_on_device(seed=1)
    w.run(2, policy)
    best = 1e9
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        w.band.run_local(K, policy)
        e1.record()
        torch.cuda.synchronize()
        w._pending += K
        w.end_chunk()
        best = min(best, e0.elapsed_time(e1))
    print(f"N={N} n={n} {policy}: {best / K * 1e3:.1f} us/step -> {N * N * K / best / 1e-3:.3e} cell-updates/s, "
          f"HBM {8 * N * N * K / best / 1e-3 / 1e9:.0f} GB/s algorithmic, slow cells {w.band.slow_count()}", flush=True)

def gpu_label():
    """Name and power limit of the GPU the numbers were taken on (read-only query)."""
    try:
        out = subprocess.check_output(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i",
                                       str(torch.cuda.current_device())], text=True).strip()
    except (OSError, subprocess.CalledProcessError):
        out = f"{torch.cuda.get_device_name()}, power limit unknown"
    return out


def bench_series(N, n, policy, K=256, reps=5):
    """Per-step time of K steps (dwt_run, no host sync inside) with series mode off and on, alternating arm by arm."""
    w = BandedDaisyWorld(N, n)
    w.reset_on_device(seed=1)
    w.run(2, policy)
    times = {False: [], True: []}
    for _ in range(reps):
        for on in (False, True):
            w.band.set_series(on)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            e0.record()
            w.band.run_local(K, policy)
            e1.record()
            torch.cuda.synchronize()
            if on:
                s = w.band.take_series(K)
                assert 200.0 < s[-1, 0] / (N * N) < 400.0       # a plausible mean temperature: the series was recorded
            w._pending += K
            w.end_chunk()
            w.band.set_series(False)
            times[on].append(e0.elapsed_time(e1) / K * 1e3)
    off, on = np.array(times[False]), np.array(times[True])
    print(f"N={N} n={n} {policy}, K={K} steps per arm, {reps} alternating repetitions per arm")
    print("  series off us/step: " + " ".join(f"{t:.1f}" for t in off))
    print("  series on  us/step: " + " ".join(f"{t:.1f}" for t in on))
    print(f"  median off {np.median(off):.1f} us, on {np.median(on):.1f} us: series mode costs "
          f"{100.0 * (np.median(on) / np.median(off) - 1.0):+.1f} % per step", flush=True)


if __name__ == "__main__":
    if "--series" in sys.argv:
        args = [a for a in sys.argv[1:] if a != "--series"]
        N = int(args[0]) if args else 16384
        print(f"GPU: {gpu_label()}")
        bench_series(N, N, "greedy")
        sys.exit(0)
    if len(sys.argv) > 1:                       # profiling target: one size, few steps
        N = int(sys.argv[1])
        bench(N, N, "greedy", K=8, reps=1)
        sys.exit(0)
    for N, n in ((1024, 1024), (4096, 4096), (16384, 16384), (16384, 0)):
        bench(N, n, "greedy")
