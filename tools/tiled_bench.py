"""Time the giant-grid path in isolation on one GPU: N x N torus, n agents, K steps after the literal first step.

--series: the cost of series mode (BandedDaisyWorld.run_series): the same K steps with series mode off and on, the two arms
alternating, five repetitions each (optional argument: N, default 16384).

--sides N1 N2 ...: the stencil kernel alone (dwt_debug_time_stencil) and whole steps at each side, N agents, the sides
alternating over five repetitions; the rates are reported against the first side. Sides that are not a multiple of 64 run
the masked instance of the stencil kernel over their partial tiles.

--policy mlp [N]: the MLP policy on the giant world (default N = 16384, N agents, golden weights): whole steps with greedy and
with mlp decisions (dwt_run; an mlp step also observes), alternating over five repetitions; the latency of observe() (host
clock, download included) and of the device observation alone (CUDA events); and the mean time per launch of each kernel
of an mlp step from torch.profiler (k_band_obs, k_mlp_act, ...), in a separate profiled run.

--vs-ensemble N: whole greedy steps of one N x N world as the giant world (BandedDaisyWorld.run) and as an ensemble of one
(RLDaisyWorld, batch_size = 1, run()), 4 agents like RLDaisyWorld's default, alternating over five repetitions.

--diag [N]: the diagnostics and plot feed (default N = 16384, N agents): diag_stats("temp"), image("temp", 16),
image("grid_light", 16), cover_stats() and the device part of image() alone (dwt_pool), each timed with CUDA events around
the whole call (download included), next to a greedy step, alternating over five repetitions.

--snapshot [N]: save() and restore() of the giant world (default N = 16384, N agents, after 3 greedy steps: lattice state and
lattice pre-state, 4 B per cell each), split into the band's copies between device and host memory (dwt_save_state /
dwt_restore_state with in-memory arrays: DMA through the page-locked staging buffer, host copies, ghost-column kernel),
the file I/O of the .npy shards (to a temporary directory), the checksums, and the whole calls; next to the raw PCIe rate
of one pinned device -> host / host -> device copy of the same size. Host clock around synchronising calls, three
repetitions after a warm-up.

--f32 [N]: fp32 mode (default N = 16384, N agents, after 3 greedy steps: lattice pre-state): the device time of one
materialisation in fp32 mode (k_band_forward_f32 + stamp) and of the fp64 grid (k_band_materialise + stamp) through
dwt_debug_time_materialise, warmed up, the two arms alternating over five repetitions of 10 calls; cells/s, algorithmic
bytes (fp32: 4 + 4 B read, 28 B written per cell; fp64: 4 B read, 56 B written) and their share of the 7.7 TB/s data-sheet
HBM bandwidth; the fp64-tier and literal fractions (f32_stats); the host wall time of local_grid_f32() and local_grid()
(download included), three repetitions each."""
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


def bench_sides(sides, K=64, reps=5, stencil_reps=50):
    worlds = {}
    for N in sides:
        w = BandedDaisyWorld(N, N)
        w.reset_on_device(seed=1)
        w.run(2, "greedy")
        worlds[N] = w
    sten, step = {N: [] for N in sides}, {N: [] for N in sides}
    for _ in range(reps):
        for N in sides:
            w = worlds[N]
            sten[N].append(w.band.time_stencil(stencil_reps))
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            e0.record()
            w.band.run_local(K, "greedy")
            e1.record()
            torch.cuda.synchronize()
            w._pending += K
            w.end_chunk()
            step[N].append(e0.elapsed_time(e1) / K * 1e3)
    base = sides[0]
    rate = lambda N, us: N * N / (us * 1e-6)
    print(f"{len(sides)} sides, N agents each, {reps} alternating repetitions; stencil: {stencil_reps} launches, steps: K={K} greedy")
    for N in sides:
        ms, mt = np.median(sten[N]), np.median(step[N])
        print(f"  N={N}: stencil us " + " ".join(f"{t:.1f}" for t in sten[N]) + f" | median {ms:.1f} us = {rate(N, ms):.4e} "
              f"cell-updates/s, {rate(N, ms) / rate(base, np.median(sten[base])):.4f} of N={base}")
        print(f"  N={N}: step    us " + " ".join(f"{t:.1f}" for t in step[N]) + f" | median {mt:.1f} us = {rate(N, mt):.4e} "
              f"cell-updates/s, {rate(N, mt) / rate(base, np.median(step[base])):.4f} of N={base}", flush=True)


def bench_mlp(N, K=64, reps=5):
    from torch.profiler import ProfilerActivity, profile
    params = np.load(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden",
                                  "mlp_n16_b4_mixed_150.npz"))["mlp_params"]
    w = BandedDaisyWorld(N, N)
    w.set_mlp(params)
    w.reset_on_device(seed=1)
    w.run(2, "mlp")
    w.run(2, "greedy")

    def timed(fn):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) * 1e3

    steps = {"greedy": [], "mlp": []}
    for _ in range(reps):
        for pol in steps:
            steps[pol].append(timed(lambda: w.band.run_local(K, pol)) / K)
            w._pending += K
            w.end_chunk()
    obs_host, obs_dev, decide = [], [], []
    for _ in range(reps):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        o = w.observe()
        obs_host.append((time.perf_counter() - t0) * 1e6)
        obs_dev.append(timed(lambda: [w.band.observe() for _ in range(20)]) / 20)
        decide.append(timed(lambda: [w.band.decide("mlp") for _ in range(20)]) / 20)
    assert o.shape == (1, N, 7, 3, 3)
    print(f"N={N}, {N} agents, K={K} steps per arm (dwt_run), {reps} alternating repetitions, golden MLP weights")
    for pol, ts in steps.items():
        print(f"  {pol:6s} us/step: " + " ".join(f"{t:.1f}" for t in ts) + f" | median {np.median(ts):.1f}")
    print(f"  mlp - greedy: {np.median(steps['mlp']) - np.median(steps['greedy']):+.1f} us/step "
          f"({100.0 * (np.median(steps['mlp']) / np.median(steps['greedy']) - 1.0):+.2f} %)")
    print("  observe() us (host clock, obs download included): " + " ".join(f"{t:.0f}" for t in obs_host) +
          f" | median {np.median(obs_host):.0f}")
    print("  dwt_observe us (events, stamp claim + k_band_obs + claim reset): " + " ".join(f"{t:.1f}" for t in obs_dev) +
          f" | median {np.median(obs_dev):.1f}")
    print("  dwt_decide(mlp) us (events, k_mlp_act + k_band_decide): " + " ".join(f"{t:.1f}" for t in decide) +
          f" | median {np.median(decide):.1f}")
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        w.band.run_local(16, "mlp")
        torch.cuda.synchronize()
    w._pending += 16
    w.end_chunk()
    print("  kernels of 16 mlp steps (torch.profiler, separate run): mean us per launch x launches")
    for ev in sorted(prof.key_averages(), key=lambda e: -e.device_time_total):
        if ev.device_time_total > 0 and ev.count > 0:
            print(f"    {ev.key[:60]:60s} {ev.device_time_total / ev.count:9.1f} x {ev.count}")
    sys.stdout.flush()


def bench_diag(N, K=32, reps=5):
    w = BandedDaisyWorld(N, N)
    w.reset_on_device(seed=1)
    w.run(2, "greedy")

    def timed(fn):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) * 1e3

    def step():
        w.band.run_local(K, "greedy")
        w._pending += K
        w.end_chunk()

    calls = {"greedy step": lambda: timed(step) / K,
             'diag_stats("temp")': lambda: timed(lambda: w.diag_stats("temp")),
             'image("temp", 16)': lambda: timed(lambda: w.image("temp", 16)),
             'image("grid_light", 16)': lambda: timed(lambda: w.image("grid_light", 16)),
             "cover_stats()": lambda: timed(w.cover_stats),
             'dwt_pool("temp", 16) alone': lambda: timed(lambda: w.band.pool("temp", 16))}
    for fn in calls.values():                    # warm-up: module loading, lazy buffers
        fn()
    times = {k: [] for k in calls}
    for _ in range(reps):
        for k, fn in calls.items():
            times[k].append(fn())
    print(f"N={N}, {N} agents, greedy, {reps} alternating repetitions (CUDA events around each call, download included)")
    for k, ts in times.items():
        print(f"  {k:26s} us: " + " ".join(f"{t:.0f}" for t in ts) + f" | median {np.median(ts):.0f}")
    t, img = w.diag_stats("temp"), w.image("temp", 16)
    print(f"  check: temp mean {t['mean']:.6f} K, std {t['std']:.6f}; mean of the 16-block image {img.mean():.6f}", flush=True)


def bench_snapshot(N, reps=3):
    import shutil, tempfile
    w = BandedDaisyWorld(N, N)
    w.reset_on_device(seed=1)
    w.run(3, "greedy")
    b = w.band
    tmp = tempfile.mkdtemp(prefix="dw_snapshot_bench_")
    path = os.path.join(tmp, "snap")

    def clock(fn):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        r = fn()
        torch.cuda.synchronize()
        return (time.perf_counter() - t0) * 1e3, r

    nbytes = N * N * 4
    dev = torch.empty(nbytes // 4, dtype=torch.int32, device="cuda")
    pin = torch.empty(nbytes // 4, dtype=torch.int32, pin_memory=True)
    meta, cur, pre, ada = b.save_state()                # warm-up: staging buffer, page faults of the arrays
    rows = np.concatenate([cur[-1:], cur, cur[:1]])        # the band's rows with both ghost rows (one band: the torus wrap)
    prows = np.concatenate([pre[-1:], pre, pre[:1]])
    b.restore_state(meta, rows, prows, ada)
    w.save(path)
    w.restore(path)
    cs = w.cover_checksum()
    times = {k: [] for k in ("pcie d2h (pinned, 1 copy)", "pcie h2d (pinned, 1 copy)", "save_state -> RAM (cur + pre)",
                             "np.save of both shards", "save() whole", "read both shards (np.load)",
                             "restore_state <- RAM (cur + pre)", "checksums (cur + pre)", "restore() whole")}
    for _ in range(reps):
        times["pcie d2h (pinned, 1 copy)"].append(clock(lambda: pin.copy_(dev))[0])
        times["pcie h2d (pinned, 1 copy)"].append(clock(lambda: dev.copy_(pin))[0])
        times["save_state -> RAM (cur + pre)"].append(clock(lambda: b.save_state(lambda which, shape, dtype: cur if which == "cur" else pre))[0])
        times["np.save of both shards"].append(clock(lambda: [np.save(os.path.join(tmp, f"{k}.npy"), a) for k, a in (("c", cur), ("p", pre))])[0])
        times["save() whole"].append(clock(lambda: w.save(path))[0])
        times["read both shards (np.load)"].append(clock(lambda: [np.array(np.load(os.path.join(tmp, f"{k}.npy"), mmap_mode="r")) for k in "cp"])[0])
        times["restore_state <- RAM (cur + pre)"].append(clock(lambda: b.restore_state(meta, rows, prows, ada))[0])
        times["checksums (cur + pre)"].append(clock(lambda: (b.cover_checksum(), b.pre_checksum()))[0])
        times["restore() whole"].append(clock(lambda: w.restore(path))[0])
    assert w.cover_checksum() == cs
    shutil.rmtree(tmp)
    print(f"N={N}, {N} agents, after 3 greedy steps (lattice + lattice pre-state, {nbytes / 2**30:.2f} GiB per state and band); "
          f"{reps} repetitions, host clock around synchronising calls (ms)")
    for k, ts in times.items():
        print(f"  {k:36s} ms: " + " ".join(f"{t:.1f}" for t in ts) + f" | median {np.median(ts):.1f}")
    print(f"  pcie floor of one state: {nbytes / np.median(times['pcie d2h (pinned, 1 copy)']) / 1e6:.1f} GB/s d2h, "
          f"{nbytes / np.median(times['pcie h2d (pinned, 1 copy)']) / 1e6:.1f} GB/s h2d", flush=True)


def bench_f32(N, reps=5, calls=10):
    w = BandedDaisyWorld(N, N)
    w.reset_on_device(seed=1)
    w.run(3, "greedy")
    b = w.band
    for fp32 in (True, False):                   # warm-up: module loading, the fp32 buffer and the fp64 scratch
        b.time_materialise(fp32, 2)
    s0 = b.f32_stats()
    times = {True: [], False: []}
    for _ in range(reps):
        for fp32 in (True, False):
            times[fp32].append(b.time_materialise(fp32, calls))
    s1 = b.f32_stats()
    cells = N * N
    tier, lit = (s1["fp64_tier"] - s0["fp64_tier"]) / (s1["cells"] - s0["cells"]), (s1["literal"] - s0["literal"]) / (s1["cells"] - s0["cells"])
    print(f"N={N}, {N} agents, after 3 greedy steps; device time per materialisation (dwt_debug_time_materialise, CUDA events), "
          f"{reps} alternating repetitions of {calls} calls")
    for fp32, name, nbytes in ((True, "fp32 mode", 36), (False, "fp64 grid", 60)):
        ts = np.array(times[fp32])
        med = np.median(ts)
        rate = nbytes * cells / (med * 1e-6)
        print(f"  {name} us: " + " ".join(f"{t:.0f}" for t in ts) + f" | median {med:.0f} us = {cells / (med * 1e-6):.3e} cells/s, "
              f"{nbytes} B/cell algorithmic = {rate / 1e12:.2f} TB/s = {rate / 7.7e12:.2f} of the 7.7 TB/s data-sheet HBM bandwidth")
    print(f"  fp32 / fp64 device time: {np.median(times[True]) / np.median(times[False]):.3f}")
    print(f"  fp32 mode tiers: {100 * tier:.3f} % of cells to the fp64 tier, {100 * lit:.5f} % to the literal cell")
    host = {"local_grid_f32()": [], "local_grid()": []}
    for _ in range(3):
        for name, fn in (("local_grid_f32()", w.local_grid_f32), ("local_grid()", w.local_grid)):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            g = fn()
            host[name].append((time.perf_counter() - t0) * 1e3)
            del g
    for name, ts in host.items():
        print(f"  {name:17s} ms (host clock, download included): " + " ".join(f"{t:.0f}" for t in ts) + f" | median {np.median(ts):.0f}")
    t = w.local_grid_f32_tensor()
    print(f"  check: local_grid_f32_tensor() {tuple(t.shape)} {t.dtype}, mean T {t[3].double().mean().item():.4f} K", flush=True)


def bench_vs_ensemble(N, K=200, reps=5):
    from therldaisyworld_b200 import RLDaisyWorld
    n = 4
    giant = BandedDaisyWorld(N, n)
    giant.reset_on_device(seed=1)
    giant.run(2, "greedy")
    env = RLDaisyWorld(grid_dimension=N, n_agents=n, device=0)
    env.batch_size = 1
    env.reset()
    env.run(2, policy="greedy")
    times = {"giant": [], "ensemble": []}
    for _ in range(reps):
        for arm in times:
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            if arm == "giant":
                giant.run(K, "greedy", chunk=K)
            else:
                env.run(K, policy="greedy")
            torch.cuda.synchronize()
            times[arm].append((time.perf_counter() - t0) / K * 1e6)
    print(f"N={N}, {n} agents, greedy, K={K} steps per run() call, {reps} alternating repetitions (host clock, synchronised)")
    for arm, ts in times.items():
        print(f"  {arm:8s} us/step: " + " ".join(f"{t:.1f}" for t in ts) + f" | median {np.median(ts):.1f}")
    print(f"  ensemble / giant: {np.median(times['ensemble']) / np.median(times['giant']):.2f}x", flush=True)


if __name__ == "__main__":
    if "--sides" in sys.argv or "--vs-ensemble" in sys.argv:
        print(f"GPU: {gpu_label()}")
        args = [int(a) for a in sys.argv[1:] if not a.startswith("--")]
        if "--sides" in sys.argv:
            bench_sides(args)
        else:
            bench_vs_ensemble(args[0])
        sys.exit(0)
    if "--policy" in sys.argv:
        args = [a for a in sys.argv[1:] if not a.startswith("--")]
        assert args and args[0] == "mlp", "--policy mlp [N]"
        print(f"GPU: {gpu_label()}")
        bench_mlp(int(args[1]) if len(args) > 1 else 16384)
        sys.exit(0)
    if "--diag" in sys.argv:
        args = [a for a in sys.argv[1:] if a != "--diag"]
        print(f"GPU: {gpu_label()}")
        bench_diag(int(args[0]) if args else 16384)
        sys.exit(0)
    if "--snapshot" in sys.argv:
        args = [a for a in sys.argv[1:] if a != "--snapshot"]
        print(f"GPU: {gpu_label()}")
        bench_snapshot(int(args[0]) if args else 16384)
        sys.exit(0)
    if "--f32" in sys.argv:
        args = [a for a in sys.argv[1:] if a != "--f32"]
        print(f"GPU: {gpu_label()}")
        bench_f32(int(args[0]) if args else 16384)
        sys.exit(0)
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
