"""Every lattice kernel past the fast path's rounding window. The fast path rounds x + 0.5 (milli-cover) through a fixed-point
word with 12 integer bits, exact for x + 0.5 in [-2048, 2048); a cover update outside it must saturate at 0 or 1000 like the
reference's clip, not wrap modulo 4096 (csrc/dw_fused.cuh, DESIGN.md section 2). The shocks of kernel_sets.SCENARIOS reach that
regime through the public API only; each one's crossing of the window is proved on the CPU before anything runs on the GPU
(tests/test_fast_path_window_coverage.py runs the same proof without a GPU)."""
import ctypes as C

import numpy as np
import pytest

from band_helpers import ThreadComm, full_oracle, make_state, run_threads
from kernel_sets import SCENARIOS, apply_shock, make_env, undo_shock, window_crossings

pytestmark = pytest.mark.gpu


def _proved(name, *args, **kw):
    """The shocked step of this very configuration leaves the 12-bit window, stays inside the 16-bit one, and its fields are
    finite (NumPy oracle, before anything runs on the GPU)."""
    below, above, wide, finite = window_crossings(name, *args, **kw)
    assert finite, name
    assert below + above > 0 or not SCENARIOS[name]["crosses"], (name, args, below, above)
    assert wide == 0, (name, args, wide)
    return below, above


def _pair(name, shape, seed):
    """Product env and C oracle in scenario `name`'s reset state."""
    from oracle.daisy_c import COracleWorld
    from oracle.daisy_numpy import OracleDaisyWorld
    from therldaisyworld_b200 import RLDaisyWorld
    N, B, n = shape
    env = make_env(RLDaisyWorld, name, N, B, n, seed)
    oenv = make_env(OracleDaisyWorld, name, N, B, n, seed)
    return env, COracleWorld(oenv)


def _segments(name):
    sc = SCENARIOS[name]
    return [(sc["grow"], False), (1, True), (sc["settle"], False)]


def _slow_count(env):
    """Literal recomputations since the handle was created (the counter is never reset in between)."""
    count = C.c_uint64()
    assert env._lib.dw_debug_slow_count(env._h, C.byref(count), 0) == 0
    return count.value


def _assert_rare(slow, cell_updates):
    assert slow < 1e-3 * cell_updates + 10, (slow, cell_updates)


# every fused family (tests/kernel_sets.py::SHAPES, csrc/dw_run.inl::fused_kernel); (64, 3, 33) has more agents than the
# persistent 64x64 kernel takes (k_fused_n64), (32, 3, 4) is the third sub-64 instance
FAMILIES = [(64, 4, 4), (64, 3, 33), (8, 70, 3), (16, 9, 4), (32, 3, 4), (20, 5, 3), (13, 4, 3), (33, 3, 5), (5, 3, 2)]
# heat_graze crosses the window in a handful of cells only: none in the worlds of these two shapes
NOT_CROSSING = {("heat_graze", (13, 4, 3)), ("heat_graze", (5, 3, 2))}
FAMILY_CASES = [(s, name) for s in FAMILIES for name in SCENARIOS if (name, s) not in NOT_CROSSING]


@pytest.mark.parametrize("shape,name", FAMILY_CASES, ids=[f"N{s[0]}_B{s[1]}_n{s[2]}-{name}" for s, name in FAMILY_CASES])
def test_fused_families_saturate_like_the_oracle(shape, name):
    """run() in three segments (grow, the shocked step, settle), greedy and replay: grid, agents, lifespans, clock as the C
    oracle's, and the literal recomputations stay as rare as on unshocked runs."""
    N, B, n = shape
    for policy in ("greedy", "replay"):
        K = sum(k for k, _ in _segments(name))
        acts = np.random.RandomState(N).randint(9, size=(K, B, n)) if policy == "replay" else None
        _proved(name, N, B, n, N + B + n, actions=acts)
        env, w = _pair(name, shape, seed=N + B + n)
        env.reset_lifespans()
        done_at, ada, t = np.zeros(B, dtype=np.int64), np.zeros((B, n, 1), dtype=np.int64), 0
        for k, shocked in _segments(name):
            saved = apply_shock(name, env, w) if shocked else None
            a = None if acts is None else acts[t:t + k]
            env.run(k, policy=policy, actions=a)
            _, d, g = w.run(k, policy, actions=a)
            done_at += d
            ada += g
            t += k
            if shocked:
                undo_shock(name, saved, env, w)
        np.testing.assert_array_equal(env.grid, w.grid, err_msg=policy)
        np.testing.assert_array_equal(env.agent_indices, w.agent_indices)
        np.testing.assert_array_equal(env.agent_states, w.agent_states)
        got_done_at, got_ada = env.lifespans()
        np.testing.assert_array_equal(got_done_at, done_at)
        np.testing.assert_array_equal(got_ada, ada)
        assert env.L == w.L and env.step_count == w.step_count == K
        _assert_rare(_slow_count(env), K * B * N * N)


@pytest.mark.parametrize("N", [64, 16, 20])
def test_in_kernel_series_under_the_heat_step(N):
    """run_series (series instances of the 64x64 and sub-64 kernels, and the 4x4-tile kernel's per-step path) across the heat
    step: per-step means as the NumPy oracle's, final grid equal."""
    from oracle.daisy_numpy import OracleDaisyWorld, OracleGreedy
    from therldaisyworld_b200 import RLDaisyWorld
    _proved("heat_step", N, 4, 4, N)
    K = 30
    env = make_env(RLDaisyWorld, "heat_step", N, 4, 4, seed=N)
    oenv = make_env(OracleDaisyWorld, "heat_step", N, 4, 4, seed=N)
    series = env.run_series(K, policy="greedy")
    agent = OracleGreedy()
    obs = oenv.get_obs(oenv.agent_indices)
    ref = np.zeros((K, 3))
    for t in range(K):
        obs, _, _, _ = oenv.step(agent(obs))
        ref[t] = [oenv.temp.mean(), oenv.grid[:, 1].mean(), oenv.grid[:, 2].mean()]
    np.testing.assert_allclose(series[:, 0], ref[:, 0], rtol=1e-9)
    np.testing.assert_allclose(series[:, 1:], ref[:, 1:], rtol=1e-12)
    np.testing.assert_array_equal(env.grid, oenv.grid)


def test_in_kernel_mlp_under_the_heat_pulse():
    """The MLP policy inside the persistent 64x64 kernel, across the heat pulse, against the NumPy MLP on the C oracle."""
    from helpers import load_golden
    from oracle.daisy_numpy import OracleMLP
    z, _ = load_golden("mlp_n64_b2_n6_60")
    params = z["mlp_params"]
    _proved("heat_pulse", 64, 4, 6, 9, actions=OracleMLP(params))
    env, w = _pair("heat_pulse", (64, 4, 6), seed=9)
    env.set_mlp(params)
    agent = OracleMLP(params)
    for k, shocked in _segments("heat_pulse"):
        saved = apply_shock("heat_pulse", env, w) if shocked else None
        env.run(k, policy="mlp")
        obs = w.get_obs()
        for _ in range(k):
            obs, _, _, _ = w.step(agent(obs))
        if shocked:
            undo_shock("heat_pulse", saved, env, w)
    np.testing.assert_array_equal(env.grid, w.grid)
    np.testing.assert_array_equal(env.agent_indices, w.agent_indices)
    np.testing.assert_array_equal(env.agent_states, w.agent_states)


@pytest.mark.parametrize("N", [64, 16])
def test_trimmed_segments_under_the_heat_step(N):
    """ensemble.simulate_lifespan (segments run masked past the stopping step, then trimmed): lifespans as the oracle's."""
    from therldaisyworld_b200.ensemble import DeviceShard, simulate_lifespan
    _proved("heat_step", N, 6, 4, 3)
    env, w = _pair("heat_step", (N, 6, 4), seed=3)
    out = simulate_lifespan(DeviceShard(env), policy="greedy", device="cuda")
    steps, done_at, ada = w.run(100000, "greedy", stop_all_done=True)
    assert out["steps"] == steps and out["all_done"]
    _assert_rare(_slow_count(env), steps * 6 * N * N)
    got_done_at, got_ada = env.lifespans()
    np.testing.assert_array_equal(got_done_at, done_at)
    np.testing.assert_array_equal(got_ada, ada)


def test_drop_in_step_under_every_shock():
    """step() one step at a time (lattice-resident one-step launches), the shocks set as attributes between steps: obs, reward,
    done, grid and agents every step; after each shock the fp32 mode's covers and bare fraction as the oracle's."""
    for name in SCENARIOS:
        K = sum(k for k, _ in _segments(name))
        rng = np.random.RandomState(5)
        acts = [rng.randint(9, size=(3, 4, 1)) for _ in range(K)]
        _proved(name, 64, 3, 4, 21, actions=acts)
        env, w = _pair(name, (64, 3, 4), seed=21)
        steps = iter(acts)
        for k, shocked in _segments(name):
            saved = apply_shock(name, env, w) if shocked else None
            for _ in range(k):
                a = next(steps)
                o1, r1, d1, _ = env.step(a)
                o2, r2, d2, _ = w.step(a)
                np.testing.assert_array_equal(env.grid, w.grid, err_msg=f"{name} step {env.step_count}")
                np.testing.assert_array_equal(o1, o2)
                np.testing.assert_array_equal(r1, r2)
                np.testing.assert_array_equal(d1, d2)
                np.testing.assert_array_equal(env.agent_states, w.agent_states)
            if shocked:           # fp32 mode of the shocked step, materialised with the constants it ran with
                g32 = env.grid_f32()
                for ch in (0, 1, 2):
                    np.testing.assert_array_equal(g32[:, ch], w.grid[:, ch].astype(np.float32), err_msg=name)
                undo_shock(name, saved, env, w)
        _assert_rare(_slow_count(env), K * 3 * 64 * 64)


def _grown_state(N, n, seed, steps=40):
    """A state grown for `steps` steps at the default constants on the C oracle, for the giant world to load: its heat step
    then hits living covers."""
    from oracle.daisy_numpy import OracleDaisyWorld
    light, dark, ai, st = make_state(N, n, seed=seed)
    ref = full_oracle(OracleDaisyWorld(grid_dimension=N, n_agents=n), light, dark, ai, st)
    ref.run(steps, "greedy")
    return ref.grid[0, 1].copy(), ref.grid[0, 2].copy(), ref.agent_indices[0].copy(), ref.agent_states[0, :, 0].copy()


def _world(N, n, **kw):
    from therldaisyworld_b200.banded import BandedDaisyWorld
    return BandedDaisyWorld(N, n, **SCENARIOS["heat_step"]["ctor"], **kw)


def _heat(w):
    """The heat step's max_L on a giant world, with the clock step it implies (what load_state sets as well), so that an
    oracle built from the world before load_state runs the same clock."""
    for k, v in SCENARIOS["heat_step"]["attrs"].items():
        setattr(w, k, v)
    w.dL = (w.max_L - w.min_L) / w.ramp_period
    return w


def _compare_band(w, ref, done_at, ada):
    np.testing.assert_array_equal(w.local_grid(), ref.grid[0])
    xy, st = w.agents()
    np.testing.assert_array_equal(xy, ref.agent_indices[0])
    np.testing.assert_array_equal(st, ref.agent_states[0, :, 0])
    d, a = w.lifespans()
    assert d == int(done_at[0])
    np.testing.assert_array_equal(a, ada[0, :, 0])


@pytest.mark.parametrize("N", [128, 100])
def test_giant_world_one_band_under_the_heat_step(N):
    """k_tiled_step (N = 128) and its masked instance (N = 100): step 2 after load_state is the first tiled step, at L = 2.5."""
    n = 12
    state = _grown_state(N, n, seed=N)
    _proved("heat_step", N, 1, n, 0, state=state)
    w = _heat(_world(N, n))
    w.load_state(*state)
    ref = full_oracle(w, *state)
    w.run(24, "greedy", chunk=8)
    _, done_at, ada = ref.run(24, "greedy")
    assert w.L == ref.L and w.step_count == 24
    _compare_band(w, ref, done_at, ada)
    _assert_rare(w.band.slow_count(), 24 * N * N)


def test_giant_world_series_under_the_heat_step():
    """Series instance of k_tiled_step across the heat step: covers, agents, lifespans as the C oracle's."""
    N, n = 128, 10
    state = _grown_state(N, n, seed=3)
    _proved("heat_step", N, 1, n, 0, state=state)
    w = _heat(_world(N, n))
    w.load_state(*state)
    ref = full_oracle(w, *state)
    s = w.run_series(20, "greedy", chunk=8)
    _, done_at, ada = ref.run(20, "greedy")
    assert s.shape == (20, 3) and w.L == ref.L
    _compare_band(w, ref, done_at, ada)
    _assert_rare(w.band.slow_count(), 20 * N * N)


def test_giant_world_two_peer_bands_under_the_heat_step():
    """Two bands of one GPU in peer-memory mode: k_band_lookahead_decide re-evaluates the cells the agents look at through
    dw_fast_cell while the interior is still being stepped."""
    import torch
    N, n, bands = 256, 200, 2
    light, dark, ai, st = _grown_state(N, n, seed=17)
    _proved("heat_step", N, 1, n, 0, state=(light, dark, ai, st))
    shared = ThreadComm.Shared(bands)
    worlds = [_heat(_world(N, n, rank=r, world_size=bands, comm=ThreadComm(r, bands, shared), mode="p2p")) for r in range(bands)]
    streams = [torch.cuda.Stream() for _ in range(bands)]
    tables = [w.band.peer_buffers() for w in worlds]
    for r, w in enumerate(worlds):
        w.band.set_stream(streams[r].cuda_stream)
        w.band.attach_peers(r, tables)
    ref = full_oracle(worlds[0], light, dark, ai, st)
    out = {}

    def go(w):
        with torch.cuda.stream(streams[w.rank]):
            w.load_state(light, dark, ai, st)
            w.run(20, "greedy", chunk=8)
            out[w.rank] = (w.agents(), w.lifespans(), w.local_grid(), w.band.peer_timed_out(), w.L, w.band.slow_count())

    run_threads(worlds, go)
    _, done_at, ada = ref.run(20, "greedy")
    assert not any(out[r][3] for r in range(bands)), "a peer barrier timed out"
    np.testing.assert_array_equal(np.concatenate([out[r][2] for r in range(bands)], axis=1), ref.grid[0])
    for r in range(bands):
        assert out[r][4] == ref.L
        _assert_rare(out[r][5], 20 * N * N // bands)
        np.testing.assert_array_equal(out[r][0][0], ref.agent_indices[0])
        np.testing.assert_array_equal(out[r][0][1], ref.agent_states[0, :, 0])
        assert out[r][1][0] == int(done_at[0])
        np.testing.assert_array_equal(out[r][1][1], ada[0, :, 0])
