"""Every kernel family against the C oracle under non-default stencil kernels and physics constants (tests/kernel_sets.py):
reset, single steps with their unrounded diagnostics, fused runs under three policies, the per-step series, the fp32
mode, and the giant world's refusal of what its tiled kernels cannot run."""
import ctypes as C

import numpy as np
import pytest

from kernel_sets import ASYMMETRIC, DRAWS, KERNEL_SETS, SHAPES, apply_draw, set_kernels  # noqa: F401 (SHAPES: the families)

pytestmark = pytest.mark.gpu

MAIN = [(64, 6, 4), (16, 9, 4), (20, 5, 3), (33, 3, 5), (5, 3, 2)]


def _cases():
    names = list(KERNEL_SETS)
    out = [(s, name, None) for name in names for s in MAIN]
    for i, s in enumerate([(8, 70, 3), (13, 4, 3), (2, 2, 1), (1, 2, 1)]):
        out += [(s, names[i % len(names)], None), (s, names[(i + 3) % len(names)], None)]
    for i in range(len(DRAWS)):
        out += [(s, "default", i) for s in (MAIN[i % len(MAIN)], MAIN[(i + 2) % len(MAIN)])]
    return out


CASES = _cases()
IDS = [f"N{s[0]}_B{s[1]}_n{s[2]}-{name}-{'draw%d' % d if d is not None else 'const'}" for s, name, d in CASES]


def _fused(name, draw):
    return name not in ASYMMETRIC and (draw is None or DRAWS[draw]["g"] > 0)


def _pair(shape, name, draw, seed):
    """Product env and NumPy oracle env in the same reset state (same draws from the global stream, same constants)."""
    from oracle.daisy_numpy import OracleDaisyWorld
    from therldaisyworld_b200 import RLDaisyWorld
    N, B, n = shape
    envs = []
    for cls in (RLDaisyWorld, OracleDaisyWorld):
        np.random.seed(seed)
        env = cls(grid_dimension=N, n_agents=n)
        env.batch_size = B
        if draw is not None:
            apply_draw(env, DRAWS[draw])
        set_kernels(env, name)
        env.reset()
        envs.append(env)
    return envs


def _diag_equal(env, w):
    d = w.forward_diag()
    for i, attr in enumerate(("temp", "temp_light", "temp_dark", "temp_effective", "beta", "beta_l", "beta_d")):
        np.testing.assert_array_equal(getattr(env, attr)[:, 0], d[:, i], err_msg=attr)
    np.testing.assert_array_equal(env.growth, d[:, 7:9])


@pytest.mark.parametrize("shape,name,draw", CASES, ids=IDS)
def test_reset_and_steps_match_c_oracle(shape, name, draw):
    from oracle.daisy_c import COracleWorld
    env, oenv = _pair(shape, name, draw, seed=sum(shape))
    w = COracleWorld(oenv)
    g = env.grid
    np.testing.assert_array_equal(g[:, 0:3], oenv.grid[:, 0:3])
    np.testing.assert_array_equal(g[:, 3:6], w.forward_diag()[:, 0:3])
    np.testing.assert_array_equal(env.agent_indices, w.agent_indices)
    B, n = shape[1], shape[2]
    rng = np.random.RandomState(7)
    for t in range(10):
        a = rng.randint(9, size=(B, n, 1))
        o1, r1, d1, _ = env.step(a)
        o2, r2, d2, _ = w.step(a)
        np.testing.assert_array_equal(env.grid, w.grid, err_msg=f"step {t}")
        np.testing.assert_array_equal(o1, o2)
        np.testing.assert_array_equal(r1, r2)
        np.testing.assert_array_equal(d1, d2)
        np.testing.assert_array_equal(env.agent_indices, w.agent_indices)
        np.testing.assert_array_equal(env.agent_states, w.agent_states)
    assert env.L == w.L and env.step_count == w.step_count
    env.forward(env.grid.copy())
    _diag_equal(env, w)


@pytest.mark.parametrize("shape,name,draw", CASES, ids=IDS)
def test_runs_match_c_oracle(shape, name, draw):
    from oracle.daisy_c import COracleWorld
    N, B, n = shape
    K = 300
    for policy in ("greedy", "antigreedy", "replay"):
        env, oenv = _pair(shape, name, draw, seed=sum(shape) + 1)
        w = COracleWorld(oenv)
        acts = np.random.RandomState(N).randint(9, size=(K, B, n)) if policy == "replay" else None
        env.reset_lifespans()
        env.run(K, policy=policy, actions=acts)
        _, done_at, agents_done_at = w.run(K, policy, actions=acts)
        np.testing.assert_array_equal(env.grid, w.grid, err_msg=policy)
        np.testing.assert_array_equal(env.agent_indices, w.agent_indices)
        np.testing.assert_array_equal(env.agent_states, w.agent_states)
        got_done_at, got_agents = env.lifespans()
        np.testing.assert_array_equal(got_done_at, done_at)
        np.testing.assert_array_equal(got_agents, agents_done_at)
        assert env.L == w.L and env.step_count == w.step_count == K
        if _fused(name, draw):
            slow = C.c_uint64()
            assert env._lib.dw_debug_slow_count(env._h, C.byref(slow), 0) == 0
            cells = K * B * N * N
            assert slow.value < 1e-3 * cells + 10, (policy, slow.value, cells)


@pytest.mark.parametrize("variant", ["daisy_asym", "g0"])
@pytest.mark.parametrize("N", [8, 16, 20, 64])
def test_run_series_off_the_fast_path_matches_oracle(N, variant):
    """run_series with constants the in-kernel series does not take: the device refuses before any step and the per-step
    loop runs instead, with the oracle's per-step means."""
    from oracle.daisy_numpy import OracleGreedy
    envs = _pair((N, 3, 4), "daisy_asym" if variant == "daisy_asym" else "default", None, seed=N)
    if variant == "g0":
        for e in envs:
            e.g = 0.0
    env, oenv = envs
    K = 40
    series = env.run_series(K, policy="greedy")
    agent = OracleGreedy()
    obs = oenv.get_obs(oenv.agent_indices)
    ref = np.zeros((K, 3))
    for t in range(K):
        obs, _, _, _ = oenv.step(agent(obs))
        ref[t] = [oenv.temp.mean(), oenv.grid[:, 1].mean(), oenv.grid[:, 2].mean()]
    np.testing.assert_array_equal(env.grid[:, 1:3], oenv.grid[:, 1:3])
    np.testing.assert_allclose(series, ref, rtol=1e-12, atol=0)
    assert env.step_count == K


@pytest.mark.parametrize("name", ["daisy_asym", "d4_custom"])
def test_fp32_mode_under_other_kernels(name):
    from oracle.daisy_c import COracleWorld
    env, oenv = _pair((64, 4, 4), name, None, seed=3)
    w = COracleWorld(oenv)
    env.run(50, policy="greedy")
    w.run(50, "greedy")
    g32 = env.grid_f32()
    ref = w.grid
    for ch in (0, 1, 2):
        np.testing.assert_array_equal(g32[:, ch], ref[:, ch].astype(np.float32))
    np.testing.assert_allclose(g32[:, 3:6], ref[:, 3:6], rtol=1e-5, atol=0)


def test_giant_world_refuses_what_its_kernels_cannot_run_and_runs_d4_custom():
    """dwt_set_config refuses non-D4 kernels and g = 0 like dwt_create (the tiled kernels read only the D4 classes and scale
    by g^2); an accepted D4 configuration with other values runs like the oracle."""
    from band_helpers import full_oracle, make_state
    from therldaisyworld_b200._lib import DaisyWorldError
    from therldaisyworld_b200.banded import BandedDaisyWorld
    N, n = 64, 6
    light, dark, ai, st = make_state(N, n, seed=5)
    w = BandedDaisyWorld(N, n)
    for bad in ("daisy_asym", "adj_asym", "g0"):
        saved = (w.daisy_kernel.copy(), w.adjacent_albedo_kernel.copy(), w.g)
        if bad == "g0":
            w.g = 0.0
        else:
            set_kernels(w, bad)
        with pytest.raises(DaisyWorldError, match="dwt_set_config"):
            w.load_state(light, dark, ai, st)
        w.daisy_kernel, w.adjacent_albedo_kernel, w.g = saved
    set_kernels(w, "d4_custom")
    w.load_state(light, dark, ai, st)
    ref = full_oracle(w, light, dark, ai, st)
    w.run(30, "greedy")
    _, done_at, ada = ref.run(30, "greedy")
    np.testing.assert_array_equal(w.local_grid(), ref.grid[0])
    xy, s = w.agents()
    np.testing.assert_array_equal(xy, ref.agent_indices[0])
    np.testing.assert_array_equal(s, ref.agent_states[0, :, 0])
    d, a = w.lifespans()
    assert d == int(done_at[0])
    np.testing.assert_array_equal(a, ada[0, :, 0])
