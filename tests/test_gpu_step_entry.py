"""Every source of a step's actions through the public stepping calls: explicit actions (full and partial), step(None), the
device policies greedy, eps_greedy and random, and the device MLP, each on the lean (fused) path and on the materialising
path (partial actions, the daisy_asym kernels), without and with collisions, at 16x16 and 64x64. Every step's outputs,
agents and clock equal the oracle's (the C oracle; the NumPy oracle with collisions, on the same global stream), and
every step launches the kernels a fixed table records, so no path can drift to another one unnoticed."""
import ctypes as C

import numpy as np
import pytest

from kernel_sets import set_kernels

pytestmark = pytest.mark.gpu

SHAPES = {16: (3, 4), 64: (2, 5)}          # N -> (worlds, agents)
SOURCES = ["full", "partial", "none", "greedy", "eps_greedy", "random", "mlp"]
STEPS = 4
SEED = 7
EPSILON = 0.5

# kernel launches of each step ("source-kernels-collision_mode-N"; update_run: the two update_agents calls, then the two
# runs), as recorded from the library before a step's action sources were resolved in one place
LAUNCHES = {
    "full-default-0-16": [4, 2, 2, 2], "full-default-0-64": [4, 2, 2, 2],
    "full-default-1-16": [5, 5, 5, 5], "full-default-1-64": [5, 5, 5, 5],
    "full-daisy_asym-0-16": [4, 4, 4, 4], "full-daisy_asym-0-64": [4, 4, 4, 4],
    "full-daisy_asym-1-16": [5, 5, 5, 5], "full-daisy_asym-1-64": [5, 5, 5, 5],
    "partial-default-0-16": [4, 4, 4, 4], "partial-default-0-64": [4, 4, 4, 4],
    "partial-default-1-16": [5, 5, 5, 5], "partial-default-1-64": [5, 5, 5, 5],
    "partial-daisy_asym-0-16": [4, 4, 4, 4], "partial-daisy_asym-0-64": [4, 4, 4, 4],
    "partial-daisy_asym-1-16": [5, 5, 5, 5], "partial-daisy_asym-1-64": [5, 5, 5, 5],
    "none-default-0-16": [4, 2, 2, 2], "none-default-0-64": [4, 2, 2, 2],
    "none-default-1-16": [5, 5, 5, 5], "none-default-1-64": [5, 5, 5, 5],
    "none-daisy_asym-0-16": [4, 4, 4, 4], "none-daisy_asym-0-64": [4, 4, 4, 4],
    "none-daisy_asym-1-16": [5, 5, 5, 5], "none-daisy_asym-1-64": [5, 5, 5, 5],
    "greedy-default-0-16": [4, 2, 2, 2], "greedy-default-0-64": [4, 2, 2, 2],
    "greedy-default-1-16": [5, 5, 5, 5], "greedy-default-1-64": [5, 5, 5, 5],
    "greedy-daisy_asym-0-16": [4, 4, 4, 4], "greedy-daisy_asym-0-64": [4, 4, 4, 4],
    "greedy-daisy_asym-1-16": [5, 5, 5, 5], "greedy-daisy_asym-1-64": [5, 5, 5, 5],
    "eps_greedy-default-0-16": [4, 2, 2, 2], "eps_greedy-default-0-64": [4, 2, 2, 2],
    "eps_greedy-default-1-16": [5, 5, 5, 5], "eps_greedy-default-1-64": [5, 5, 5, 5],
    "eps_greedy-daisy_asym-0-16": [4, 4, 4, 4], "eps_greedy-daisy_asym-0-64": [4, 4, 4, 4],
    "eps_greedy-daisy_asym-1-16": [5, 5, 5, 5], "eps_greedy-daisy_asym-1-64": [5, 5, 5, 5],
    "random-default-0-16": [4, 2, 2, 2], "random-default-0-64": [4, 2, 2, 2],
    "random-default-1-16": [5, 5, 5, 5], "random-default-1-64": [5, 5, 5, 5],
    "random-daisy_asym-0-16": [4, 4, 4, 4], "random-daisy_asym-0-64": [4, 4, 4, 4],
    "random-daisy_asym-1-16": [5, 5, 5, 5], "random-daisy_asym-1-64": [5, 5, 5, 5],
    "mlp-default-0-16": [6, 3, 3, 3], "mlp-default-0-64": [6, 3, 3, 3],
    "mlp-default-1-16": [7, 6, 6, 6], "mlp-default-1-64": [7, 6, 6, 6],
    "mlp-daisy_asym-0-16": [6, 5, 5, 5], "mlp-daisy_asym-0-64": [6, 5, 5, 5],
    "mlp-daisy_asym-1-16": [7, 6, 6, 6], "mlp-daisy_asym-1-64": [7, 6, 6, 6],
    "update_run-0-16": [1, 1, 6, 1], "update_run-0-64": [1, 1, 6, 1],
    "update_run-1-16": [2, 2, 12, 12], "update_run-1-64": [2, 2, 12, 12],
}

M64 = (1 << 64) - 1


def _hash_rng(seed, world, agent, step):
    """dw_hash_rng (csrc/dw_generic.cuh), the device counter RNG of the random and eps_greedy policies."""
    z = (seed + 0x9E3779B97F4A7C15 * (world * 0x10001 + agent + 1) + (step << 32)) & M64
    z = ((z ^ (z >> 30)) * 0xBF58476D1CE4E5B9) & M64
    z = ((z ^ (z >> 27)) * 0x94D049BB133111EB) & M64
    return (z ^ (z >> 31)) >> 32


def _greedy(obs):
    """Greedy's argmax branch on the observation of the current state (first maximum of the four neighbours' covers)."""
    B, n = obs.shape[:2]
    food = (obs[..., 1, :, :] + obs[..., 2, :, :]).reshape(B, n, 9)[:, :, [3, 1, 7, 5]]
    return 4 + np.argmax(food, axis=-1)[..., None]


def _random(B, n, step):
    return np.array([[_hash_rng(SEED, b, i, step) % 9 for i in range(n)] for b in range(B)])[..., None]


def _device_action(source, obs, step, mlp):
    """The action a device policy takes at clock step `step`, from the observation of the current state."""
    B, n = obs.shape[:2]
    if source == "greedy":
        return _greedy(obs)
    if source == "random":
        return _random(B, n, step)
    if source == "eps_greedy":        # one coin per step for the whole ensemble (dw_resolve_policy)
        coin = _hash_rng(SEED ^ 0x5EEDC01D5EEDC01D, 0xFFFFFFFF, 0xFFFFFFFF, step) * (1.0 / 4294967296.0)
        return _random(B, n, step) if coin < EPSILON else _greedy(obs)
    return mlp(obs)


def _profile_start(env):
    assert env._lib.dw_set_profiling(env._h, 1) == 0


def _launches(env):
    from therldaisyworld_b200._lib import DwProfile
    prof = DwProfile()
    assert env._lib.dw_get_profile(env._h, C.byref(prof)) == 0
    assert env._lib.dw_set_profiling(env._h, 0) == 0
    return int(prof.kernel_launches)


def _worlds(N, collision_mode, kernels, seed):
    """The product env after reset() and an oracle holding the same state (C oracle, or NumPy oracle with collisions)."""
    from therldaisyworld_b200 import RLDaisyWorld
    from oracle.daisy_c import COracleWorld
    from oracle.daisy_numpy import OracleDaisyWorld
    B, n = SHAPES[N]
    np.random.seed(seed)
    env = RLDaisyWorld(grid_dimension=N, n_agents=n, collision_mode=collision_mode)
    env.batch_size = B
    set_kernels(env, kernels)
    env.reset()
    if collision_mode == 0:
        return env, COracleWorld(env)
    ref = OracleDaisyWorld(grid_dimension=N, n_agents=n, collision_mode=1)
    ref.batch_size = B
    set_kernels(ref, kernels)
    ref.reset()
    ref.grid, ref.agent_indices, ref.agent_states = env.grid.copy(), env.agent_indices.copy(), env.agent_states.copy()
    return env, ref


def _same_stream(env_call, ref_call):
    """Both calls draw the collision noise from the global stream: run them from the same stream state."""
    state = np.random.get_state()
    got = env_call()
    after_env = np.random.get_state()
    np.random.set_state(state)
    want = ref_call()
    after_ref = np.random.get_state()
    assert after_env[2] == after_ref[2] and np.array_equal(after_env[1], after_ref[1])
    return got, want


def _assert_agents_and_clock(env, ref):
    B, n = SHAPES[env.dim]
    np.testing.assert_array_equal(env.agent_indices, ref.agent_indices)
    np.testing.assert_array_equal(env.agent_states.reshape(B, n), ref.agent_states.reshape(B, n))
    assert env.L == ref.L and env.step_count == ref.step_count


@pytest.mark.parametrize("N", sorted(SHAPES))
@pytest.mark.parametrize("collision_mode", [0, 1])
@pytest.mark.parametrize("kernels", ["default", "daisy_asym"])
@pytest.mark.parametrize("source", SOURCES)
def test_step_from_every_action_source(source, kernels, collision_mode, N):
    from oracle.daisy_numpy import OracleMLP
    B, n = SHAPES[N]
    env, ref = _worlds(N, collision_mode, kernels, seed=N + collision_mode)
    rng = np.random.RandomState(SOURCES.index(source))
    mlp = None
    if source == "mlp":
        params = rng.randn(OracleMLP.N_PARAMS)
        env.set_mlp(params)
        mlp = OracleMLP(params)
    if source == "eps_greedy":
        env.set_epsilon(EPSILON)
    obs_ref = ref.get_obs() if collision_mode == 0 else ref.get_obs(ref.agent_indices)
    launches = []
    for t in range(STEPS):
        if source == "full":
            action = rng.randint(9, size=(B, n, 1))
        elif source == "partial":
            action = rng.randint(9, size=(B - 1, n - 2, 1))
        elif source == "none":
            action = None
        else:
            action = _device_action(source, obs_ref, ref.step_count, mlp)
        if source in ("full", "partial", "none"):
            def env_step():
                return env.step(action)
        else:
            def env_step():
                return env.step_policy(source, seed=SEED)
        _profile_start(env)
        if collision_mode == 0:
            (o1, r1, d1, info), (obs_ref, r2, d2, _) = env_step(), ref.step(action)
        else:
            (o1, r1, d1, info), (obs_ref, r2, d2, _) = _same_stream(env_step, lambda: ref.step(action))
        launches.append(_launches(env))
        assert info == {}
        assert o1.shape == (B, n, 7, 3, 3) and r1.shape == d1.shape == (B, n, 1) and d1.dtype == np.bool_
        np.testing.assert_array_equal(o1, obs_ref)
        np.testing.assert_array_equal(r1, r2)
        np.testing.assert_array_equal(d1, d2)
        _assert_agents_and_clock(env, ref)
    np.testing.assert_array_equal(env.grid, ref.grid)
    case = f"{source}-{kernels}-{collision_mode}-{N}"
    assert launches == LAUNCHES.get(case), f"LAUNCHES {case!r}: {launches},"


@pytest.mark.parametrize("N", sorted(SHAPES))
@pytest.mark.parametrize("collision_mode", [0, 1])
def test_update_agents_and_run(N, collision_mode):
    """update_agents (full and partial actions) and run() under greedy and replay: with collisions run() steps through
    dw_agents_begin like step() does."""
    from oracle.daisy_numpy import OracleDaisyWorld
    B, n = SHAPES[N]
    env, _ = _worlds(N, collision_mode, "default", seed=100 + N)
    ref = OracleDaisyWorld(grid_dimension=N, n_agents=n, collision_mode=collision_mode)
    ref.batch_size = B
    ref.reset()
    ref.grid, ref.agent_indices, ref.agent_states = env.grid.copy(), env.agent_indices.copy(), env.agent_states.copy()
    rng = np.random.RandomState(N)
    launches = []
    for shape in [(B, n, 1), (B - 1, n - 2, 1)]:
        action = rng.randint(9, size=shape)
        _profile_start(env)
        _same_stream(lambda: env.update_agents(action), lambda: ref.update_agents(action))
        launches.append(_launches(env))
        _assert_agents_and_clock(env, ref)
    K = 3
    actions = rng.randint(9, size=(K, B, n))

    def ref_run(policy):
        for t in range(K):
            ref.step(_greedy(ref.get_obs(ref.agent_indices)) if policy == "greedy" else actions[t][..., None])

    for policy in ["greedy", "replay"]:
        _profile_start(env)
        _same_stream(lambda: env.run(K, policy=policy, actions=actions if policy == "replay" else None),
                     lambda: ref_run(policy))
        launches.append(_launches(env))
        _assert_agents_and_clock(env, ref)
    np.testing.assert_array_equal(env.grid, ref.grid)
    case = f"update_run-{collision_mode}-{N}"
    assert launches == LAUNCHES.get(case), f"LAUNCHES {case!r}: {launches},"
