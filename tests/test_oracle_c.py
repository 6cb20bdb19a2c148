"""C oracle == NumPy oracle == reference-recorded fixtures (all value-identical in fp64)."""
import itertools
import json
import os

import numpy as np
import pytest

from conftest import GOLDEN_DIR, golden_names
from kernel_sets import DRAWS, KERNEL_SETS, apply_draw, set_kernels
from oracle.daisy_c import COracleWorld
from oracle.daisy_numpy import OracleDaisyWorld, OracleGreedy, env_from_golden, lifespan_loop


# collision_mode == 1 (collide_*) is restated in the NumPy oracle only: its RNG is NumPy's global stream
@pytest.mark.parametrize("name", [n for n in golden_names() if not n.startswith("collide_")])
def test_c_oracle_replays_reference_trajectory(name):
    z = np.load(os.path.join(GOLDEN_DIR, name + ".npz"))
    env, meta = env_from_golden(z)
    w = COracleWorld(env)
    ck = {int(s): i for i, s in enumerate(z["ckpt_steps"])}
    np.testing.assert_array_equal(w.get_obs(), z["init_obs"])
    for t in range(meta["steps"]):
        a = z["actions"][t]
        action = None if (a.shape == (1, 1, 1) and a[0, 0, 0] == -1) else a
        if meta["attrs"].get("ramp_up_down"):
            # min_L/max_L drift lives in the clock; compare L only
            pass
        assert w.L == z["L"][t]
        obs, reward, done, _ = w.step(action)
        np.testing.assert_array_equal(w.agent_indices, z["agent_indices"][t])
        np.testing.assert_array_equal(w.agent_states, z["agent_states"][t])
        np.testing.assert_array_equal(reward, z["reward"][t])
        np.testing.assert_array_equal(done, z["done"][t])
        np.testing.assert_array_equal(w.grid.sum(axis=(-2, -1)), z["chan_sum"][t])
        if (t + 1) in ck:
            np.testing.assert_array_equal(w.grid, z["ckpt_grid"][ck[t + 1]])
            np.testing.assert_array_equal(obs, z["ckpt_obs"][ck[t + 1]])
    assert w.L == z["L"][meta["steps"]]


@pytest.mark.parametrize("name,policy", [("greedy_n16_b4_todeath", "greedy"), ("antigreedy_n8_b16_todeath", "antigreedy"),
                                         ("random_n8_b8_todeath", "replay"), ("greedy_n5_b3_n2_todeath", "greedy"),
                                         ("cfg1_n16_b1_noagents_todeath", "none")])
def test_c_oracle_lifespan_run(name, policy):
    """dwo_run (fused policy + lifespan counters) reproduces the notebook metric of the reference."""
    z = np.load(os.path.join(GOLDEN_DIR, name + ".npz"))
    env, meta = env_from_golden(z)
    w = COracleWorld(env)
    steps, done_at, agents_done_at = w.run(100000 if policy != "replay" else meta["steps"], policy,
                                           actions=z["actions"] if policy == "replay" else None, stop_all_done=True)
    assert steps == meta["steps"]
    np.testing.assert_array_equal(done_at, z["done_at"])
    np.testing.assert_array_equal(agents_done_at, z["agents_done_at"])
    np.testing.assert_array_equal(w.grid, z["ckpt_grid"][-1])


def test_c_oracle_matches_numpy_oracle_random_states():
    """Arbitrary (off-lattice) states, odd N, many agents, degenerate 1x1 and 2x2 tori, every kernel set and constant
    draw of tests/kernel_sets.py: bit-identical to the NumPy oracle."""
    names = list(KERNEL_SETS)
    cases = [(name, None) for name in names] + [(names[(i + 1) % len(names)], d) for i, d in enumerate(DRAWS)]
    rng = np.random.RandomState(123)
    for (N, B, n), (kernels, draw) in itertools.product([(1, 2, 1), (2, 2, 1), (3, 2, 1), (4, 2, 3), (6, 3, 2), (9, 2, 5), (33, 2, 7)],
                                                        cases):
        np.random.seed(N)
        env = OracleDaisyWorld(grid_dimension=N, n_agents=n)
        env.batch_size = B
        if draw is not None:
            apply_draw(env, draw)
        set_kernels(env, kernels)
        env.reset()
        env.grid[:, 1] = rng.rand(B, N, N) * 0.6
        env.grid[:, 2] = rng.rand(B, N, N) * 0.4
        w = COracleWorld(env)
        for t in range(12):
            action = rng.randint(9, size=(B, n, 1))
            o1, r1, d1, _ = env.step(action)
            o2, r2, d2, _ = w.step(action)
            np.testing.assert_array_equal(env.grid, w.grid)
            np.testing.assert_array_equal(o1, o2)
            np.testing.assert_array_equal(r1, r2)
            np.testing.assert_array_equal(d1, d2)
            np.testing.assert_array_equal(env.agent_indices, w.agent_indices)
        diag = w.forward_diag()
        env.forward(env.grid.copy())
        np.testing.assert_array_equal(diag[:, 0:1], env.temp)
        np.testing.assert_array_equal(diag[:, 5:6], env.beta_l)
        np.testing.assert_array_equal(diag[:, 7:9], env.growth)


def test_markstein_division_exhaustive():
    """The kernels replace rint(x*1000)/1000 by a division-free sequence; it must equal the IEEE quotient for every
    lattice index that can occur (covers 0..1 -> 0..1000, temperatures up to 2000 K -> 2e6)."""
    from oracle.daisy_c import lib
    import ctypes as C
    fn = lib().dwo_check_markstein
    fn.restype = C.c_long
    fn.argtypes = [C.c_long]
    assert fn(2000000) == 0
