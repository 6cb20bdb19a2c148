"""Next-row N2 on the GPU: the population fitness rollout reproduces the values recorded from the live reference's
SimpleGaussianES.get_fitness (oracle/gen_golden_es.py) -- same reset draws, same stopping steps, same per-agent step
totals; fitness within the summation-order tolerance stated below."""
import json
import os

import numpy as np
import pytest

from conftest import GOLDEN_DIR

pytestmark = pytest.mark.gpu


def test_population_rollout_matches_reference_get_fitness():
    from therldaisyworld_b200.es import evaluate_population
    z = np.load(os.path.join(GOLDEN_DIR, "es_fitness_p4_n16.npz"))
    meta = json.loads(str(z["meta"]))
    np.random.seed(meta["reset_seed"])
    fitness, total_steps, member_steps, env = evaluate_population(z["params"], adversary_idx=meta["adversary_idx"],
                                                                   max_steps=meta["max_steps"], worlds_per_member=meta["batch_size"],
                                                                   grid_dimension=meta["grid_dimension"])
    np.testing.assert_array_equal(member_steps, meta["steps_run"])
    np.testing.assert_array_equal(total_steps, z["total_steps"])
    np.testing.assert_array_equal(total_steps, z["done_at"])
    # fitness is a sum over steps of means over 64 rewards: the device reduces in a different order than np.mean
    np.testing.assert_allclose(fitness, z["fitness"], rtol=1e-12, atol=0)


def test_population_rollout_at_n64_matches_oracle():
    """64x64 worlds (the fused kernel's path), 3 members x 8 worlds, against the NumPy restatement of get_fitness."""
    from therldaisyworld_b200.es import evaluate_population
    from oracle.daisy_numpy import OracleDaisyWorld, OracleMLP, es_get_fitness
    base = np.load(os.path.join(GOLDEN_DIR, "mlp_n16_b4_mixed_150.npz"))["mlp_params"]
    members = np.stack([np.zeros_like(base), base, base + np.random.RandomState(4).randn(base.size)])
    np.random.seed(5)
    fitness, total_steps, member_steps, env = evaluate_population(members, adversary_idx=1, max_steps=30, worlds_per_member=8,
                                                                   grid_dimension=64, n_agents=6)
    oenv = OracleDaisyWorld(grid_dimension=64, n_agents=6)
    oenv.batch_size = 8
    pop = [OracleMLP(p) for p in members]
    np.random.seed(5)
    for m in range(3):
        f, ts, da, steps = es_get_fitness(oenv, pop[m], pop[1], max_steps=30)
        assert steps == member_steps[m]
        np.testing.assert_array_equal(ts, total_steps[m])
        np.testing.assert_allclose(fitness[m], f, rtol=1e-12)


@pytest.mark.parametrize("N,P,W,n,max_steps", [(64, 3, 8, 6, 90)])
def test_fused_population_segments_equal_the_per_step_path(monkeypatch, N, P, W, n, max_steps):
    """Population rollouts run as fused 64-step segments (policy inside the persistent 64x64 kernel, per-step agent states recorded,
    members' bookkeeping in one post-pass, k_pop_post); DW_POP_UNFUSED=1 keeps the per-step launch sequence: same fitness bit
    for bit (same summation order), same stopping steps and step totals."""
    from therldaisyworld_b200.es import evaluate_population
    rng = np.random.RandomState(9)
    members = rng.randn(P, 1808) * 0.7
    members[0] = 0.0
    out = []
    for unfused in (False, True):
        if unfused:
            monkeypatch.setenv("DW_POP_UNFUSED", "1")
        else:
            monkeypatch.delenv("DW_POP_UNFUSED", raising=False)
        np.random.seed(21)
        fitness, total_steps, member_steps, env = evaluate_population(members, adversary_idx=1, max_steps=max_steps, worlds_per_member=W,
                                                                       grid_dimension=N, n_agents=n)
        out.append((fitness, total_steps, member_steps, env.agent_states.copy(), env.agent_indices.copy()))
    a, b = out
    np.testing.assert_array_equal(a[2], b[2])
    np.testing.assert_array_equal(a[1], b[1])
    np.testing.assert_array_equal(a[0], b[0])
    assert (a[2] > 1).all()
