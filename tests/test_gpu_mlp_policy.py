"""Next-row N1: the reference's MLP policy (daisy/agents/mlp.py) evaluated on the device (DW_POLICY_MLP). Fixtures were
recorded from the live reference MLP + RLDaisyWorld (oracle/gen_golden.py, cases mlp_*): actions are not fed in, the
device must pick them itself -- every state, reward and lifespan must still match the recording."""
import numpy as np
import pytest

from helpers import load_golden, product_env_from_golden

pytestmark = pytest.mark.gpu

# mlp_moore_* / mlp_circular_*: row A15, non-default observation masks applied on the device
CASES = ["mlp_n16_b4_200", "mlp_n64_b2_n6_60", "mlp_n16_b4_mixed_150", "mlp_moore_n16_b3_100", "mlp_circular_n16_b2_60"]


@pytest.mark.parametrize("name", CASES)
def test_fused_run_with_device_mlp_matches_reference(name):
    z, meta = load_golden(name)
    env = product_env_from_golden(z, meta)
    env.set_mlp(z["mlp_params"])
    env.reset_lifespans()
    K = meta["steps"]
    t = 0
    for s, i in sorted((int(s), i) for i, s in enumerate(z["ckpt_steps"])):
        env.run(s - t, policy="mlp")
        t = s
        np.testing.assert_array_equal(env.agent_indices, z["agent_indices"][t - 1])
        np.testing.assert_array_equal(env.agent_states, z["agent_states"][t - 1])
        np.testing.assert_array_equal(env.observe(), z["ckpt_obs"][i])          # lean observation path (windows only)
        np.testing.assert_array_equal(env.grid, z["ckpt_grid"][i])
    assert t == K
    done_at, agents_done_at = env.lifespans()
    np.testing.assert_array_equal(done_at, z["done_at"])
    np.testing.assert_array_equal(agents_done_at, z["agents_done_at"])
    assert env.L == z["L"][K] and env.step_count == meta["final_step_count"]


@pytest.mark.parametrize("name", ["mlp_n16_b4_mixed_150", "mlp_moore_n16_b3_100"])
def test_single_steps_with_device_mlp_match_reference(name):
    z, meta = load_golden(name)
    env = product_env_from_golden(z, meta)
    env.set_mlp(z["mlp_params"])
    for t in range(40):
        obs, reward, done, _ = env.step_policy("mlp")
        np.testing.assert_array_equal(env.agent_indices, z["agent_indices"][t])
        np.testing.assert_array_equal(reward, z["reward"][t])
        np.testing.assert_array_equal(done, z["done"][t])


def test_device_mlp_equals_oracle_mlp_on_random_weights():
    """Random networks (diverse actions incl. ties at 0 after ReLU): device MLP vs the NumPy restatement on the C oracle."""
    from therldaisyworld_b200 import RLDaisyWorld
    from oracle.daisy_c import COracleWorld
    from oracle.daisy_numpy import OracleMLP
    rng = np.random.RandomState(3)
    for trial in range(3):
        params = rng.randn(OracleMLP.N_PARAMS) * (0.3, 1.0, 3.0)[trial]
        np.random.seed(40 + trial)
        env = RLDaisyWorld(grid_dimension=64, n_agents=5)
        env.batch_size = 6
        env.reset()
        ref = COracleWorld(env)
        agent = OracleMLP(params)
        env.set_mlp(params)
        env.run(50, policy="mlp")
        obs = ref.get_obs()
        hist = np.zeros(9, dtype=int)
        for _ in range(50):
            a = agent(obs)
            hist += np.bincount(a.ravel(), minlength=9)
            obs, _, _, _ = ref.step(a)
        np.testing.assert_array_equal(env.grid, ref.grid)
        np.testing.assert_array_equal(env.agent_indices, ref.agent_indices)
        print("action histogram", hist)


def test_mlp_policy_needs_weights():
    from therldaisyworld_b200 import RLDaisyWorld, DaisyWorldError
    np.random.seed(0)
    env = RLDaisyWorld(grid_dimension=8)
    with pytest.raises(DaisyWorldError):
        env.run(2, policy="mlp")
    with pytest.raises(DaisyWorldError):
        env.set_mlp(np.zeros(7))


def test_in_kernel_mlp_equals_the_per_step_policy_path(monkeypatch):
    """64x64 worlds: windows + network run inside the persistent fused kernel (dw_mlp_decide64). Same worlds through the
    per-step path (k_obs_mlp between one-step launches, DW_MLP_UNFUSED=1): identical state, agents, rewards and lifespans.
    70 steps = several 16-step work items per world (the pre-state is handed from item to item through lat_pre), 300 worlds
    = more work items than resident CTAs."""
    from therldaisyworld_b200 import RLDaisyWorld
    rng = np.random.RandomState(11)
    params = rng.randn(1808) * 1.5
    out = []
    for unfused in (False, True):
        if unfused:
            monkeypatch.setenv("DW_MLP_UNFUSED", "1")
        else:
            monkeypatch.delenv("DW_MLP_UNFUSED", raising=False)
        np.random.seed(5)
        env = RLDaisyWorld(grid_dimension=64, n_agents=7)
        env.batch_size = 300
        env.reset()
        env.set_mlp(params)
        env.reset_lifespans()
        env.run(3, policy="mlp")
        env.run(70, policy="mlp")
        obs = env.observe()
        out.append((env.grid.copy(), env.agent_indices.copy(), env.agent_states.copy(), obs, env.lifespans()))
    a, b = out
    np.testing.assert_array_equal(a[0], b[0])
    np.testing.assert_array_equal(a[1], b[1])
    np.testing.assert_array_equal(a[2], b[2])
    np.testing.assert_array_equal(a[3], b[3])
    np.testing.assert_array_equal(a[4][0], b[4][0])
    np.testing.assert_array_equal(a[4][1], b[4][1])
    assert len(np.unique(a[1])) > 10          # the agents did move around
