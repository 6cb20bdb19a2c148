"""The oracles' 3x3 stencil is the reference's ft_convolve (daisy/nn/functional.py:12-49), a circular CONVOLUTION, for
every kernel and not only for the D4-symmetric defaults: stencil9 against the FFT restatement, both NumPy conv modes
against each other over whole trajectories, and the reference itself where it is installed. Kernel sets and constant
draws: tests/kernel_sets.py."""
import numpy as np
import pytest

from kernel_sets import DRAWS, KERNEL_SETS, apply_draw, set_kernels
from oracle.daisy_numpy import OracleDaisyWorld, OracleGreedy, fft_circular, stencil9


@pytest.mark.parametrize("role", ["daisy", "adjacent"])
@pytest.mark.parametrize("N", [5, 7, 8, 9, 16, 17, 64])
@pytest.mark.parametrize("name", list(KERNEL_SETS))
def test_stencil9_equals_fft_circular(name, N, role):
    w = KERNEL_SETS[name][0 if role == "daisy" else 1]
    x = np.random.RandomState(N).rand(3, N, N)
    np.testing.assert_allclose(stencil9(x, w), fft_circular(x, w), rtol=0, atol=1e-14)


def test_asymmetric_kernel_is_not_a_correlation():
    """A kernel turned 180 degrees gives a different field: the orientation is really pinned by the test above."""
    x = np.random.RandomState(0).rand(2, 9, 9)
    for name in ("daisy_asym", "adj_asym", "adj_centre"):
        w = KERNEL_SETS[name][0 if name == "daisy_asym" else 1]
        assert np.abs(stencil9(x, w) - stencil9(x, w[::-1, ::-1])).max() > 1e-3


def _oracle(N, B, n, kernels, draw=None, conv="stencil", seed=0):
    np.random.seed(seed)
    env = OracleDaisyWorld(conv=conv, grid_dimension=N, n_agents=n)
    env.batch_size = B
    if draw is not None:
        apply_draw(env, draw)
    set_kernels(env, kernels)
    env.reset()
    return env


def _greedy_run(env, steps, seed=1):
    np.random.seed(seed)
    agent = OracleGreedy()
    obs = env.get_obs(env.agent_indices)
    for _ in range(steps):
        obs, _, _, _ = env.step(agent(obs))
    return env


@pytest.mark.parametrize("name", list(KERNEL_SETS))
def test_stencil_and_fft_oracles_agree(name):
    a = _greedy_run(_oracle(16, 3, 4, name, conv="stencil"), 60)
    b = _greedy_run(_oracle(16, 3, 4, name, conv="fft"), 60)
    np.testing.assert_array_equal(a.grid[:, 0:3], b.grid[:, 0:3])
    np.testing.assert_array_equal(a.agent_indices, b.agent_indices)
    np.testing.assert_array_equal(a.agent_states, b.agent_states)
    np.testing.assert_allclose(a.grid[:, 3:6], b.grid[:, 3:6], rtol=1e-12, atol=0)


def test_adjacent_albedo_kernel_attribute_is_read():
    """The NumPy oracle reads the reference's attribute name, in the reference's (1, 1, 3, 3) shape too."""
    base = _greedy_run(_oracle(9, 2, 2, "default"), 5)
    assert not hasattr(base, "adjacent_kernel")
    other = _oracle(9, 2, 2, "default")
    other.adjacent_albedo_kernel = KERNEL_SETS["adj_asym"][1].reshape(1, 1, 3, 3).copy()
    _greedy_run(other, 5)
    assert not np.array_equal(base.grid[:, 3], other.grid[:, 3])
    flat = _oracle(9, 2, 2, "default")
    flat.adjacent_albedo_kernel = KERNEL_SETS["adj_asym"][1].copy()
    _greedy_run(flat, 5)
    np.testing.assert_array_equal(flat.grid, other.grid)


def test_constant_draws_cover_the_issue_ranges():
    """The draws leave the fast path where they should: one has g = 0, some run without microclimate, some ramp."""
    assert DRAWS[-1]["g"] == 0.0 and all(d["g"] > 0 for d in DRAWS[:-1])
    assert any(not d["use_microclimate"] for d in DRAWS) and any(d.get("ramp_up_down") for d in DRAWS)
    assert all(0.8 <= d["p"] <= 1.0 for d in DRAWS)


# ---- the unmodified reference, when it is installed (baseline/install_ref.py) or checked out at oracle/_ref -------------
def _reference():
    from ref_harness import find_ref
    d = find_ref()
    if d is None:
        pytest.skip("the unmodified reference is not installed")
    return d


@pytest.mark.parametrize("N", [5, 8, 17])
@pytest.mark.parametrize("name", ["daisy_asym", "adj_asym"])
def test_reference_ft_convolve_equals_stencil9(name, N):
    import importlib.util
    import os
    d = _reference()
    spec = importlib.util.spec_from_file_location("ref_functional", os.path.join(d, "daisy", "nn", "functional.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    w = KERNEL_SETS[name][0 if name == "daisy_asym" else 1]
    x = np.random.RandomState(N).rand(2, 1, N, N)
    got = mod.ft_convolve(x, w.reshape(1, 1, 3, 3))
    np.testing.assert_allclose(np.asarray(got).reshape(2, N, N), stencil9(x[:, 0], w), rtol=0, atol=1e-14)


@pytest.mark.parametrize("name", ["daisy_asym", "adj_asym"])
def test_reference_env_matches_numpy_oracle_with_asymmetric_kernels(name):
    from ref_harness import import_reference
    _reference()
    gen = import_reference()
    ref = next(gen)
    try:
        np.random.seed(5)
        env = ref["ref_class"](grid_dimension=16, n_agents=4)
        env.batch_size = 3
        set_kernels(env, name)
        env.reset()
        o = _oracle(16, 3, 4, name)
        o.grid, o.agent_indices, o.agent_states = env.grid.copy(), env.agent_indices.copy(), env.agent_states.copy()
        rng = np.random.RandomState(2)
        for _ in range(30):
            a = rng.randint(9, size=(3, 4, 1))
            env.step(a)
            o.step(a)
            np.testing.assert_array_equal(env.grid[:, 1:3], o.grid[:, 1:3])
    finally:
        next(gen, None)          # restores the reference's module state
