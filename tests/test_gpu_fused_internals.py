"""Internals of the fused lattice path: accuracy of the fast fourth root (the only approximation in the fast
path), the tie filter's literal fallback rate, and fused == materialising path on the same inputs."""
import ctypes as C
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def _env(N=8, B=2, n=2, seed=0):
    from therldaisyworld_b200 import RLDaisyWorld
    np.random.seed(seed)
    env = RLDaisyWorld(grid_dimension=N, n_agents=n)
    env.batch_size = B
    env.reset()
    return env


def test_fast_root4_relative_error_bound():
    """dw_root4_fast must stay far inside the error budget of the tie filter: the filter half-width is
    derived from a 3e-12 bound on this error (csrc/dw_run.inl::make_fast_coef, DESIGN.md section 2); measured 2.2e-12."""
    env = _env()
    rng = np.random.RandomState(0)
    # the kernels take the root of X' = g^2 * T^4 (g = 0.003265: 1e4..2e5; other g shift the range), the literal T^4 is ~1e10
    x = np.concatenate([10.0 ** rng.uniform(2, 11.5, size=600000), np.linspace(3e9, 2e10, 100000), np.linspace(1e4, 3e5, 100000)])
    y = np.empty_like(x)
    rc = env._lib.dw_debug_root4(env._h, x.ctypes.data_as(C.POINTER(C.c_double)), y.ctypes.data_as(C.POINTER(C.c_double)), x.size)
    assert rc == 0
    ref = np.sqrt(np.sqrt(x))
    rel = np.abs(y - ref) / ref
    print("max rel err of dw_root4_fast:", rel.max())
    assert rel.max() < 3e-12          # the bound make_fast_coef derives the tie-filter width from


@pytest.mark.parametrize("N,B,n,policy", [(64, 16, 4, "greedy"), (16, 8, 4, "antigreedy"), (33, 4, 7, "random"),
                                          (5, 3, 2, "greedy"), (2, 2, 1, "greedy"), (1, 2, 1, "none"), (12, 4, 0, "none"),
                                          (40, 2, 40, "greedy"),
                                          # worlds below 64x64 share a CTA (k_fused_sub64_persist): partial last group,
                                          # agent count at the shared-memory limit (64 worlds x 4), and over it (generic kernel)
                                          (8, 70, 4, "greedy"), (8, 130, 3, "random"), (16, 19, 9, "antigreedy"),
                                          (32, 7, 33, "greedy"), (32, 9, 0, "none"), (8, 5, 5, "greedy"),
                                          # other multiples of 4 run the 4x4-tile kernel with a host-chosen block size (k_fused_tile4)
                                          (20, 9, 3, "antigreedy"), (96, 3, 5, "greedy"), (128, 2, 6, "random"), (156, 1, 4, "greedy"),
                                          (32, 3, 70, "greedy"),
                                          # sides that are not a multiple of 4: the same kernel with padded rows and masked edge tiles
                                          # (1, 2 and 3 columns in the last tile); 157 still fits with its rows padded to 160 words
                                          (13, 6, 3, "greedy"), (18, 5, 4, "random"), (61, 3, 5, "greedy"), (150, 1, 4, "antigreedy"),
                                          (157, 1, 2, "greedy")])
def test_fused_equals_materialising_path(N, B, n, policy):
    """Same inputs through dw_run with the fused kernel and with DW_DISABLE_FUSED=1 DW_LITERAL_ONLY=1 (materialising
    kernels in literal arithmetic only: the ground truth)."""
    res = []
    for disable in (False, True):
        if disable:
            os.environ["DW_DISABLE_FUSED"] = "1"
            os.environ["DW_LITERAL_ONLY"] = "1"
        else:
            os.environ.pop("DW_DISABLE_FUSED", None)
        try:
            env = _env(N, B, n, seed=N)
            env.reset_lifespans()
            env.run(150, policy=policy, seed=5)
            mid = env.grid.copy()
            env.run(400, policy=policy, seed=5)
            count = C.c_uint64()
            assert env._lib.dw_debug_slow_count(env._h, C.byref(count), 0) == 0
            res.append((mid, env.grid.copy(), env.agent_indices.copy(), env.agent_states.copy(), env.lifespans(),
                        env.L, env.step_count, env.temp.copy(), count.value))
        finally:
            os.environ.pop("DW_DISABLE_FUSED", None)
            os.environ.pop("DW_LITERAL_ONLY", None)
    a, b = res
    for u, v in zip(a[:4], b[:4]):
        np.testing.assert_array_equal(u, v)
    np.testing.assert_array_equal(a[4][0], b[4][0])
    np.testing.assert_array_equal(a[4][1], b[4][1])
    assert a[5:7] == b[5:7]
    np.testing.assert_array_equal(a[7], b[7])
    assert b[8] == 0                      # materialising path never uses the literal fallback counter
    cells = 549 * B * N * N
    print(f"literal recomputations: {a[8]} of {cells} cell-updates ({a[8] / cells:.2e})")
    assert a[8] < 1e-3 * cells + 10


def test_division_free_rounding_is_exact_on_device():
    env = _env()
    bad = C.c_uint32(123)
    assert env._lib.dw_debug_markstein(env._h, 2000000, C.byref(bad)) == 0
    assert bad.value == 0
    # binary32 twin of the fp32 mode: every integer the fp32 grid divides by 1000 (covers <= 1000, 1000 T <= 4e5 < 2^19)
    bad = C.c_uint32(123)
    assert env._lib.dw_debug_markstein_f32(env._h, 1 << 19, C.byref(bad)) == 0
    assert bad.value == 0


def test_eps_greedy_limits_and_kernel_consistency():
    """DW_POLICY_EPS_GREEDY: epsilon 0 is the greedy policy, epsilon 1 the random one (same counter RNG), and for
    0 < epsilon < 1 the fused kernel and the materialising kernels agree step for step (one coin per step, resolved on
    the host from (seed, step_count))."""
    def run(policy, eps, disable=False, N=64, B=6):
        if disable:
            os.environ["DW_DISABLE_FUSED"] = "1"
        try:
            env = _env(N, B, 4, seed=21)
            env.set_epsilon(eps)
            env.reset_lifespans()
            env.run(120, policy=policy, seed=9)
            return env.grid.copy(), env.agent_states.copy(), env.agent_indices.copy(), env.lifespans()[1].copy()
        finally:
            os.environ.pop("DW_DISABLE_FUSED", None)

    for a, b in ((run("eps_greedy", 0.0), run("greedy", 0.0)), (run("eps_greedy", 1.0), run("random", 0.0)),
                 (run("eps_greedy", 0.5), run("eps_greedy", 0.5, disable=True))):
        for u, v in zip(a, b):
            np.testing.assert_array_equal(u, v)
    half, greedy, rnd = run("eps_greedy", 0.5), run("greedy", 0.0), run("random", 0.0)
    assert not np.array_equal(half[2], greedy[2]) and not np.array_equal(half[2], rnd[2])


def test_fast_path_fuzz_random_physics():
    """Random albedos, solar constant, growth/death constants, time step, ramps and sizes: the fused kernels must stay
    identical to the literal materialising kernels (tools/fuzz_fast_path.py runs the same check over hundreds of draws)."""
    import importlib.util
    spec = importlib.util.spec_from_file_location("fuzz", os.path.join(os.path.dirname(os.path.dirname(__file__)), "tools", "fuzz_fast_path.py"))
    fuzz = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(fuzz)
    rng = np.random.RandomState(123)
    for c in range(12):
        attrs, N, n, ramp, no_micro = fuzz.draw(rng)
        ok, slow, diff, life = fuzz.run_config(attrs, N, n, ramp, no_micro, seed=1000 + c, B=8, steps=250)
        assert ok, (c, attrs, N, n, ramp, no_micro, diff)


def test_screened_forward_equals_literal_forward():
    """The materialising kernels evaluate every cell with the fast fourth root and FMAs and keep the result only where no
    rounded channel sits within the error bound of a rounding tie (dw_screened_cell); DW_LITERAL_ONLY=1 forces the literal
    evaluation everywhere. Both must give the same seven channels on random off-lattice states, on lattice states, with
    random physics, and on inputs outside the range the bound assumes (covers beyond [0, 1], dead-hot planets, NaN)."""
    import importlib.util
    from therldaisyworld_b200 import RLDaisyWorld
    spec = importlib.util.spec_from_file_location("fuzz", os.path.join(os.path.dirname(os.path.dirname(__file__)), "tools", "fuzz_fast_path.py"))
    fuzz = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(fuzz)
    rng = np.random.RandomState(2024)
    cells = 0
    for case in range(24):
        N, B = int(rng.choice([5, 16, 33, 64])), 6
        np.random.seed(case)
        env = RLDaisyWorld(grid_dimension=N, n_agents=2)
        env.batch_size = B
        if case % 3:
            attrs, _, _, _, no_micro = fuzz.draw(rng)
            for k, v in attrs.items():
                setattr(env, k, v)
            env.q = 0.2 * env.S / env.sigma
            env.set_use_microclimate(not no_micro)
        env.reset()
        env.L = float(rng.uniform(env.min_L, env.max_L))
        g = env.grid.copy()
        mode = case % 4
        if mode == 0:      # arbitrary off-lattice covers
            g[:, 1], g[:, 2] = rng.rand(B, N, N) * 0.7, rng.rand(B, N, N) * 0.3
        elif mode == 1:    # lattice covers, sparse
            g[:, 1] = np.round(rng.rand(B, N, N) * (rng.rand(B, N, N) < 0.4), 3)
            g[:, 2] = np.round(rng.rand(B, N, N) * 0.5 * (rng.rand(B, N, N) < 0.4), 3)
        elif mode == 2:    # out-of-range inputs: covers beyond [0, 1], negative, one NaN
            g[:, 1], g[:, 2] = rng.randn(B, N, N), rng.rand(B, N, N) * 3
            g[0, 1, 0, 0] = np.nan
        else:              # a reset state as is
            pass
        outs = []
        for literal in (False, True):
            if literal:
                os.environ["DW_LITERAL_ONLY"] = "1"
            try:
                outs.append(env.forward(g.copy()))
            finally:
                os.environ.pop("DW_LITERAL_ONLY", None)
        np.testing.assert_array_equal(outs[0], outs[1])
        cells += B * N * N
    assert cells > 100000


def test_screened_evaluation_stays_inside_its_tie_filters():
    """The error budget of dw_screened_cell, measured: over random off-lattice and lattice states, default and random
    physics, the largest |screened - literal| of every unrounded channel (units of 0.001) must stay at least 3x below the
    tie-filter half-width derived on the host (make_params_cfg) -- the margin the exactness argument relies on."""
    import importlib.util
    from therldaisyworld_b200 import RLDaisyWorld
    spec = importlib.util.spec_from_file_location("fuzz", os.path.join(os.path.dirname(os.path.dirname(__file__)), "tools", "fuzz_fast_path.py"))
    fuzz = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(fuzz)
    rng = np.random.RandomState(77)
    worst = np.zeros(3)
    for case in range(30):
        N, B = 64, 16
        np.random.seed(case)
        env = RLDaisyWorld(grid_dimension=N, n_agents=0)
        env.batch_size = B
        if case % 2:
            attrs, _, _, _, no_micro = fuzz.draw(rng)
            for k, v in attrs.items():
                setattr(env, k, v)
            env.q = 0.2 * env.S / env.sigma
            env.set_use_microclimate(not no_micro)
        env.reset()
        env.L = float(rng.uniform(env.min_L, env.max_L))
        g = env.grid.copy()
        if case % 3 == 0:
            g[:, 1], g[:, 2] = rng.rand(B, N, N) * 0.7, rng.rand(B, N, N) * 0.3
        elif case % 3 == 1:
            g[:, 1] = np.round(rng.rand(B, N, N) * (rng.rand(B, N, N) < 0.5), 3)
            g[:, 2] = np.round(rng.rand(B, N, N) * (1 - g[:, 1]) * (rng.rand(B, N, N) < 0.5), 3)
        env._push()
        out = np.zeros(6)
        rc = env._lib.dw_debug_screen_error(env._h, np.ascontiguousarray(g).ctypes.data_as(C.POINTER(C.c_double)),
                                            out.ctypes.data_as(C.POINTER(C.c_double)))
        assert rc == 0
        assert (out[:3] * 3.0 < out[3:]).all(), (case, out)
        worst = np.maximum(worst, out[:3] / out[3:])
    print("largest measured error / filter half-width (covers, bare, temperatures):", worst)
