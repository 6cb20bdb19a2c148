"""Which fused kernel runs a shape (fused_kernel in csrc/dw_run.inl, DESIGN.md section 4), seen through the public
surface at each capability edge: the trimmed lifespan runs (alive_mask), the in-kernel series mode and the in-kernel MLP
policy. The fused families compute bit-identical results, so the result tests cannot see a shape that moves to another
family; these checks pin one case on each side of every boundary."""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def _env(N, n, B=4):
    """A short greedy run first: trim and the in-kernel MLP policy need a lattice-resident state."""
    from therldaisyworld_b200 import RLDaisyWorld
    np.random.seed(N * 1000 + n)
    env = RLDaisyWorld(grid_dimension=N, n_agents=n)
    env.batch_size = B
    env.reset()
    env.run(3, policy="greedy")
    return env


@pytest.mark.parametrize("N,n,yes", [(64, 32, 1), (64, 33, 0),      # k_fused_n64_persist / k_fused_n64
                                     (16, 16, 1), (16, 17, 0),      # k_fused_sub64_persist<16> / k_fused_tile4
                                     (8, 4, 1), (8, 5, 0)])         # k_fused_sub64_persist<8> / k_fused_generic
def test_trim_supported_edges(N, n, yes):
    from therldaisyworld_b200._lib import DW_POLICY
    env = _env(N, n)
    got = C.c_int32(-1)
    assert env._lib.dw_trim_supported(env._h, DW_POLICY["greedy"], C.byref(got)) == 0
    assert got.value == yes


@pytest.mark.parametrize("N,n,in_kernel", [(64, 32, True), (64, 33, False),
                                           (16, 16, True), (16, 17, False),
                                           (12, 2, False), (20, 2, True), (21, 2, False),     # k_fused_tile4: from side 20, no padding
                                           (32, 65, True),                                    # k_fused_tile4<false, true>
                                           (11, 2, False), (157, 2, False)])                  # k_fused_generic, k_fused_tile4<true>
def test_run_series_in_kernel_edges(N, n, in_kernel):
    """dw_run_series either records the series in the kernel (returns 0, the clock advances K steps) or refuses with
    DW_E_UNSUPPORTED before any step has run (the clock is unchanged), and RLDaisyWorld.run_series then steps on its own."""
    from therldaisyworld_b200._lib import DW_E_UNSUPPORTED, DW_POLICY, DwClock
    env = _env(N, n, B=1 if N > 64 else 4)
    env._push()
    before, after = DwClock(), DwClock()
    assert env._lib.dw_get_clock(env._h, C.byref(before)) == 0
    K = 5
    out = np.zeros((K, 3))
    rc = env._lib.dw_run_series(env._h, K, DW_POLICY["greedy"], None, C.c_uint64(0), out.ctypes.data_as(C.POINTER(C.c_double)))
    assert env._lib.dw_get_clock(env._h, C.byref(after)) == 0
    if in_kernel:
        assert rc == 0
        assert after.step_count == before.step_count + K
        assert (out[:, 0] > 0).all()
    else:
        assert rc == DW_E_UNSUPPORTED
        assert bytes(after) == bytes(before)


@pytest.mark.parametrize("n", [32, 33])
def test_in_kernel_mlp_edge(n):
    """64x64 worlds with at most 32 agents run K MLP steps in one launch of the persistent kernel; with more agents each step
    has its own policy launch and its own step launch (the coefficient-table copy is not a kernel launch)."""
    from therldaisyworld_b200._lib import DwProfile
    env = _env(64, n)
    env.set_mlp(np.random.RandomState(0).randn(1808))
    K = 6
    lib, h = env._lib, env._h
    assert lib.dw_set_profiling(h, 1) == 0
    env.run(K, policy="mlp")
    prof = DwProfile()
    assert lib.dw_get_profile(h, C.byref(prof)) == 0
    assert lib.dw_set_profiling(h, 0) == 0
    if n <= 32:
        assert prof.kernel_launches == 1
    else:
        assert prof.kernel_launches >= 2 * K
