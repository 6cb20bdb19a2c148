"""fp32 mode of the giant world (dwt_grid_f32, k_band_forward_f32; BandedDaisyWorld.local_grid_f32 / local_grid_f32_tensor /
f32_stats): bit for bit against the ensemble's fp32 mode (RLDaisyWorld.grid_f32, batch 1) on the same state, against the
exact fp64 grid (covers, bare fraction, stamp exact as binary32; temperatures within 1e-5 relative), after the first step
of a reset, on bands of one GPU (NCCL-style and peer-memory mode), under random physics and a heat step, after snapshots,
as a device tensor, and the refusals."""
import os
import sys

import numpy as np
import pytest

from band_helpers import make_state
from test_banded_obs_gloo import golden_mlp_params, state
from test_gpu_tiled_obs import _bands, _run_bands, _world

pytestmark = pytest.mark.gpu


def _ensemble(N, n, light, dark, ai, st, **attrs):
    """RLDaisyWorld with one world holding the same reset state (and constants)."""
    from therldaisyworld_b200 import RLDaisyWorld
    env = RLDaisyWorld(grid_dimension=N, n_agents=n)
    env.batch_size = 1
    for k, v in attrs.items():
        setattr(env, k, v)
    env.reset()
    grid = np.zeros((1, 7, N, N))
    grid[0, 1], grid[0, 2] = light, dark
    env.grid = grid
    env.agent_indices = ai[None].copy()
    env.agent_states = st[None, :, None].copy()
    return env


def _delta(a, b):
    return {k: b[k] - a[k] for k in a}


def _check_against_f64(w, g32=None):
    """local_grid_f32() against local_grid() of the same state; returns the grid and the counters' delta of the call."""
    before = w.f32_stats()
    if g32 is None:
        g32 = w.local_grid_f32()
    d = _delta(before, w.f32_stats())
    g64 = w.local_grid()
    assert g32.dtype == np.float32 and g32.shape == g64.shape
    for ch in (0, 1, 2, 6):
        np.testing.assert_array_equal(g32[ch], g64[ch].astype(np.float32), err_msg=f"channel {ch}")
    ai, _ = w.agents()
    stamp = np.zeros(g64[4].shape, dtype=bool)
    rows = (ai[:, 0] - w.row0) % w.dim
    own = rows < w.rows
    stamp[rows[own], ai[own, 1]] = True
    np.testing.assert_array_equal(g32[4][stamp], g64[4][stamp].astype(np.float32))
    for ch in (3, 4, 5):
        m = ~stamp if ch == 4 else np.ones_like(stamp)
        rel = np.abs(g32[ch][m].astype(np.float64) - g64[ch][m]) / np.abs(g64[ch][m])
        assert rel.max() <= 1e-5, (ch, rel.max())
    return g32, d


@pytest.mark.parametrize("N", [64, 97, 130])
def test_bit_equal_to_the_ensemble_fp32_mode(N):
    """97 is odd: one cell per thread (W = 1). Agents clustered around (0, 0): the stamp wraps and cells hold several."""
    n, steps = 300, 12
    light, dark, ai, st = make_state(N, n, seed=N, clustered=True)
    w = _world(N, n)
    w.load_state(light, dark, ai, st)
    env = _ensemble(N, n, light, dark, ai, st)
    w.run(steps, "greedy")
    env.run(steps, policy="greedy")
    assert env.residency()["lattice"]
    wb, eb = w.f32_stats(), env.f32_stats()
    got, exp = w.local_grid_f32(), env.grid_f32()[0]
    np.testing.assert_array_equal(got.view(np.uint32), exp.view(np.uint32))
    assert _delta(wb, w.f32_stats()) == _delta(eb, env.f32_stats())
    assert _delta(wb, w.f32_stats())["cells"] == N * N


@pytest.mark.parametrize("N", [256, 333])
@pytest.mark.parametrize("policy", ["greedy", "replay", "mlp"])
def test_single_band_against_the_fp64_grid(N, policy):
    n, steps = 400, 10
    light, dark, ai, st = make_state(N, n, seed=N + 7, clustered=True)
    w = _world(N, n)
    if policy == "mlp":
        w.set_mlp(golden_mlp_params())
    w.load_state(light, dark, ai, st)
    acts = np.random.RandomState(5).randint(9, size=(2 * steps, n))
    w.run(steps, policy, actions=acts[:steps] if policy == "replay" else None)
    for k in range(2):
        _, d = _check_against_f64(w)
        assert d["cells"] == N * N
        assert d["fp64_tier"] <= 0.2 * d["cells"], d
        assert d["literal"] <= d["fp64_tier"]
        w.run(steps, policy, actions=acts[steps:] if policy == "replay" else None)


def test_first_step_after_a_reset_converts_the_fp64_grid():
    """The pre-state of the first step is the fp64 planes of the reset: the whole grid is local_grid() as float32, and no
    cell counts as evaluated with fp32 arithmetic."""
    N, n = 130, 200
    light, dark, ai, st = make_state(N, n, seed=3, clustered=True)
    w = _world(N, n)
    w.load_state(light, dark, ai, st)
    w.step("greedy")
    before = w.f32_stats()
    g32 = w.local_grid_f32()
    assert w.f32_stats() == before
    np.testing.assert_array_equal(g32, w.local_grid().astype(np.float32))
    w.step("greedy")                                     # the lattice from here on
    _, d = _check_against_f64(w)
    assert d["cells"] == N * N


@pytest.mark.parametrize("mode", ["nccl", "p2p"])
@pytest.mark.parametrize("N,bands", [(200, 3), (333, 4)])
def test_bands_equal_one_band(mode, N, bands):
    """Bands of 66/67/67 or 83/83/83/84 rows, a second agent cluster on the first band boundary. The steps after the call
    still equal the single band's: the peer-memory fence held."""
    n, steps, more = 300, 9, 4
    light, dark, ai, st = state(N, bands, n=n)
    one = _world(N, n)
    one.load_state(light, dark, ai, st)
    one.run(steps, "greedy")
    s0 = one.f32_stats()
    ref = one.local_grid_f32()
    ref_stats = _delta(s0, one.f32_stats())
    one.run(more, "greedy")
    ref_covers = one.local_covers()
    worlds, streams = _bands(N, n, bands, mode)

    def fn(w):
        w.load_state(light, dark, ai, st)
        for _ in range(steps):
            w.step("greedy")
        s = w.f32_stats()
        g = w.local_grid_f32()
        d = _delta(s, w.f32_stats())
        for _ in range(more):
            w.step("greedy")
        return g, d, w.local_covers()

    res = _run_bands(worlds, streams, fn)
    np.testing.assert_array_equal(np.concatenate([r[0] for r in res], axis=1).view(np.uint32), ref.view(np.uint32))
    for r in res:
        assert r[1] == ref_stats                         # summed over the ranks
    np.testing.assert_array_equal(np.concatenate([r[2] for r in res], axis=1), ref_covers)


def test_random_physics_and_a_heat_step():
    """Eight draws of random constants (tools/fuzz_fast_path.draw) and the heat_step scenario of tests/kernel_sets.py,
    whose first lattice step runs at max_L = 2.5: the screen keeps channels 0..2 exact."""
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools"))
    from fuzz_fast_path import draw
    from kernel_sets import SCENARIOS
    rng = np.random.RandomState(41)
    cases = []
    for _ in range(8):
        attrs, N, n, ramp, no_micro = draw(rng, sizes=(64, 96, 130))
        cases.append((dict(ramp_period=ramp), attrs, N, n, no_micro, int(rng.randint(3, 40))))
    sc = SCENARIOS["heat_step"]
    cases.append((sc["ctor"], sc["attrs"], 96, 40, False, sc["grow"] + sc["settle"]))
    tiers = []
    for ctor, attrs, N, n, no_micro, steps in cases:
        light, dark, ai, st = make_state(N, n, seed=N + steps, clustered=True)
        w = _world(N, n, **ctor)
        for k, v in attrs.items():
            setattr(w, k, v)
        w.q = 0.2 * w.S / w.sigma                        # as the reference's constructor, and its microclimate switch
        w.q2 = 0.0 if no_micro else w.q / 8.0
        w.load_state(light, dark, ai, st)
        w.run(steps, "greedy")
        _, d = _check_against_f64(w)
        assert d["cells"] == N * N
        tiers.append(d["fp64_tier"] / d["cells"])
    assert np.mean(tiers) < 0.25, tiers


def test_snapshots(tmp_path):
    """save / restore into a fresh world and onto 3 bands: the fp32 grid equals the uninterrupted world's."""
    from test_gpu_tiled_snapshot import _release
    N, n, k = 200, 300, 6
    light, dark, ai, st = state(N, 3, n=n)
    w = _world(N, n)
    w.load_state(light, dark, ai, st)
    w.run(k, "greedy")
    w.save(str(tmp_path))
    exp = w.local_grid_f32()
    x = _world(N, n)
    x.restore(str(tmp_path))
    np.testing.assert_array_equal(x.local_grid_f32().view(np.uint32), exp.view(np.uint32))
    _release([])
    worlds, streams = _bands(N, n, 3, "nccl")
    res = _run_bands(worlds, streams, lambda b: (b.restore(str(tmp_path)), b.local_grid_f32())[1])
    np.testing.assert_array_equal(np.concatenate(res, axis=1).view(np.uint32), exp.view(np.uint32))
    _release(worlds)


def test_device_view():
    import torch
    N, n = 130, 100
    light, dark, ai, st = make_state(N, n, seed=9, clustered=True)
    w = _world(N, n)
    w.load_state(light, dark, ai, st)
    w.run(5, "greedy")
    t = w.local_grid_f32_tensor()
    assert t.dtype == torch.float32 and t.device == torch.device(f"cuda:{w.device}")
    assert tuple(t.shape) == (7, N, N) and t.is_contiguous()
    host = w.local_grid_f32()
    np.testing.assert_array_equal(t.cpu().numpy(), host)
    w.run(3, "greedy")
    u = w.local_grid_f32_tensor()
    assert u.data_ptr() == t.data_ptr()                  # the same library buffer, overwritten
    np.testing.assert_array_equal(u.cpu().numpy(), w.local_grid_f32())
    _check_against_f64(w, g32=u.cpu().numpy())


def test_refusals():
    from therldaisyworld_b200 import DaisyWorldError
    N, n = 64, 10
    light, dark, ai, st = make_state(N, n, seed=1)
    w = _world(N, n)
    w.load_state(light, dark, ai, st)
    with pytest.raises(DaisyWorldError, match="dwt_grid_f32.*needs a step"):
        w.local_grid_f32()
    with pytest.raises(DaisyWorldError, match="dwt_grid_f32.*needs a step"):
        w.local_grid_f32_tensor()
    w.step("greedy")
    w.band.time_stencil(2)
    with pytest.raises(DaisyWorldError, match="dwt_grid_f32.*dwt_debug_time_stencil"):
        w.local_grid_f32()
    w.step("greedy")
    w.band.move_graze()                                  # a step's agents not finished
    with pytest.raises(DaisyWorldError, match="dwt_grid_f32.*not finished"):
        w.band.grid_f32()
    w.band.finish_agents()
    w.step("greedy")
    _check_against_f64(w)
    assert w.band.time_materialise(True, 2) > 0 and w.band.time_materialise(False, 2) > 0
    b = w.band
    assert b._lib.dwt_get_grid_f32(b._h, None) == -1 and b._lib.dwt_f32_stats(b._h, None) == -1
    assert b._lib.dwt_get_grid_f32_ptr(b._h, None) == -1
