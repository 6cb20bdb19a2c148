"""Diagnostics and plot feed of the giant world (dwt_get_diag / dwt_get_diag_stats / dwt_get_cover_stats / dwt_pool and
BandedDaisyWorld.local_diag / diag_stats / cover_stats / image): the unrounded fields bit for bit against the ensemble
path (RLDaisyWorld, batch 1) on the same state, statistics and block-averaged images against NumPy, bands of one GPU
(NCCL-style and peer-memory mode) against one band, repeatability, the peer-memory fence, and the refusals."""
import ctypes as C

import numpy as np
import pytest

from band_helpers import full_oracle, make_state
from test_banded_diag_gloo import DIAG, GRID, block_means
from test_banded_obs_gloo import oracle_env, state
from test_gpu_tiled_obs import _bands, _run_bands, _world

pytestmark = pytest.mark.gpu


def _ensemble(N, n, light, dark, ai, st):
    """RLDaisyWorld with one world holding the same reset state."""
    from therldaisyworld_b200 import RLDaisyWorld
    env = RLDaisyWorld(grid_dimension=N, n_agents=n)
    env.batch_size = 1
    env.reset()
    grid = np.zeros((1, 7, N, N))
    grid[0, 1], grid[0, 2] = light, dark
    env.grid = grid
    env.agent_indices = ai[None].copy()
    env.agent_states = st[None, :, None].copy()
    return env


def _numpy_temp(world, light, dark, ai, st, steps):
    """env.temp of the NumPy oracle after `steps` greedy steps from the reset state."""
    from oracle.daisy_numpy import OracleGreedy
    env = oracle_env(world, light, dark, ai, st)
    greedy = OracleGreedy(greedy=True)
    obs = env.get_obs(env.agent_indices)
    for _ in range(steps):
        obs = env.step(greedy(obs))[0]
    return env.temp[0, 0]


def _fields(w):
    f = {k: w.local_diag(k) for k in DIAG}
    g = w.local_grid()
    f.update({k: g[ch] for k, ch in GRID.items()})
    f["growth_l"], f["growth_d"] = f["growth"]
    return f


def _check_stats_and_images(w, f, N):
    for k in DIAG:
        s, v = w.diag_stats(k), f[k]
        np.testing.assert_allclose(s["mean"], v.mean(), rtol=1e-12)
        np.testing.assert_allclose(s["std"], v.std(), rtol=1e-9)
        assert s["min"] == v.min() and s["max"] == v.max()
    c, cov = w.cover_stats(), w.local_covers()
    np.testing.assert_allclose([c["mean_light"], c["mean_dark"]], [cov[0].mean(), cov[1].mean()], rtol=1e-12)
    assert c["max_light"] == cov[0].max() and c["max_dark"] == cov[1].max()
    for k in ("temp", "beta_d", "growth", *GRID):
        for b in (1, 7, 16, 64, N):
            img = w.image(k, b)
            if b == 1:
                np.testing.assert_array_equal(img, f[k])
            else:
                np.testing.assert_allclose(img, block_means(f[k], b), rtol=1e-12, atol=1e-300)


@pytest.mark.parametrize("N", [64, 130, 333])
def test_single_band_fields_stats_images(N):
    """After step 1 (pre-state: the fp64 planes of the reset) and after step 12 (the lattice)."""
    n = 300
    light, dark, ai, st = make_state(N, n, seed=N, clustered=True)
    w = _world(N, n)
    w.load_state(light, dark, ai, st)
    env = _ensemble(N, n, light, dark, ai, st)
    done = 0
    for steps in (1, 12):
        w.run(steps - done, "greedy")
        env.run(steps - done, policy="greedy")
        done = steps
        f = _fields(w)
        for k in DIAG:
            exp = env._diag(k)[0]
            np.testing.assert_array_equal(f[k], exp if k == "growth" else exp[0], err_msg=k)
        np.testing.assert_allclose(f["temp"], _numpy_temp(w, light, dark, ai, st, steps), rtol=1e-12)
        _check_stats_and_images(w, f, N)
        assert w.dead_temp[0] == env.dead_temp[0]


def _everything(w, N):
    out = {"stats": [w.diag_stats(k) for k in DIAG], "cover": w.cover_stats(),
           "images": [w.image(k, b) for k in ("temp", "growth", "grid_light", "grid_temp") for b in (1, 16, 64, 128, N)]}
    return out


@pytest.mark.parametrize("mode", ["nccl", "p2p"])
@pytest.mark.parametrize("bands", [3, 4])
def test_bands_agree_with_one_band(mode, bands):
    """N = 200: bands of 66/67/67 or 50 rows, so 64- and 128-blocks span several bands. Every rank returns the same bits,
    twice; the one-band world agrees exactly on min, max and cover maxima, to 1e-12 otherwise."""
    N, n, steps = 200, 120, 9
    light, dark, ai, st = state(N, bands, n=n)
    one = _world(N, n)
    one.load_state(light, dark, ai, st)
    one.run(steps, "greedy")
    ref = _everything(one, N)
    ref_local = one.local_diag("temp")
    worlds, streams = _bands(N, n, bands, mode)

    def fn(w):
        w.load_state(light, dark, ai, st)
        for _ in range(steps):
            w.step("greedy")
        return _everything(w, N), _everything(w, N), w.local_diag("temp")

    res = _run_bands(worlds, streams, fn)
    for a, b, _ in res:
        for x, y in ((a, b), (a, res[0][0])):
            for s, t in zip(x["stats"], y["stats"]):
                assert s == t
            assert x["cover"] == y["cover"]
            for p, q in zip(x["images"], y["images"]):
                np.testing.assert_array_equal(p, q)
        for s, t in zip(a["stats"], ref["stats"]):
            assert s["min"] == t["min"] and s["max"] == t["max"]
            np.testing.assert_allclose([s["mean"], s["std"]], [t["mean"], t["std"]], rtol=1e-12)
        assert (a["cover"]["max_light"], a["cover"]["max_dark"]) == (ref["cover"]["max_light"], ref["cover"]["max_dark"])
        np.testing.assert_allclose([a["cover"]["mean_light"], a["cover"]["mean_dark"]],
                                   [ref["cover"]["mean_light"], ref["cover"]["mean_dark"]], rtol=1e-12)
        for k, (p, q) in enumerate(zip(a["images"], ref["images"])):
            if k % 5 == 0:                                      # block 1: single cells
                np.testing.assert_array_equal(p, q)
            else:
                np.testing.assert_allclose(p, q, rtol=1e-12, atol=1e-300)
    np.testing.assert_array_equal(np.concatenate([r[2] for r in res]), ref_local)


def test_peer_memory_diagnostics_between_steps():
    """Statistics, images and local fields read the pre-state that the next step's halo push overwrites: with them between
    every two steps the world must still equal the C oracle and no barrier may time out."""
    N, n, bands, steps = 200, 150, 3, 8
    light, dark, ai, st = state(N, bands, n=n)
    worlds, streams = _bands(N, n, bands, "p2p")
    ref = full_oracle(worlds[0], light, dark, ai, st)     # the reset clock, before the world runs

    def fn(w):
        w.load_state(light, dark, ai, st)
        temps = []
        for _ in range(steps):
            w.step("greedy")
            temps.append((w.diag_stats("temp")["mean"], w.image("temp", 16), w.local_diag("beta")))
        return temps, w.local_covers(), w.agents(), w.lifespans()

    res = _run_bands(worlds, streams, fn)
    _, done_at, ada = ref.run(steps, "greedy")
    covers = np.concatenate([r[1] for r in res], axis=1)
    np.testing.assert_array_equal(covers[0], ref.grid[0, 1])
    np.testing.assert_array_equal(covers[1], ref.grid[0, 2])
    for _, _, (xy, s), (d, a) in res:
        np.testing.assert_array_equal(xy, ref.agent_indices[0])
        np.testing.assert_array_equal(s, ref.agent_states[0, :, 0])
        assert d == np.asarray(done_at).ravel()[0]
        np.testing.assert_array_equal(a, np.asarray(ada).reshape(-1))
    for r in res[1:]:
        for (m0, i0, _), (m1, i1, _) in zip(res[0][0], r[0]):
            assert m0 == m1
            np.testing.assert_array_equal(i0, i1)


def test_refusals():
    from therldaisyworld_b200 import DaisyWorldError
    N, n = 64, 10
    light, dark, ai, st = make_state(N, n, seed=3)
    w = _world(N, n)
    w.load_state(light, dark, ai, st)
    for call in (lambda: w.diag_stats("temp"), lambda: w.image("temp", 16), lambda: w.local_diag("temp")):
        with pytest.raises(DaisyWorldError, match="needs a step"):
            call()
    c = w.cover_stats()                                  # the current state: the reset planes
    assert c["mean_light"] == pytest.approx(light.mean(), rel=1e-12) and c["max_dark"] == dark.max()
    w.step("greedy")
    w.band.time_stencil(2)
    with pytest.raises(DaisyWorldError, match="dwt_get_diag_stats.*needs a step"):
        w.diag_stats("temp")
    with pytest.raises(DaisyWorldError, match="dwt_pool.*needs a step"):
        w.image("temp", 16)
    w.step("greedy")
    assert np.isfinite(w.diag_stats("temp")["std"])
    with pytest.raises(ValueError):
        w.diag_stats("nope")
    b = w.band
    out = np.zeros((2, N, N))
    pd = out.ctypes.data_as(C.POINTER(C.c_double))
    assert b._lib.dwt_get_diag(b._h, 8, pd) == -1 and b._lib.dwt_get_diag(b._h, -1, pd) == -1
    assert b._lib.dwt_get_diag_stats(b._h, 8, pd) == -1
    assert b._lib.dwt_pool(b._h, 14, 16) == -1 and b._lib.dwt_pool(b._h, -1, 16) == -1
    for block in (0, -3, N + 1):
        with pytest.raises(DaisyWorldError, match="dwt_pool.*block"):
            w.image("temp", block)
    assert w.image("temp", N).shape == (1, 1)
    b.move_graze()                                       # a step's agents not finished
    with pytest.raises(DaisyWorldError, match="not finished"):
        b.diag_stats("temp")
    with pytest.raises(DaisyWorldError, match="not finished"):
        b.cover_stats()
    b.finish_agents()
