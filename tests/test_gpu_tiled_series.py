"""Climate series of the single giant world (BandedDaisyWorld.run_series, series mode of the tiled stencil kernels): the
per-step global mean temperature and mean covers against the NumPy oracle, which exposes the unrounded temperature, on one
band and on several bands of one GPU (NCCL-style exchanges and peer-memory mode)."""
import numpy as np
import pytest

from band_helpers import ThreadComm, full_oracle, make_state, run_threads

pytestmark = pytest.mark.gpu


def _world(N, n, **kw):
    from therldaisyworld_b200.banded import BandedDaisyWorld
    return BandedDaisyWorld(N, n, **kw)


def _oracle_series(N, light, dark, ai, st, steps, policy, acts=None):
    """[steps, 3] per-step (mean T, mean light, mean dark) of the NumPy oracle from the given reset state; covers as the
    exact milli-cover sums over 1000 N^2, the way the device series divides them."""
    from oracle.daisy_numpy import OracleDaisyWorld, OracleGreedy
    n = ai.shape[0]
    env = OracleDaisyWorld(grid_dimension=N, n_agents=n)
    env.batch_size = 1
    env.grid = np.zeros((1, 7, N, N))
    env.grid[0, 1], env.grid[0, 2] = light, dark
    env.agent_indices = ai[None].copy()
    env.agent_states = st[None, :, None].copy()
    agent = OracleGreedy(greedy=policy == "greedy")
    obs = env.get_obs(env.agent_indices)
    out = np.zeros((steps, 3))
    cells = float(N * N)
    for t in range(steps):
        if policy in ("greedy", "antigreedy"):
            a = agent(obs)
        elif policy == "replay":
            a = acts[t][None, :, None]
        else:
            a = None                                     # "none": action 0 for every agent
        obs, _, _, _ = env.step(a)
        out[t] = [env.temp.mean(), np.rint(env.grid[0, 1] * 1000).sum() / (1000 * cells),
                  np.rint(env.grid[0, 2] * 1000).sum() / (1000 * cells)]
    return out


def _check_series(s, ref):
    assert s.shape == ref.shape
    np.testing.assert_array_equal(s[:, 1:], ref[:, 1:])
    np.testing.assert_allclose(s[:, 0], ref[:, 0], rtol=1e-9)


@pytest.mark.parametrize("N,n,policy,steps", [(64, 8, "greedy", 40), (128, 37, "antigreedy", 35), (256, 64, "replay", 30),
                                              (128, 16, "none", 20), (256, 40, "greedy", 25)])
def test_single_band_series_matches_oracle(N, n, policy, steps):
    """Starts right after load_state, so step 1 is the literal first step (k_band_first_step); several chunks."""
    light, dark, ai, st = make_state(N, n, seed=N + n, clustered=True)
    acts = np.random.RandomState(1).randint(9, size=(steps, n)) if policy == "replay" else None
    w = _world(N, n)
    w.load_state(light, dark, ai, st)
    cref = full_oracle(w, light, dark, ai, st)
    s = w.run_series(steps, policy, actions=acts, chunk=16)
    _check_series(s, _oracle_series(N, light, dark, ai, st, steps, policy, acts))
    # the series mode does not alter the run: covers, agents and lifespans as the C oracle's
    _, done_at, ada = cref.run(steps, policy, actions=None if acts is None else acts[:, None, :])
    cov = w.local_covers()
    np.testing.assert_array_equal(cov[0], cref.grid[0, 1])
    np.testing.assert_array_equal(cov[1], cref.grid[0, 2])
    xy, stt = w.agents()
    np.testing.assert_array_equal(xy, cref.agent_indices[0])
    np.testing.assert_array_equal(stt, cref.agent_states[0, :, 0])
    d, a = w.lifespans()
    assert d == int(done_at[0]) and w.step_count == steps
    np.testing.assert_array_equal(a, ada[0, :, 0])


def test_series_after_run_over_several_chunks():
    N, n, pre, steps = 128, 30, 7, 45
    light, dark, ai, st = make_state(N, n, seed=21, clustered=True)
    ref = _oracle_series(N, light, dark, ai, st, pre + steps, "greedy")
    w = _world(N, n)
    w.load_state(light, dark, ai, st)
    w.run(pre, "greedy", chunk=4)
    s = w.run_series(steps, "greedy", chunk=16)
    _check_series(s, ref[pre:])
    w.run(3, "greedy")                                   # series mode is off again: run() records nothing
    s2 = w.run_series(2, "greedy")
    ref2 = _oracle_series(N, light, dark, ai, st, pre + steps + 5, "greedy")
    _check_series(s2, ref2[-2:])


@pytest.mark.parametrize("bands,mode", [(2, "nccl"), (4, "nccl"), (2, "p2p"), (4, "p2p")])
def test_banded_series_equals_single_band(bands, mode):
    """Bands of one GPU in lock-step threads (the exchanges of test_gpu_tiled_parity.py): the series summed over the bands
    is the single band's, covers exactly and T to 1e-12 relative (fp64 sums in another order); every rank gets it."""
    import torch
    N, n, steps, policy = 256, 200, 30, "greedy"
    light, dark, ai, st = make_state(N, n, seed=31, clustered=True)
    ai[n // 2:, 0] = (ai[n // 2:, 0] + N // bands) % N          # second cluster on the first interior band boundary
    one = _world(N, n)
    one.load_state(light, dark, ai, st)
    ref = one.run_series(steps, policy, chunk=8)
    shared = ThreadComm.Shared(bands)
    worlds = [_world(N, n, rank=r, world_size=bands, comm=ThreadComm(r, bands, shared), mode=mode) for r in range(bands)]
    streams = [torch.cuda.Stream() for _ in range(bands)]
    if mode == "p2p":
        tables = [w.band.peer_buffers() for w in worlds]
        for r, w in enumerate(worlds):
            w.band.set_stream(streams[r].cuda_stream)
            w.band.attach_peers(r, tables)
    out = {}

    def go(w):
        with torch.cuda.stream(streams[w.rank]):
            w.load_state(light, dark, ai, st)
            s = w.run_series(steps, policy, chunk=8)
            out[w.rank] = (s, w.local_covers(), w.band.peer_timed_out() if mode == "p2p" else False)

    run_threads(worlds, go)
    assert not any(out[r][2] for r in range(bands)), "a peer barrier timed out"
    for r in range(bands):
        s = out[r][0]
        np.testing.assert_array_equal(s[:, 1:], ref[:, 1:])
        np.testing.assert_allclose(s[:, 0], ref[:, 0], rtol=1e-12)
    np.testing.assert_array_equal(np.concatenate([out[r][1] for r in range(bands)], axis=1), one.local_covers())


def test_refused_series_configurations_and_zero_g_at_reset():
    """Series mode cannot be switched inside an open chunk and has nothing to read while off. g = 0 never reaches the
    handle: the temperature is summed as sqrt(g) * T and the tiled kernels scale by g^2, so dwt_set_config refuses it at
    reset (like dwt_create) and keeps the old constants, with which the world still runs its series."""
    from therldaisyworld_b200 import DaisyWorldError
    N, n = 64, 4
    light, dark, ai, st = make_state(N, n, seed=3)
    w = _world(N, n)
    w.load_state(light, dark, ai, st)
    w.step("greedy")                                     # a chunk is open: series mode cannot be switched
    with pytest.raises(DaisyWorldError, match="dwt_set_series"):
        w.band.set_series(True)
    with pytest.raises(DaisyWorldError, match="dwt_get_series"):    # series mode is off: nothing to read
        w.band.take_series(1)
    w.end_chunk()
    g = w.g
    w.g = 0.0
    with pytest.raises(DaisyWorldError, match="dwt_set_config.*g > 0"):
        w.load_state(light, dark, ai, st)
    w.g = g
    w.load_state(light, dark, ai, st)
    s = w.run_series(4, "greedy")
    assert s.shape == (4, 3) and np.isfinite(s).all() and (s[:, 0] > 200).all()
