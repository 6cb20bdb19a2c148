"""Observations of the giant world (dwt_observe, k_band_obs) and the MLP policy on it (DW_POLICY_MLP over the observation
buffer): exact parity with the full-torus C oracle on one band and on bands of one GPU, NCCL-style and in peer-memory
mode, with agents clustered on the torus wrap and on band boundaries (several agents per cell: the highest-index stamp),
the reset observation, non-default masks, a host MLP driving env_step, the device MLP in run / run_series, and the
refusals."""
import numpy as np
import pytest

from band_helpers import ThreadComm, full_oracle, make_state, run_threads
from test_banded_obs_gloo import golden_mlp_params, oracle_env, state

pytestmark = pytest.mark.gpu


def _world(N, n, **kw):
    from therldaisyworld_b200.banded import BandedDaisyWorld
    return BandedDaisyWorld(N, n, **kw)


def _bands(N, n, bands, mode, **kw):
    """`bands` handles of one world on one GPU, each on its own stream; peer-memory mode attaches them to each other."""
    import torch
    shared = ThreadComm.Shared(bands)
    worlds = [_world(N, n, rank=r, world_size=bands, comm=ThreadComm(r, bands, shared), mode=mode, **kw) for r in range(bands)]
    streams = [torch.cuda.Stream() for _ in range(bands)]
    if mode == "p2p":
        tables = [w.band.peer_buffers() for w in worlds]
        for r, w in enumerate(worlds):
            w.band.set_stream(streams[r].cuda_stream)
            w.band.attach_peers(r, tables)
    return worlds, streams


def _reference(world, light, dark, ai, st):
    """C oracle of the whole torus, holding initialize_grid's fields so that its first observation is the reset one."""
    from oracle.daisy_c import COracleWorld
    env = oracle_env(world, light, dark, ai, st)          # the reset clock, whatever the world has run since
    return COracleWorld(env, grid=env.grid, agent_indices=ai[None].copy(), agent_states=st[None, :, None].copy())


def _random_params(scale, seed):
    """Random weights as in test_device_mlp_equals_oracle_mlp_on_random_weights, except for the first layer's rows of the
    bare fraction and the temperatures (zero) and of ch4 (scaled by 1/300): inputs that are nearly the same everywhere
    would otherwise dominate a network without biases and pick one action for every agent. The covers and the agent
    stamp decide then."""
    from oracle.daisy_numpy import OracleMLP
    p = np.random.RandomState(seed).randn(OracleMLP.N_PARAMS) * scale
    w1 = p[:63 * 16].reshape(63, 16)
    w1[0:9], w1[27:36], w1[45:54] = 0.0, 0.0, 0.0
    w1[36:45] /= 300.0
    return p


class _Script:
    """The policies of a run, applied to the oracle's own observations: the same actions the world takes."""

    def __init__(self, policy, n, steps, params=None):
        from oracle.daisy_numpy import OracleGreedy, OracleMLP
        self.policy = policy
        self.acts = np.random.RandomState(11).randint(9, size=(steps, n))
        self.greedy = OracleGreedy(greedy=True)
        self.mlp = OracleMLP(params) if params is not None else None
        self.hist = np.zeros(9, dtype=int)

    def oracle_action(self, t, obs):
        if self.policy == "replay":
            a = self.acts[t][None, :, None]
        elif self.policy == "greedy":
            a = self.greedy(obs)
        else:
            a = self.mlp(obs)
        self.hist += np.bincount(np.asarray(a).ravel(), minlength=9)
        return a


def _oracle_loop(ref, script, steps):
    """[(obs, reward, done)] of each step of the C oracle; obs[0] is its observation before the first step."""
    out = [(ref.get_obs(), None, None)]
    for t in range(steps):
        out.append(ref.step(script.oracle_action(t, out[-1][0])))
    return out


def _world_step(w, script, t):
    """One step of the world: env_step for replay (host actions), the device policy otherwise."""
    if script.policy == "replay":
        return w.env_step(script.acts[t])[:3]
    w.step(script.policy)
    return w.observe(), None, None


def _check_step(got, exp):
    np.testing.assert_array_equal(got[0], exp[0])
    if got[1] is not None:
        np.testing.assert_array_equal(got[1], exp[1])
        np.testing.assert_array_equal(got[2], exp[2])


@pytest.mark.parametrize("N", [64, 130, 333])
@pytest.mark.parametrize("policy", ["greedy", "replay"])
def test_single_band_observe_matches_oracle(N, policy):
    """300 agents in a 5x5 patch around (0, 0): windows wrap in both directions and cells hold several agents."""
    n, steps = 300, 12
    light, dark, ai, st = make_state(N, n, seed=N, clustered=True)
    w = _world(N, n)
    w.load_state(light, dark, ai, st)
    ref = _reference(w, light, dark, ai, st)
    script = _Script(policy, n, steps)
    exp = _oracle_loop(ref, script, steps)
    np.testing.assert_array_equal(w.observe(), exp[0][0])              # the reset observation
    for t in range(steps):
        _check_step(_world_step(w, script, t), exp[t + 1])
    np.testing.assert_array_equal(w.agents()[0], ref.agent_indices[0])
    np.testing.assert_array_equal(w.agents()[1], ref.agent_states[0, :, 0])


def test_reset_observation_is_initialize_grid():
    """Right after load_state: initialize_grid's unrounded fields at min_L, no agent stamp (NumPy oracle), also after a
    second load_state over a stepped world."""
    N, n = 96, 40
    light, dark, ai, st = make_state(N, n, seed=2, clustered=True)
    w = _world(N, n)
    exp = oracle_env(w, light, dark, ai, st).get_obs(ai[None])
    w.load_state(light, dark, ai, st)
    np.testing.assert_array_equal(w.observe(), exp)
    w.run(3, "greedy")
    w.load_state(light, dark, ai, st)
    np.testing.assert_array_equal(w.observe(), exp)


@pytest.mark.parametrize("mode", ["moore", "circular"])
def test_masks(mode):
    """The mask comes from dw_config.obs_mask (at kr = 1 the circular mask is the Von Neumann cross)."""
    N, n, steps = 130, 200, 8
    light, dark, ai, st = make_state(N, n, seed=5, clustered=True)
    w = _world(N, n, neighborhood_mode=mode)
    w.load_state(light, dark, ai, st)
    ref = _reference(w, light, dark, ai, st)
    script = _Script("replay", n, steps)
    exp = _oracle_loop(ref, script, steps)
    np.testing.assert_array_equal(w.observe(), exp[0][0])
    for t in range(steps):
        _check_step(_world_step(w, script, t), exp[t + 1])


def test_env_step_without_agents():
    """n_agents == 0: reward [[any light, any dark]] and done its negation, every step."""
    N = 64
    light, dark, _, _ = make_state(N, 0, seed=4)
    w = _world(N, 0)
    ai, st = np.zeros((0, 2), dtype=np.int64), np.zeros(0)
    w.load_state(light, dark, ai, st)
    ref = full_oracle(w, light, dark, ai, st)
    assert w.observe().shape == (1, 0, 7, 3, 3)
    for _ in range(5):
        obs, reward, done, info = w.env_step()
        e_obs, e_reward, e_done, _ = ref.step(None)
        assert obs.shape == e_obs.shape and info == {}
        np.testing.assert_array_equal(reward, e_reward)
        np.testing.assert_array_equal(done, e_done)
        assert reward.dtype == e_reward.dtype and done.dtype == e_done.dtype


def _run_bands(worlds, streams, fn):
    import torch
    out = {}

    def go(w):
        with torch.cuda.stream(streams[w.rank]):
            out[w.rank] = fn(w)
            if w.mode == "p2p":
                assert not w.band.peer_timed_out(), "a peer barrier timed out"

    run_threads(worlds, go)
    return [out[r] for r in range(len(worlds))]


@pytest.mark.parametrize("mode", ["nccl", "p2p"])
@pytest.mark.parametrize("N,bands,policy", [(200, 3, "greedy"), (333, 4, "replay"), (200, 4, "greedy")])
def test_uneven_bands_observe_matches_oracle(mode, N, bands, policy):
    """Every rank's observe() equals the oracle's: windows of agents on a band boundary straddle two owners."""
    n, steps = 300, 10
    worlds, streams = _bands(N, n, bands, mode)
    light, dark, ai, st = state(N, bands, n=n)
    ref = _reference(worlds[0], light, dark, ai, st)
    script = _Script(policy, n, steps)
    exp = _oracle_loop(ref, script, steps)

    def fn(w):
        w.load_state(light, dark, ai, st)
        res = [(w.observe(), None, None)]
        for t in range(steps):
            res.append(_world_step(w, script, t))
        return res

    for res in _run_bands(worlds, streams, fn):
        for got, e in zip(res, exp):
            _check_step(got, e)


def _closed_loop(w, mlp, steps):
    """A host policy (OracleMLP) drives env_step; returns the observations, rewards, done flags and the final state."""
    obs = w.observe()
    res = [obs]
    for _ in range(steps):
        obs, reward, done, _ = w.env_step(mlp(obs))
        res += [obs, reward, done]
    return res + [w.local_covers(), *w.agents(), *w.lifespans()]


@pytest.mark.parametrize("bands,mode", [(1, "local"), (3, "nccl"), (3, "p2p")])
def test_host_mlp_closed_loop(bands, mode):
    from oracle.daisy_numpy import OracleMLP
    N, n, steps = 200, 150, 30
    mlp = OracleMLP(golden_mlp_params())
    light, dark, ai, st = state(N, bands, n=n)
    if bands == 1:
        w = _world(N, n)
        w.load_state(light, dark, ai, st)
        results = [_closed_loop(w, mlp, steps)]
        carrier = w
    else:
        worlds, streams = _bands(N, n, bands, mode)

        def fn(w):
            w.load_state(light, dark, ai, st)
            return _closed_loop(w, mlp, steps)

        results = _run_bands(worlds, streams, fn)
        carrier = worlds[0]
    ref = _reference(carrier, light, dark, ai, st)
    obs = ref.get_obs()
    exp = [obs]
    done_at, ada = 0, np.zeros(n, dtype=np.int64)
    for _ in range(steps):
        obs, reward, done, _ = ref.step(mlp(obs))
        exp += [obs, reward, done]
        done_at += int(ref.grid[0, 1:3].max() > 0.005)
        ada += ~done[0, :, 0]
    for res in results:
        for k, (a, b) in enumerate(zip(res[:len(exp)], exp)):
            np.testing.assert_array_equal(a, b, err_msg=f"item {k}")
        np.testing.assert_array_equal(res[-3], ref.agent_states[0, :, 0])
        np.testing.assert_array_equal(res[-4], ref.agent_indices[0])
        assert res[-2] == done_at
        np.testing.assert_array_equal(res[-1], ada)
    covers = np.concatenate([r[len(exp)] for r in results], axis=1)
    np.testing.assert_array_equal(covers[0], ref.grid[0, 1])
    np.testing.assert_array_equal(covers[1], ref.grid[0, 2])


def _oracle_mlp_run(world, light, dark, ai, st, params, steps):
    """The NumPy oracle stepped with OracleMLP on its own observations from the reset: per-step series (mean T, mean light,
    mean dark), final state, action histogram."""
    from oracle.daisy_numpy import OracleMLP
    env = oracle_env(world, light, dark, ai, st)
    mlp = OracleMLP(params)
    obs = env.get_obs(env.agent_indices)
    series = np.zeros((steps, 3))
    hist = np.zeros(9, dtype=int)
    N = light.shape[0]
    for t in range(steps):
        a = mlp(obs)
        hist += np.bincount(a.ravel(), minlength=9)
        obs = env.step(a)[0]
        series[t] = [env.temp.mean(), np.rint(env.grid[0, 1] * 1000).sum() / (1000.0 * N * N),
                     np.rint(env.grid[0, 2] * 1000).sum() / (1000.0 * N * N)]
    return env, obs, series, hist


PARAM_SETS = [("golden", None), ("random", 0.3), ("random", 1.0), ("random", 3.0)]
# One network per scale. A network without biases picks the same actions at every scale (the logits scale by scale^3), so
# the seed is what makes the networks differ; these seeds give networks that pick at least 6 distinct actions on the
# states of both tests below (most seeds give 4 or more, some only 2 or 3).
_SEEDS = {0.3: 1, 1.0: 2, 3.0: 7}


def _params(which, scale):
    return golden_mlp_params() if which == "golden" else _random_params(scale, seed=_SEEDS[scale])


@pytest.mark.parametrize("N", [130, 256])
@pytest.mark.parametrize("which,scale", PARAM_SETS)
def test_device_mlp_run_and_series_match_oracle(N, which, scale):
    """run(K, "mlp") and run_series from a reset (the first decision reads the reset observation)."""
    n, steps = 200, 24
    params = _params(which, scale)
    light, dark, ai, st = make_state(N, n, seed=N + 1, clustered=True)
    w = _world(N, n)
    env, obs, series, hist = _oracle_mlp_run(w, light, dark, ai, st, params, steps)
    assert (hist > 0).sum() >= (2 if which == "golden" else 4), hist        # the golden network picks 5 and 6 here
    w.set_mlp(params)
    w.load_state(light, dark, ai, st)
    w.run(steps, "mlp", chunk=10)
    np.testing.assert_array_equal(w.observe(), obs)
    np.testing.assert_array_equal(w.agents()[0], env.agent_indices[0])
    np.testing.assert_array_equal(w.agents()[1], env.agent_states[0, :, 0])
    np.testing.assert_array_equal(w.local_covers(), env.grid[0, 1:3])
    w.load_state(light, dark, ai, st)
    s = w.run_series(steps, "mlp", chunk=10)
    np.testing.assert_array_equal(s[:, 1:], series[:, 1:])
    np.testing.assert_allclose(s[:, 0], series[:, 0], rtol=1e-9)
    np.testing.assert_array_equal(w.agents()[0], env.agent_indices[0])


@pytest.mark.parametrize("N,bands", [(200, 3), (333, 4)])
@pytest.mark.parametrize("which,scale", [("golden", None), ("random", 1.0)])
def test_device_mlp_over_nccl_bands_matches_oracle(N, bands, which, scale):
    n, steps = 200, 20
    params = _params(which, scale)
    worlds, streams = _bands(N, n, bands, "nccl")
    light, dark, ai, st = state(N, bands, n=n)
    env, obs, series, hist = _oracle_mlp_run(worlds[0], light, dark, ai, st, params, steps)
    assert (hist > 0).sum() >= (2 if which == "golden" else 4), hist

    def fn(w):
        w.set_mlp(params)
        w.load_state(light, dark, ai, st)
        s = w.run_series(steps, "mlp", chunk=7)
        return s, w.observe(), w.agents(), w.local_covers()

    res = _run_bands(worlds, streams, fn)
    for s, o, (xy, stt), _ in res:
        np.testing.assert_array_equal(s[:, 1:], series[:, 1:])
        np.testing.assert_allclose(s[:, 0], series[:, 0], rtol=1e-9)
        np.testing.assert_array_equal(o, obs)
        np.testing.assert_array_equal(xy, env.agent_indices[0])
        np.testing.assert_array_equal(stt, env.agent_states[0, :, 0])
    np.testing.assert_array_equal(np.concatenate([r[3] for r in res], axis=1), env.grid[0, 1:3])


def test_mlp_refused_in_peer_memory_mode_before_the_step():
    from therldaisyworld_b200 import DaisyWorldError
    N, n = 200, 40
    worlds, streams = _bands(N, n, 2, "p2p")
    light, dark, ai, st = state(N, 2, n=n)

    def fn(w):
        w.set_mlp(golden_mlp_params())
        w.load_state(light, dark, ai, st)
        w.step("greedy")
        clk = w.band.get_clock().step_count
        with pytest.raises(DaisyWorldError, match="peer-memory"):
            w.step("mlp")
        with pytest.raises(DaisyWorldError, match="peer-memory"):
            w.run(3, "mlp")
        assert w.band.get_clock().step_count == clk and w._pending == 1
        w.step("greedy")
        return w.observe()

    a, b = _run_bands(worlds, streams, fn)
    np.testing.assert_array_equal(a, b)


def test_refusals():
    from therldaisyworld_b200 import DaisyWorldError
    from therldaisyworld_b200.banded import DeviceBand
    N, n = 64, 10
    light, dark, ai, st = make_state(N, n, seed=1)
    w = _world(N, n)
    with pytest.raises(DaisyWorldError, match="dwt_observe.*no state"):
        w.band.observe()
    w.load_state(light, dark, ai, st)
    with pytest.raises(DaisyWorldError, match="dwt_set_mlp"):
        w.step("mlp")                                    # no weights
    with pytest.raises(DaisyWorldError, match="dwt_set_mlp.*1808"):
        w.set_mlp(np.zeros(1807))
    w.set_mlp(golden_mlp_params())
    w.step("greedy")
    with pytest.raises(DaisyWorldError, match="dwt_decide.*dwt_observe"):
        w.band.decide("mlp")                             # stale: the step changed the state since the last observe
    w.band.observe()
    w.band.decide("mlp")
    w.band.time_stencil(2)
    with pytest.raises(DaisyWorldError, match="dwt_observe.*dwt_debug_time_stencil"):
        w.observe()
    w.step("greedy")
    assert w.observe().shape == (1, n, 7, 3, 3)
    d = DeviceBand(w, N, n, 0, N, 1)                     # a handle that never observes
    with pytest.raises(DaisyWorldError, match="dwt_get_obs"):
        d.get_obs()
    with pytest.raises(DaisyWorldError, match="dwt_decide"):
        d.decide("mlp")
