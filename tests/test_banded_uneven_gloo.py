"""Host-side logic of the giant world over bands of unequal height (therldaisyworld_b200/banded.py, balanced partition) on
CPU: oracle-backed bands (tests/band_helpers.OracleBand) over in-process threads and over real torch.distributed gloo must
reproduce the full-torus C oracle exactly -- covers, agents, lifespans -- and the climate series of the NumPy oracle."""
import os
import socket
import sys

import numpy as np
import pytest

from conftest import ROOT

N_AGENTS, STEPS = 24, 20
SHAPES = [(200, 3), (333, 4)]        # bands of 66/67/67 and 83/83/83/84 rows


def _state(N, bands):
    from band_helpers import make_state
    from therldaisyworld_b200.banded import balanced_rows
    light, dark, ai, st = make_state(N, N_AGENTS, seed=N, clustered=True)
    ai[N_AGENTS // 2:, 0] = (ai[N_AGENTS // 2:, 0] + balanced_rows(N, bands, 1)[0]) % N   # second cluster on a band boundary
    return light, dark, ai, st


def _actions():
    return np.random.RandomState(3).randint(9, size=(STEPS, N_AGENTS))


def _reference(N, bands, policy):
    from band_helpers import OracleBand, full_oracle
    from therldaisyworld_b200.banded import BandedDaisyWorld
    light, dark, ai, st = _state(N, bands)
    w = BandedDaisyWorld(N, N_AGENTS, band_factory=OracleBand)      # only used as a parameter carrier here
    ref = full_oracle(w, light, dark, ai, st)
    acts = _actions() if policy == "replay" else None
    _, done_at, ada = ref.run(STEPS, policy, actions=None if acts is None else acts[:, None, :])
    return ref, done_at, ada


def _check(results, ref, done_at, ada):
    """results: per rank (covers, (xy, st), (done_at, agents_done_at), step_count)."""
    covers = np.concatenate([r[0] for r in results], axis=1)
    np.testing.assert_array_equal(covers[0], ref.grid[0, 1])
    np.testing.assert_array_equal(covers[1], ref.grid[0, 2])
    for r in results:                                    # agents and counters are replicated: every rank must agree
        np.testing.assert_array_equal(r[1][0], ref.agent_indices[0])
        np.testing.assert_array_equal(r[1][1], ref.agent_states[0, :, 0])
        assert r[2][0] == int(done_at[0])
        np.testing.assert_array_equal(r[2][1], ada[0, :, 0])
        assert r[3] == STEPS


@pytest.mark.parametrize("policy", ["greedy", "antigreedy", "replay"])
@pytest.mark.parametrize("N,bands", SHAPES)
def test_uneven_thread_bands_match_full_torus_oracle(N, bands, policy):
    from band_helpers import OracleBand, ThreadComm, run_threads
    from therldaisyworld_b200.banded import BandedDaisyWorld
    ref, done_at, ada = _reference(N, bands, policy)
    light, dark, ai, st = _state(N, bands)
    shared = ThreadComm.Shared(bands)
    worlds = [BandedDaisyWorld(N, N_AGENTS, rank=r, world_size=bands, band_factory=OracleBand, comm=ThreadComm(r, bands, shared))
              for r in range(bands)]
    assert len({w.rows for w in worlds}) == 2

    def go(w):
        w.load_state(light, dark, ai, st)
        w.run(STEPS, policy, actions=_actions() if policy == "replay" else None, chunk=7)

    run_threads(worlds, go)
    _check([(w.local_covers(), w.agents(), w.lifespans(), w.step_count) for w in worlds], ref, done_at, ada)


def _worker(rank, world_size, port, N, policy, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world_size))
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import torch.distributed as dist
    from band_helpers import OracleBand
    from therldaisyworld_b200.banded import BandedDaisyWorld
    dist.init_process_group("gloo", rank=rank, world_size=world_size)
    light, dark, ai, st = _state(N, world_size)
    w = BandedDaisyWorld(N, N_AGENTS, rank=rank, world_size=world_size, band_factory=OracleBand)
    w.load_state(light, dark, ai, st)
    w.run(STEPS, policy, actions=_actions() if policy == "replay" else None, chunk=8)
    q.put((rank, w.local_covers(), w.agents(), w.lifespans(), w.step_count))
    dist.destroy_process_group()


@pytest.mark.parametrize("N,bands,policy", [(200, 3, "greedy"), (333, 4, "antigreedy"), (200, 3, "replay")])
def test_uneven_gloo_ranks_match_full_torus_oracle(N, bands, policy):
    import torch.multiprocessing as mp
    ref, done_at, ada = _reference(N, bands, policy)
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    procs = [ctx.Process(target=_worker, args=(r, bands, port, N, policy, q)) for r in range(bands)]
    for p in procs:
        p.start()
    res = sorted((q.get(timeout=300) for _ in procs), key=lambda r: r[0])
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    _check([r[1:] for r in res], ref, done_at, ada)


def test_balanced_partition():
    from therldaisyworld_b200.banded import balanced_rows, band_rows
    assert [balanced_rows(200, 3, r) for r in range(3)] == [(0, 66), (66, 133), (133, 200)]
    assert [balanced_rows(333, 4, r) for r in range(4)] == [(0, 83), (83, 166), (166, 249), (249, 333)]
    assert [balanced_rows(192, 2, r) for r in range(2)] == [(0, 96), (96, 192)]
    for N in (64, 65, 127, 192, 200, 333, 1000, 16350, 16384):
        for R in range(1, 9):
            parts = [balanced_rows(N, R, r) for r in range(R)]
            assert parts[0][0] == 0 and parts[-1][1] == N
            assert all(a[1] == b[0] for a, b in zip(parts, parts[1:]))              # contiguous, in rank order
            heights = [hi - lo for lo, hi in parts]
            assert max(heights) - min(heights) <= 1 and min(heights) >= 8
            try:
                equal = [band_rows(N, R, r) for r in range(R)]
            except ValueError:
                continue
            assert parts == equal
    with pytest.raises(ValueError):
        balanced_rows(200, 3, 3)


@pytest.mark.parametrize("N,bands", SHAPES)
def test_uneven_thread_bands_series_match_full_torus_oracle(N, bands):
    from band_helpers import ThreadComm, run_threads
    from test_banded_series_gloo import SeriesOracleBand
    from therldaisyworld_b200.banded import BandedDaisyWorld
    from oracle.daisy_numpy import OracleDaisyWorld, OracleGreedy
    light, dark, ai, st = _state(N, bands)
    env = OracleDaisyWorld(grid_dimension=N, n_agents=N_AGENTS)
    env.batch_size = 1
    env.grid = np.zeros((1, 7, N, N))
    env.grid[0, 1], env.grid[0, 2] = light, dark
    env.agent_indices = ai[None].copy()
    env.agent_states = st[None, :, None].copy()
    agent, obs = OracleGreedy(greedy=True), env.get_obs(env.agent_indices)
    ref = np.zeros((STEPS, 3))
    for t in range(STEPS):
        obs, _, _, _ = env.step(agent(obs))
        ref[t] = [env.temp.mean(), np.rint(env.grid[0, 1] * 1000).sum() / (1000.0 * N * N),
                  np.rint(env.grid[0, 2] * 1000).sum() / (1000.0 * N * N)]
    shared = ThreadComm.Shared(bands)
    worlds = [BandedDaisyWorld(N, N_AGENTS, rank=r, world_size=bands, band_factory=SeriesOracleBand, comm=ThreadComm(r, bands, shared))
              for r in range(bands)]
    out = {}

    def go(w):
        w.load_state(light, dark, ai, st)
        out[w.rank] = w.run_series(STEPS, "greedy", chunk=6)

    run_threads(worlds, go)
    for r in range(bands):
        np.testing.assert_array_equal(out[r][:, 1:], ref[:, 1:])
        np.testing.assert_allclose(out[r][:, 0], ref[:, 0], rtol=1e-12)
