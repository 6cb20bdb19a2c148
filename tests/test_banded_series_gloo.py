"""Host-side logic of BandedDaisyWorld.run_series on CPU: oracle-backed bands record their partial sums of the temperature
and covers per step, the driver sums them over the bands once per chunk, and the result must be the per-step means of
the full-torus NumPy oracle -- covers exactly, temperature to 1e-12 relative."""
import numpy as np
import pytest

from band_helpers import OracleBand, ThreadComm, make_state, run_threads

N, N_AGENTS, STEPS, CHUNK = 256, 24, 23, 8          # 4 bands of 64 rows; K spans several chunks, the last one partial


class SeriesOracleBand(OracleBand):
    """OracleBand with series mode: row j of a [4096, 3] buffer holds this band's {sum T, sum milli-light, sum milli-dark}
    of the j-th step of the open chunk, like dwt_get_series_ptr (without the device's sqrt(g) scaling)."""

    def __init__(self, *a, **kw):
        super().__init__(*a, **kw)
        self.series = self._torch.zeros((4096, 3), dtype=self._torch.float64)
        self.series_on = False

    def set_series(self, on):
        assert self.j == 0, "series mode switched while a chunk is open"
        self.series_on = bool(on)

    def stencil(self, part=0):
        if self.series_on:
            self.o.L = self.clk.L
            T = self.o.fields(self.l[None], self.d[None])["T"][0, 1:-1]     # the band's own rows, not the ghost rows
            j = self.j
        super().stencil(part)
        if self.series_on:
            kl = np.rint(self.l[1:-1] * 1000).sum()
            kd = np.rint(self.d[1:-1] * 1000).sum()
            self.series[j] = self._torch.tensor([T.sum(), kl, kd], dtype=self._torch.float64)

    def series_tensor(self, K):
        return self.series[:K]

    def take_series(self, K):
        return self.series[:K].numpy().copy()

    def end_chunk(self, K):
        self.series[:self.j] = 0.0
        return super().end_chunk(K)


def _oracle_series(light, dark, ai, st, steps, policy="greedy"):
    """Per-step (mean T, mean light, mean dark) of the full torus, the NumPy oracle stepped with its Greedy restatement."""
    from oracle.daisy_numpy import OracleDaisyWorld, OracleGreedy
    env = OracleDaisyWorld(grid_dimension=N, n_agents=N_AGENTS)
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
        obs, _, _, _ = env.step(agent(obs))
        out[t] = [env.temp.mean(), np.rint(env.grid[0, 1] * 1000).sum() / (1000 * cells),
                  np.rint(env.grid[0, 2] * 1000).sum() / (1000 * cells)]
    return out


@pytest.mark.parametrize("world_size", [1, 2, 4])
def test_thread_bands_series_match_full_torus_oracle(world_size):
    from therldaisyworld_b200.banded import BandedDaisyWorld
    light, dark, ai, st = make_state(N, N_AGENTS, seed=9, clustered=True)
    ai[N_AGENTS // 2:, 0] = (ai[N_AGENTS // 2:, 0] + N // world_size) % N     # second cluster on a band boundary
    ref = _oracle_series(light, dark, ai, st, STEPS)
    shared = ThreadComm.Shared(world_size)
    worlds = [BandedDaisyWorld(N, N_AGENTS, rank=r, world_size=world_size, band_factory=SeriesOracleBand,
                               comm=ThreadComm(r, world_size, shared) if world_size > 1 else None) for r in range(world_size)]
    out = {}

    def go(w):
        w.load_state(light, dark, ai, st)                # the literal first step is part of the series
        out[w.rank] = w.run_series(STEPS, "greedy", chunk=CHUNK)

    run_threads(worlds, go)
    for r in range(world_size):                          # every rank returns the same whole-world series
        s = out[r]
        assert s.shape == (STEPS, 3)
        np.testing.assert_array_equal(s[:, 1:], ref[:, 1:])
        np.testing.assert_allclose(s[:, 0], ref[:, 0], rtol=1e-12)
        assert worlds[r].step_count == STEPS and not worlds[r].band.series_on


def test_series_continues_after_run():
    """run() first (series off: nothing recorded), then run_series: the series picks up at the next step."""
    from therldaisyworld_b200.banded import BandedDaisyWorld
    light, dark, ai, st = make_state(N, N_AGENTS, seed=4, clustered=True)
    ref = _oracle_series(light, dark, ai, st, 5 + STEPS)
    w = BandedDaisyWorld(N, N_AGENTS, band_factory=SeriesOracleBand)
    w.load_state(light, dark, ai, st)
    w.run(5, "greedy", chunk=CHUNK)
    assert not w.band.series.any()
    s = w.run_series(STEPS, "greedy", chunk=CHUNK)
    np.testing.assert_array_equal(s[:, 1:], ref[5:, 1:])
    np.testing.assert_allclose(s[:, 0], ref[5:, 0], rtol=1e-12)
