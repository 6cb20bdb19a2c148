"""Observations of the giant world and the MLP policy on it (BandedDaisyWorld.observe / env_step / policy="mlp"), host side
on CPU: oracle-backed bands that keep their pre-state and observe only the window cells in rows they own, over in-process
threads and over torch.distributed gloo. The bands' partial observations summed over the ranks, the rewards and the
MLP-driven steps must equal the full-torus NumPy oracle exactly. This checks the host sequencing of an MLP step (finish
the last step's agents, observe, all-reduce, decide) without a GPU."""
import os
import socket
import sys

import numpy as np
import pytest

from band_helpers import OracleBand
from conftest import GOLDEN_DIR, ROOT

N_AGENTS = 24
SHAPES = [(200, 3), (333, 4)]        # bands of 66/67/67 and 83/83/83/84 rows
STEPS_ENV, STEPS_MLP, STEPS_GREEDY = 6, 8, 4


class ObsOracleBand(OracleBand):
    """OracleBand that also observes: it keeps the post-graze pre-state (and luminosity) each stencil starts from, evaluates
    the window cells whose rows it owns from it and writes 0 everywhere else, like dwt_observe; decide("mlp") maps the
    (summed) observation through OracleMLP on every rank."""

    def __init__(self, params, N, n_agents, row0, rows, n_ranks):
        super().__init__(params, N, n_agents, row0, rows, n_ranks)
        self.mask = np.asarray(params.neighborhood, dtype=np.float64)
        self.obs = self._torch.zeros((n_agents, 7, 3, 3), dtype=self._torch.float64)
        self.mlp = None

    def upload(self, light_rows, dark_rows, agent_indices, agent_states):
        super().upload(light_rows, dark_rows, agent_indices, agent_states)
        self.pre = None                  # None: the reset state itself is current

    def stencil(self, part=0):
        self.pre = (self.l.copy(), self.d.copy(), self.clk.L)
        super().stencil(part)

    def _band_grid(self):
        """[7, rows + 2, N] of the current state; only the band's own rows 1..rows are meaningful."""
        from oracle.daisy_numpy import round3
        o = self.o
        if self.pre is None:             # initialize_grid's unrounded fields, no agent stamp
            l, d = self.l, self.d
            o.L = self.clk.L
            f = o.fields(l[None], d[None])
            return np.stack([o.p - l - d, l, d, f["T"][0], f["Tl"][0], f["Td"][0], np.zeros_like(l)])
        l, d, o.L = self.pre
        f = o.fields(l[None], d[None])
        nl = np.clip(l + o.dt * f["dl"][0], 0, 1)
        nd = np.clip(d + o.dt * f["dd"][0], 0, 1)
        g = round3(np.stack([o.p - nl - nd, nl, nd, f["T"][0], f["Tl"][0], f["Td"][0], np.zeros_like(l)]))
        for i in range(self.n):          # last index wins, dead agents included
            lr = self._owned(self.xy[i, 0])
            if lr >= 0:
                g[4, lr, self.xy[i, 1]] = self.st[i]
        return g

    def observe(self):
        g = self._band_grid()
        out = np.zeros((self.n, 7, 3, 3))
        for i in range(self.n):
            for a in range(3):
                x = (self.xy[i, 0] + a - 1) % self.N
                lr = self._owned(x)
                if lr < 0:
                    continue
                for c in range(3):
                    out[i, :, a, c] = g[:, lr, (self.xy[i, 1] + c - 1) % self.N] * self.mask[a, c]
        self.obs.copy_(self._torch.from_numpy(out))

    def obs_tensor(self):
        return self.obs

    def get_obs(self):
        return self.obs.numpy().copy()

    def set_mlp(self, params):
        from oracle.daisy_numpy import OracleMLP
        self.mlp = OracleMLP(params)

    def decide(self, policy, actions_step=None, seed=0):
        if policy != "mlp":
            return super().decide(policy, actions_step, seed)
        self._absorb_halo()
        self.act[:] = self._torch.from_numpy(self.mlp(self.obs.numpy()[None])[0, :, 0] + 1.0)


def golden_mlp_params():
    return np.load(os.path.join(GOLDEN_DIR, "mlp_n16_b4_mixed_150.npz"))["mlp_params"]


def state(N, bands, n=N_AGENTS, seed=None):
    """Clustered agents around (0, 0) and a second cluster on the first interior band boundary."""
    from band_helpers import make_state
    from therldaisyworld_b200.banded import balanced_rows
    light, dark, ai, st = make_state(N, n, seed=N if seed is None else seed, clustered=True)
    if bands > 1:
        ai[n // 2:, 0] = (ai[n // 2:, 0] + balanced_rows(N, bands, 1)[0]) % N
    return light, dark, ai, st


def replay_actions(steps, n, seed=3):
    return np.random.RandomState(seed).randint(9, size=(steps, n))


def drive(w, light, dark, ai, st, params, acts):
    """The sequence both sides run: the reset observation, env_step with explicit and with no actions, MLP steps, greedy
    steps; returns the observations (with reward / done of the env_steps) and the final agents."""
    out = []
    w.load_state(light, dark, ai, st)
    out.append(w.observe())
    for t in range(STEPS_ENV):
        out.extend(w.env_step(acts[t])[:3])
    out.extend(w.env_step(None)[:3])
    w.set_mlp(params)
    for _ in range(STEPS_MLP):
        w.step("mlp")
        out.append(w.observe())
    for _ in range(STEPS_GREEDY):
        w.step("greedy")
        out.append(w.observe())
    out.extend(w.agents())
    return out


def reference_drive(world, light, dark, ai, st, params, acts):
    """drive() on the full-torus NumPy oracle (batch 1), the policies evaluated on its own observations."""
    from oracle.daisy_numpy import OracleGreedy, OracleMLP
    n = ai.shape[0]
    env = oracle_env(world, light, dark, ai, st)
    obs = env.get_obs(env.agent_indices)
    out = [obs]
    for t in range(STEPS_ENV):
        obs, reward, done, _ = env.step(np.asarray(acts[t]).reshape(1, n, 1))
        out += [obs, reward, done]
    obs, reward, done, _ = env.step(None)
    out += [obs, reward, done]
    mlp, greedy = OracleMLP(params), OracleGreedy(greedy=True)
    for _ in range(STEPS_MLP):
        obs = env.step(mlp(obs))[0]
        out.append(obs)
    for _ in range(STEPS_GREEDY):
        obs = env.step(greedy(obs))[0]
        out.append(obs)
    out += [env.agent_indices[0], env.agent_states[0, :, 0]]
    return out


def oracle_env(world, light, dark, ai, st):
    """The full-torus NumPy oracle (batch 1) with the world's constants, right after a reset to the given state."""
    from oracle.daisy_numpy import OracleDaisyWorld
    N, n = light.shape[0], ai.shape[0]
    env = OracleDaisyWorld(grid_dimension=N, n_agents=n)
    for k in ("p", "g", "S", "sigma", "gamma", "q", "q2", "temp_optimal", "dt", "agent_gamma", "albedo_bare", "albedo_light",
              "albedo_dark", "neighborhood", "min_L", "max_L", "ramp_period"):
        setattr(env, k, getattr(world, k))
    env.batch_size, env.L, env.step_count = 1, world.min_L, 0
    env.dL = (env.max_L - env.min_L) / env.ramp_period
    env.grid = reset_grid(env, light, dark)
    env.agent_indices, env.agent_states = ai[None].copy(), st[None, :, None].copy()
    return env


def reset_grid(env, light, dark):
    """initialize_grid's [1, 7, N, N] for given covers (daisy_world_rl.py:304-324): unrounded fields at env.L."""
    N = light.shape[0]
    grid = np.zeros((1, 7, N, N))
    grid[0, 0], grid[0, 1], grid[0, 2] = env.p - light - dark, light, dark
    f = env.fields(grid[:, 1], grid[:, 2])
    grid[:, 3], grid[:, 4], grid[:, 5] = f["T"], f["Tl"], f["Td"]
    return grid


def check(out, ref):
    assert len(out) == len(ref)
    for k, (a, b) in enumerate(zip(out, ref)):
        assert np.shape(a) == np.shape(b), k
        np.testing.assert_array_equal(a, b, err_msg=f"item {k}")


def _reference(N, bands):
    from therldaisyworld_b200.banded import BandedDaisyWorld
    light, dark, ai, st = state(N, bands)
    carrier = BandedDaisyWorld(N, N_AGENTS, band_factory=ObsOracleBand)
    return reference_drive(carrier, light, dark, ai, st, golden_mlp_params(), replay_actions(STEPS_ENV, N_AGENTS))


@pytest.mark.parametrize("N,bands", SHAPES)
def test_thread_bands_observe_and_mlp_match_full_torus_oracle(N, bands):
    from band_helpers import ThreadComm, run_threads
    from therldaisyworld_b200.banded import BandedDaisyWorld
    ref = _reference(N, bands)
    light, dark, ai, st = state(N, bands)
    shared = ThreadComm.Shared(bands)
    worlds = [BandedDaisyWorld(N, N_AGENTS, rank=r, world_size=bands, band_factory=ObsOracleBand, comm=ThreadComm(r, bands, shared))
              for r in range(bands)]
    assert len({w.rows for w in worlds}) == 2
    out = {}

    def go(w):
        out[w.rank] = drive(w, light, dark, ai, st, golden_mlp_params(), replay_actions(STEPS_ENV, N_AGENTS))

    run_threads(worlds, go)
    for r in range(bands):                               # every rank returns the whole observation
        check(out[r], ref)


def test_single_band_observe_and_mlp_match_full_torus_oracle():
    from therldaisyworld_b200.banded import BandedDaisyWorld
    N = 130
    ref = _reference(N, 1)
    light, dark, ai, st = state(N, 1)
    w = BandedDaisyWorld(N, N_AGENTS, band_factory=ObsOracleBand)
    check(drive(w, light, dark, ai, st, golden_mlp_params(), replay_actions(STEPS_ENV, N_AGENTS)), ref)


def test_env_step_rejects_bad_actions_before_stepping():
    from therldaisyworld_b200.banded import BandedDaisyWorld
    N, n = 64, 5
    light, dark, ai, st = state(N, 1, n=n)
    w = BandedDaisyWorld(N, n, band_factory=ObsOracleBand)
    w.load_state(light, dark, ai, st)
    for bad in (np.zeros(n + 1, dtype=int), np.zeros((2, n), dtype=int), np.zeros((1, n, 2), dtype=int), np.full(n, 9),
                np.full(n, -1), np.zeros(n) + 0.5):
        with pytest.raises(ValueError):
            w.env_step(bad)
    assert w.step_count == 0 and w._pending == 0
    for shape in ((n,), (1, n), (1, n, 1)):
        obs, reward, done, info = w.env_step(np.zeros(shape, dtype=np.int64))
        assert obs.shape == (1, n, 7, 3, 3) and reward.shape == done.shape == (1, n, 1) and info == {}
    assert w._pending == 3


def _worker(rank, world_size, port, N, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world_size))
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import torch.distributed as dist
    from test_banded_obs_gloo import ObsOracleBand, drive, golden_mlp_params, replay_actions, state
    from therldaisyworld_b200.banded import BandedDaisyWorld
    dist.init_process_group("gloo", rank=rank, world_size=world_size)
    light, dark, ai, st = state(N, world_size)
    w = BandedDaisyWorld(N, N_AGENTS, rank=rank, world_size=world_size, band_factory=ObsOracleBand)
    q.put((rank, drive(w, light, dark, ai, st, golden_mlp_params(), replay_actions(STEPS_ENV, N_AGENTS))))
    dist.destroy_process_group()


@pytest.mark.parametrize("N,bands", SHAPES)
def test_gloo_ranks_observe_and_mlp_match_full_torus_oracle(N, bands):
    import torch.multiprocessing as mp
    ref = _reference(N, bands)
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    procs = [ctx.Process(target=_worker, args=(r, bands, port, N, q)) for r in range(bands)]
    for p in procs:
        p.start()
    res = sorted((q.get(timeout=300) for _ in procs), key=lambda r: r[0])
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    for _, out in res:
        check(out, ref)
