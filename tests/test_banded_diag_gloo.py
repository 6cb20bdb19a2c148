"""Diagnostics and plot feed of the giant world (BandedDaisyWorld.local_diag / diag_stats / cover_stats / image /
dead_temp / run_with_series), host side on CPU: oracle-backed bands that keep their pre-state and return their own part
of each statistic and image, like dwt_get_diag_stats / dwt_get_cover_stats / dwt_pool, over in-process threads and over
torch.distributed gloo. Checks the merge over the ranks (one SUM all-reduce of a per-rank table, Chan's formula over
unequal counts), edge blocks of images, identical results on every rank and agreement with the full-torus NumPy world."""
import os
import socket
import sys

import numpy as np
import pytest

from band_helpers import OracleBand
from conftest import ROOT

N, BANDS, N_AGENTS, STEPS = 200, 3, 30, 5          # bands of 66 / 67 / 67 rows
BLOCKS = [1, 7, 16, 64, 200]
DIAG = ["temp", "temp_light", "temp_dark", "temp_effective", "beta", "beta_l", "beta_d", "growth"]
GRID = {"grid_bare": 0, "grid_light": 1, "grid_dark": 2, "grid_temp": 3, "grid_temp_dark": 5}
_KEYS = {"temp": "T", "temp_light": "Tl", "temp_dark": "Td", "temp_effective": "Te", "beta": "beta", "beta_l": "beta_l",
         "beta_d": "beta_d", "growth_l": "dl", "growth_d": "dd"}


class DiagOracleBand(OracleBand):
    """OracleBand with the diagnostic calls of DeviceBand: the fields come from the NumPy oracle's forward over the band
    padded with its ghost rows, from the post-graze pre-state each stencil starts from; statistics, covers and block sums
    are over the band's own rows only."""

    def upload(self, light_rows, dark_rows, agent_indices, agent_states):
        super().upload(light_rows, dark_rows, agent_indices, agent_states)
        self.pre = None
        self.L_last = self.clk.L

    def stencil(self, part=0):
        self.pre = (self.l.copy(), self.d.copy(), self.clk.L)
        self.L_last = self.clk.L
        super().stencil(part)

    def _field(self, name):
        """[rows, N] of a DWT_FIELD name (rows of the band only)."""
        from oracle.daisy_numpy import round3
        assert self.pre is not None
        l, d, self.o.L = self.pre
        f = {k: v[0] for k, v in self.o.fields(l[None], d[None]).items() if np.ndim(v) == 3}
        if name in GRID:
            nl = np.clip(l + self.o.dt * f["dl"], 0, 1)
            nd = np.clip(d + self.o.dt * f["dd"], 0, 1)
            v = round3([self.o.p - nl - nd, nl, nd, f["T"], None, f["Td"]][GRID[name]])
        else:
            v = f[_KEYS[name]]
        return v[1:-1]

    def diag(self, name):
        if name == "growth":
            return np.stack([self._field("growth_l"), self._field("growth_d")])
        return self._field(name)

    def diag_stats(self, name):
        v = self.diag(name).ravel()
        m = v.mean()
        return np.array([v.size, m, ((v - m) ** 2).sum(), v.min(), v.max()])

    def cover_stats(self):
        self._absorb_halo()
        l, d = self.l[1:-1], self.d[1:-1]
        return np.array([l.sum(), d.sum(), l.max(), d.max()])

    def pool(self, field, block):
        v = self._field(field)
        H = -(-self.N // block)
        out = np.zeros((H, H))
        rows = (self.row0 + np.arange(self.rows)) % self.N
        np.add.at(out, (rows[:, None] // block, np.arange(self.N)[None, :] // block), v)
        return self._torch.from_numpy(out)

    def synchronize(self):
        pass

    def last_L(self):
        return self.L_last


def state(seed=7):
    from band_helpers import make_state
    return make_state(N, N_AGENTS, seed=seed, clustered=True)


def drive(w, light, dark, ai, st):
    """Reset, STEPS greedy steps, then every diagnostic; a run_with_series afterwards."""
    w.load_state(light, dark, ai, st)
    out = {"cover_reset": w.cover_stats(), "dead_reset": w.dead_temp}
    for _ in range(STEPS):
        w.step("greedy")
    out["stats"] = {f: w.diag_stats(f) for f in DIAG}
    out["stats_again"] = w.diag_stats("temp")
    out["cover"] = w.cover_stats()
    out["images"] = {(f, b): w.image(f, b) for f in DIAG + list(GRID) for b in BLOCKS if f != "growth" or b in (1, 16)}
    out["local"] = {f: w.local_diag(f) for f in DIAG}
    out["dead"] = w.dead_temp
    out["series"] = w.run_with_series(7, every=3, images=("temp", "grid_light"), block=64)
    return out


def reference(world, light, dark, ai, st):
    """The full-torus NumPy world after the same reset and greedy steps."""
    from oracle.daisy_numpy import OracleGreedy
    from test_banded_obs_gloo import oracle_env
    env = oracle_env(world, light, dark, ai, st)
    reset = {"cover": (light.mean(), dark.mean(), light.max(), dark.max()),
             "dead": ((env.S * env.L * (1 - env.albedo_bare)) / env.sigma) ** 0.25}
    greedy = OracleGreedy(greedy=True)
    obs = env.get_obs(env.agent_indices)
    for _ in range(STEPS):
        L = env.L
        obs = env.step(greedy(obs))[0]
    fields = {"temp": env.temp[0, 0], "temp_light": env.temp_light[0, 0], "temp_dark": env.temp_dark[0, 0],
              "temp_effective": env.temp_effective[0, 0], "beta": env.beta[0, 0], "beta_l": env.beta_l[0, 0],
              "beta_d": env.beta_d[0, 0], "growth": env.growth[0], "growth_l": env.growth[0, 0], "growth_d": env.growth[0, 1]}
    fields.update({k: env.grid[0, ch] for k, ch in GRID.items()})
    dead = ((env.S * L * (1 - env.albedo_bare)) / env.sigma) ** 0.25
    return env, fields, reset, dead


def block_means(v, b):
    H = -(-v.shape[-1] // b)
    out = np.zeros(v.shape[:-2] + (H, H))
    for i in range(H):
        for j in range(H):
            out[..., i, j] = v[..., i * b:(i + 1) * b, j * b:(j + 1) * b].mean(axis=(-2, -1))
    return out


def check_against_reference(out, fields, reset, dead):
    c = out["cover_reset"]
    np.testing.assert_allclose([c["mean_light"], c["mean_dark"]], reset["cover"][:2], rtol=1e-12)
    assert (c["max_light"], c["max_dark"]) == reset["cover"][2:]
    assert out["dead_reset"][0] == pytest.approx(reset["dead"], rel=1e-15)
    for f in DIAG:
        v, s = fields[f], out["stats"][f]
        np.testing.assert_allclose([s["mean"], s["std"]], [v.mean(), v.std()], rtol=1e-9)
        assert s["min"] == v.min() and s["max"] == v.max()
    assert out["stats_again"] == out["stats"]["temp"]
    c = out["cover"]
    np.testing.assert_allclose([c["mean_light"], c["mean_dark"]], [fields["grid_light"].mean(), fields["grid_dark"].mean()], rtol=1e-12)
    assert c["max_light"] == fields["grid_light"].max() and c["max_dark"] == fields["grid_dark"].max()
    for (f, b), img in out["images"].items():
        H = -(-N // b)
        assert img.shape == ((2, H, H) if f == "growth" else (H, H))
        if b == 1:
            np.testing.assert_array_equal(img, fields[f])
        else:
            np.testing.assert_allclose(img, block_means(fields[f], b), rtol=1e-12, atol=1e-300)
    assert out["dead"][0] == pytest.approx(dead, rel=1e-15)
    for rec in out["series"]:
        assert list(rec) == ["step", "L", "temp_mean", "temp_std", "dead_temp", "light", "dark", "images"]
        assert set(rec["images"]) == {"temp", "grid_light"} and rec["images"]["temp"].shape == (4, 4)
    assert [rec["step"] for rec in out["series"]] == [STEPS + 3, STEPS + 6, STEPS + 7]


def test_edge_blocks_and_chan_merge():
    """Block means with blocks that do not divide N (edge blocks of 200 - 192 = 8 rows at block 64), and the pairwise merge
    over unequal counts against NumPy on the concatenated data."""
    from therldaisyworld_b200.banded import BandedDaisyWorld
    rng = np.random.RandomState(0)
    parts = [rng.randn(n) * s + m for n, s, m in ((66, 1.0, 300.0), (134, 3.0, 290.0), (1, 0.0, 250.0))]
    rows = np.array([[p.size, p.mean(), ((p - p.mean()) ** 2).sum(), p.min(), p.max()] for p in parts])
    n, mean, m2, mn, mx = BandedDaisyWorld._merge_stats(rows)
    allv = np.concatenate(parts)
    assert n == allv.size and mn == allv.min() and mx == allv.max()
    np.testing.assert_allclose([mean, np.sqrt(m2 / n)], [allv.mean(), allv.std()], rtol=1e-12)
    v = rng.rand(N, N)
    band = DiagOracleBand.__new__(DiagOracleBand)
    import torch
    band._torch, band.N, band.row0, band.rows = torch, N, 0, N
    band._field = lambda name: v
    sums = band.pool("temp", 64).numpy()
    assert sums.shape == (4, 4) and sums[3, 3] == pytest.approx(v[192:, 192:].sum())
    np.testing.assert_allclose(sums / np.outer([64, 64, 64, 8], [64, 64, 64, 8]), block_means(v, 64), rtol=1e-12)


def test_single_band_matches_full_torus():
    from therldaisyworld_b200.banded import BandedDaisyWorld
    light, dark, ai, st = state()
    w = BandedDaisyWorld(N, N_AGENTS, band_factory=DiagOracleBand)
    out = drive(w, light, dark, ai, st)
    _, fields, reset, dead = reference(w, light, dark, ai, st)
    check_against_reference(out, fields, reset, dead)
    for f in DIAG:
        np.testing.assert_array_equal(out["local"][f], fields[f])


def _same(a, b):
    """identical results (bits) on every rank"""
    if isinstance(a, dict):
        assert a.keys() == b.keys()
        for k in a:
            _same(a[k], b[k])
    elif isinstance(a, list):
        assert len(a) == len(b)
        for x, y in zip(a, b):
            _same(x, y)
    else:
        np.testing.assert_array_equal(a, b)


def _check_ranks(outs, world):
    light, dark, ai, st = state()
    _, fields, reset, dead = reference(world, light, dark, ai, st)
    for out in outs:
        without_local = {k: v for k, v in out.items() if k != "local"}
        _same(without_local, {k: v for k, v in outs[0].items() if k != "local"})
        check_against_reference(out, fields, reset, dead)
    for f in DIAG:
        axis = 1 if f == "growth" else 0
        np.testing.assert_array_equal(np.concatenate([o["local"][f] for o in outs], axis=axis), fields[f])


def test_thread_bands_match_full_torus():
    from band_helpers import ThreadComm, run_threads
    from therldaisyworld_b200.banded import BandedDaisyWorld
    shared = ThreadComm.Shared(BANDS)
    worlds = [BandedDaisyWorld(N, N_AGENTS, rank=r, world_size=BANDS, band_factory=DiagOracleBand, comm=ThreadComm(r, BANDS, shared))
              for r in range(BANDS)]
    assert len({w.rows for w in worlds}) == 2
    light, dark, ai, st = state()
    out = {}

    def go(w):
        out[w.rank] = drive(w, light, dark, ai, st)

    run_threads(worlds, go)
    _check_ranks([out[r] for r in range(BANDS)], worlds[0])


def _worker(rank, world_size, port, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world_size))
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import torch.distributed as dist
    from test_banded_diag_gloo import DiagOracleBand, drive, state
    from therldaisyworld_b200.banded import BandedDaisyWorld
    dist.init_process_group("gloo", rank=rank, world_size=world_size)
    w = BandedDaisyWorld(N, N_AGENTS, rank=rank, world_size=world_size, band_factory=DiagOracleBand)
    q.put((rank, drive(w, *state())))
    dist.destroy_process_group()


def test_gloo_ranks_match_full_torus():
    import torch.multiprocessing as mp
    from therldaisyworld_b200.banded import BandedDaisyWorld
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    procs = [ctx.Process(target=_worker, args=(r, BANDS, port, q)) for r in range(BANDS)]
    for p in procs:
        p.start()
    res = sorted((q.get(timeout=300) for _ in procs), key=lambda r: r[0])
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    _check_ranks([out for _, out in res], BandedDaisyWorld(N, N_AGENTS, band_factory=DiagOracleBand))
