"""Snapshots of the giant world (BandedDaisyWorld.save / restore), host side on CPU: oracle-backed bands that hold their
state in the representations of dwt_save_state (fp64 planes before the first step, packed lattice words after it, the
pre-state one step behind), over in-process threads and torch.distributed gloo. Checks the shard selection for every
(writer, reader) partition including the wrapped ghost rows of the first and last band, that a world saved on one banding
and restored on another continues exactly like the uninterrupted world, branching, the metadata round trip and the
refusals."""
import json
import os
import socket
import sys

import numpy as np
import pytest

from band_helpers import ThreadComm, make_state, run_threads
from conftest import ROOT
from test_banded_diag_gloo import DiagOracleBand

N, N_AGENTS = 200, 30


def _pack(l, d):
    return (np.rint(l * 1000).astype(np.uint32) | (np.rint(d * 1000).astype(np.uint32) << 16)).astype(np.uint32)


def _unpack(w):
    w = np.asarray(w, dtype=np.uint32)
    return (w & 0xffff) / 1000.0, (w >> 16) / 1000.0


class SnapOracleBand(DiagOracleBand):
    """DiagOracleBand with the snapshot calls of DeviceBand (save_state, restore_state, set_agents, the checksums). The
    current state counts as planes until the first stencil and as the lattice after it; the pre-state follows one step
    behind, like the device handle's flags."""

    def upload(self, light_rows, dark_rows, agent_indices, agent_states):
        super().upload(light_rows, dark_rows, agent_indices, agent_states)
        self.reps = ["planes", "none"]

    def stencil(self, part=0):
        super().stencil(part)
        self.reps = ["lattice", "planes" if self.reps[0] == "planes" else "lattice"]

    def _rows(self, rep, l, d):
        return _pack(l, d) if rep == "lattice" else np.stack([l, d])

    def save_state(self, alloc=None):
        self._absorb_halo()
        alloc = alloc or (lambda which, shape, dtype: np.empty(shape, dtype=dtype))
        out = {}
        for which, rep, (l, d) in (("cur", self.reps[0], (self.l, self.d)), ("pre", self.reps[1], (self.pre or (None, None))[:2])):
            if rep == "none":
                out[which] = None
                continue
            v = self._rows(rep, l[1:-1], d[1:-1])
            out[which] = alloc(which, v.shape, v.dtype)
            out[which][...] = v
        meta = dict(cur_rep=self.reps[0], pre_rep=self.reps[1], L_last=self.L_last, done_at=self.done_at)
        return meta, out["cur"], out["pre"], self.ada.copy()

    def restore_state(self, meta, cur_rows, pre_rows, agents_done_at):
        def planes(rep, rows):
            assert rows.shape == ((self.rows + 2, self.N) if rep == "lattice" else (2, self.rows + 2, self.N))
            return _unpack(rows) if rep == "lattice" else (np.array(rows[0]), np.array(rows[1]))
        self._halo = None
        self.l, self.d = planes(meta["cur_rep"], cur_rows)
        self.pre = None if meta["pre_rep"] == "none" else planes(meta["pre_rep"], pre_rows) + (meta["L_last"],)
        self.reps = [meta["cur_rep"], meta["pre_rep"]]
        self.L_last, self.done_at = meta["L_last"], meta["done_at"]
        self.ada = np.array(agents_done_at, dtype=np.int64).reshape(self.n)
        self.gz = np.zeros(self.n, dtype=bool)
        self.stepmax[:] = 0
        self.j = 0

    def set_agents(self, agent_indices, agent_states):
        self.xy = np.array(agent_indices, dtype=np.int64).reshape(self.n, 2)
        self.st = np.array(agent_states, dtype=np.float64).reshape(self.n)

    def _checksum(self, l, d):
        kl, kd = np.rint(l[1:-1] * 1000).astype(np.uint64), np.rint(d[1:-1] * 1000).astype(np.uint64)
        rows = (self.row0 + np.arange(self.rows)) % self.N
        w = ((rows[:, None] * 131 + np.arange(self.N)[None, :]) % 977 + 1).astype(np.uint64)
        return [int(v) for v in (kl.sum(), kd.sum(), (kl * w).sum(), (kd * w).sum())]

    def cover_checksum(self):
        assert self.reps[0] == "lattice"
        self._absorb_halo()
        return self._checksum(self.l, self.d)

    def pre_checksum(self):
        assert self.reps[1] == "lattice"
        return self._checksum(*self.pre[:2])


def _world(bands, rank=0, shared=None, n=N_AGENTS, dim=N, **kw):
    from therldaisyworld_b200.banded import BandedDaisyWorld
    comm = ThreadComm(rank, bands, shared) if bands > 1 else None
    return BandedDaisyWorld(dim, n, rank=rank, world_size=bands, band_factory=SnapOracleBand, comm=comm, **kw)


def _worlds(bands):
    shared = ThreadComm.Shared(bands)
    return [_world(bands, r, shared) for r in range(bands)]


def _on(worlds, fn):
    """fn(world) on every band (threads when there are several); results in rank order"""
    out = {}
    if len(worlds) == 1:
        out[0] = fn(worlds[0])
    else:
        run_threads(worlds, lambda w: out.__setitem__(w.rank, fn(w)))
    return [out[r] for r in range(len(worlds))]


def _result(w):
    done_at, ada = w.lifespans()
    xy, st = w.agents()
    return dict(covers=w.local_covers(), xy=xy, st=st, done_at=done_at, ada=ada, first=w.first_done_step, step=w.step_count,
                L=w.L, temp=w.diag_stats("temp"), image=w.image("temp", 16))


def _check_same(parts, ref):
    np.testing.assert_array_equal(np.concatenate([p["covers"] for p in parts], axis=1), ref["covers"])
    for p in parts:
        for k in ("xy", "st", "ada"):
            np.testing.assert_array_equal(p[k], ref[k])
        for k in ("done_at", "first", "step", "L"):
            assert p[k] == ref[k], k
        for k in ("mean", "std", "min", "max"):         # merged over the ranks: the same up to the order of the sums
            np.testing.assert_allclose(p["temp"][k], ref["temp"][k], rtol=1e-12)
        np.testing.assert_allclose(p["image"], ref["image"], rtol=1e-12)


def test_shard_pieces_every_partition():
    """Every reader band's rows with both ghost rows come out in order from every writer partition, 1-8 ranks each."""
    from therldaisyworld_b200.banded import balanced_rows, shard_pieces
    for n in (64, 65, 200):
        for writers in range(1, 9):
            ranges = [balanced_rows(n, writers, r) for r in range(writers)]
            shards = [np.arange(lo, hi) for lo, hi in ranges]
            for readers in range(1, 9):
                for r in range(readers):
                    lo, hi = balanced_rows(n, readers, r)
                    got = np.concatenate([shards[k][a:b] for k, a, b in shard_pieces(ranges, n, lo - 1, hi - lo + 2)])
                    np.testing.assert_array_equal(got, np.arange(lo - 1, hi + 1) % n)
    with pytest.raises(ValueError, match="tile"):
        shard_pieces([(0, 10), (11, 20)], 20, 0, 5)
    with pytest.raises(ValueError, match="tile"):
        shard_pieces([(0, 10)], 20, 0, 5)


@pytest.mark.parametrize("k", [0, 1, 3])
@pytest.mark.parametrize("writers,readers", [(1, 3), (3, 1), (2, 4)])
def test_resume_on_another_banding(tmp_path, writers, readers, k):
    """Save after k greedy steps on `writers` bands (k = 0: the reset planes, 1: lattice + planes pre-state, 3: lattice +
    lattice), restore on `readers` bands, continue: equals the uninterrupted single-band world."""
    light, dark, ai, st = make_state(N, N_AGENTS, seed=11, clustered=True)
    M = 4
    ref = _world(1)
    ref.load_state(light, dark, ai, st)
    ref.run(k + M, "greedy")
    ref_res = _result(ref)

    def first(w):
        w.load_state(light, dark, ai, st)
        w.run(k, "greedy")
        w.save(str(tmp_path))

    _on(_worlds(writers), first)

    def second(w):
        w.restore(str(tmp_path))
        w.run(M, "greedy")
        return _result(w)

    _check_same(_on(_worlds(readers), second), ref_res)


def test_pre_state_and_branching(tmp_path):
    """Right after restore the diagnostics of the pre-state equal those before save; branches restored one after the other
    into the same world each equal a fresh uninterrupted run of their policy."""
    light, dark, ai, st = make_state(N, N_AGENTS, seed=5, clustered=True)
    w = _world(1)
    w.load_state(light, dark, ai, st)
    w.run(3, "greedy")
    before = (w.diag_stats("temp"), w.image("beta", 8), w.local_diag("temp"), w.dead_temp)
    w.save(str(tmp_path))
    ws = [_world(1)]

    def branch(policy):
        def fn(x):
            x.restore(str(tmp_path))
            got = (x.diag_stats("temp"), x.image("beta", 8), x.local_diag("temp"), x.dead_temp)
            x.run(4, policy)
            return got, _result(x)
        return _on(ws, fn)

    for policy in ("antigreedy", "greedy", "antigreedy"):
        res = branch(policy)
        (got, _), = res
        assert got[0] == before[0]
        for a, b in zip(got[1:], before[1:]):
            np.testing.assert_array_equal(a, b)
        fresh = _world(1)
        fresh.load_state(light, dark, ai, st)
        fresh.run(3, "greedy")
        fresh.run(4, policy)
        _check_same([r for _, r in res], _result(fresh))


def test_metadata_round_trip_and_refusals(tmp_path):
    from therldaisyworld_b200 import DaisyWorldError
    from therldaisyworld_b200.banded import SNAPSHOT_FORMAT
    light, dark, ai, st = make_state(N, N_AGENTS, seed=2)
    ws = _worlds(3)
    for w in ws:
        w.S, w.agent_gamma = 990.0, 0.04
        w.daisy_kernel = w.daisy_kernel * 1.0
    _on(ws, lambda w: (w.load_state(light, dark, ai, st), w.run(1, "greedy"), w.save(str(tmp_path))))
    meta = json.load(open(tmp_path / "world.json"))
    assert meta["format"] == SNAPSHOT_FORMAT and (meta["N"], meta["n_agents"]) == (N, N_AGENTS)
    assert meta["writer"] == dict(world_size=3, mode="nccl", rows=[[0, 66], [66, 133], [133, 200]])
    assert (meta["cur_rep"], meta["pre_rep"], meta["step_count"], meta["clock"]["step_count"]) == ("lattice", "planes", 1, 1)
    assert meta["pre_checksum"] is None and len(meta["cover_checksum"]) == 4
    assert sorted(os.listdir(tmp_path)) == sorted(["world.json", "agents.npz"] + [f"{s}.rows-{lo:07d}-{hi:07d}.npy" for s in ("cur", "pre")
                                                                               for lo, hi in ((0, 66), (66, 133), (133, 200))])
    w = _world(1)
    w.restore(str(tmp_path))
    assert (w.S, w.agent_gamma) == (990.0, 0.04) and w.q == ws[0].q
    np.testing.assert_array_equal(w.daisy_kernel, ws[0].daisy_kernel)
    assert w.cover_checksum() == meta["cover_checksum"]

    class Untouched(SnapOracleBand):
        def restore_state(self, *a):
            raise AssertionError("the device must not be touched")
        set_params = set_agents = set_clock = restore_state

    from therldaisyworld_b200.banded import BandedDaisyWorld
    for dim, n in ((N + 1, N_AGENTS), (N, N_AGENTS + 1)):
        x = BandedDaisyWorld(dim, n, band_factory=SnapOracleBand)
        x.band.__class__ = Untouched
        with pytest.raises(ValueError, match="does not fit"):
            x.restore(str(tmp_path))
    bad = dict(meta, format=SNAPSHOT_FORMAT + 1)
    other = tmp_path / "other"
    other.mkdir()
    json.dump(bad, open(other / "world.json", "w"))
    with pytest.raises(ValueError, match="format"):
        w.restore(str(other))
    # one flipped word in a shard: the checksum refuses it
    shard = np.load(tmp_path / "cur.rows-0000066-0000133.npy", mmap_mode="r+")
    shard[5, 7] ^= np.uint32(1)
    shard.flush()
    with pytest.raises(DaisyWorldError, match="cover_checksum"):
        w.restore(str(tmp_path))


def _worker(rank, world_size, port, path, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world_size))
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import torch.distributed as dist
    from test_banded_snapshot_gloo import N, N_AGENTS, SnapOracleBand
    from band_helpers import make_state
    from therldaisyworld_b200.banded import BandedDaisyWorld
    dist.init_process_group("gloo", rank=rank, world_size=world_size)
    w = BandedDaisyWorld(N, N_AGENTS, rank=rank, world_size=world_size, band_factory=SnapOracleBand)
    w.load_state(*make_state(N, N_AGENTS, seed=9, clustered=True))
    w.run(3, "greedy")
    w.save(path)
    w.run(2, "antigreedy")
    straight = w.local_covers()
    w.restore(path)
    w.run(2, "antigreedy")
    q.put((rank, straight, w.local_covers(), w.agents()))
    dist.destroy_process_group()


def test_gloo_save_restore(tmp_path):
    """Three gloo ranks save, run on and restore (a branch back to the snapshot); a single band restores their snapshot."""
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    procs = [ctx.Process(target=_worker, args=(r, 3, port, str(tmp_path), q)) for r in range(3)]
    for p in procs:
        p.start()
    res = sorted((q.get(timeout=300) for _ in procs), key=lambda r: r[0])
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    one = _world(1)
    one.restore(str(tmp_path))
    one.run(2, "antigreedy")
    cov = one.local_covers()
    np.testing.assert_array_equal(np.concatenate([r[1] for r in res], axis=1), cov)
    np.testing.assert_array_equal(np.concatenate([r[2] for r in res], axis=1), cov)
    for r in res:
        np.testing.assert_array_equal(r[3][0], one.agents()[0])
        np.testing.assert_array_equal(r[3][1], one.agents()[1])
