"""Snapshots of the giant world on the GPU (dwt_save_state / dwt_restore_state, BandedDaisyWorld.save / restore). The
reference of every check is the uninterrupted run of the same world, compared bit for bit: a world saved, restored into a
fresh handle (or banding) and run on must give the same covers, agents, lifespans, checksum, observations, statistics,
images and series. Covers every state kind (the reset planes, lattice with the planes pre-state, lattice with the lattice
pre-state), every device policy, the pre-state right after restore, re-banding between one band and 3 / 4 bands of one
GPU in NCCL-style and peer-memory mode, branching, and the refusals."""
import ctypes as C

import numpy as np
import pytest

from band_helpers import make_state
from test_banded_obs_gloo import golden_mlp_params, state
from test_gpu_tiled_obs import _bands, _run_bands, _world

pytestmark = pytest.mark.gpu

POLICIES = ["greedy", "eps_greedy", "random", "replay", "mlp"]
M = 6                                                    # steps after the snapshot


def _start(w, N, n, k):
    """k = "device": the reset drawn on the device; k >= 0: clustered agents around (0, 0) loaded from the host, then k
    greedy steps."""
    if k == "device":
        w.reset_on_device(seed=N)
    else:
        w.load_state(*make_state(N, n, seed=N, clustered=True))
        w.run(k, "greedy")


def _policy_setup(w):
    w.band.set_epsilon(0.4)
    w.set_mlp(golden_mlp_params())


def _pre_outputs(w, has_pre):
    """what reads the pre-state (and the current state): observe, the temperature field, its statistics and image"""
    out = {"obs": w.observe()}
    if has_pre:
        out.update(temp=w.local_diag("temp"), stats=w.diag_stats("temp"), image=w.image("temp", 16))
    return out


def _continue(w, policy, actions, seed=17):
    series = w.run_series(M, policy, actions=actions, seed=seed)
    done_at, ada = w.lifespans()
    xy, st = w.agents()
    return dict(series=series, covers=w.local_covers(), xy=xy, st=st, done_at=done_at, ada=ada, first=w.first_done_step,
                step=w.step_count, L=w.L, checksum=w.cover_checksum(), obs=w.observe(), stats=w.diag_stats("temp"),
                image=w.image("temp", 16))


def _assert_same(got, ref, exact=True):
    """exact: the same banding (statistics and images bit for bit); otherwise the merged statistics and images may differ
    in the order of their sums (1e-12 relative). The series' temperature column is added up with fp64 atomics inside the
    step kernels, so its order of summation varies from run to run even on one banding (1e-12 relative); the cover columns
    are integer sums and exact."""
    for k in ("covers", "xy", "st", "ada", "obs"):
        np.testing.assert_array_equal(got[k], ref[k], err_msg=k)
    for k in ("done_at", "first", "step", "L", "checksum"):
        assert got[k] == ref[k], k
    if exact:
        assert got["stats"] == ref["stats"]
        np.testing.assert_array_equal(got["image"], ref["image"])
    else:
        for s in ("mean", "std", "min", "max"):
            np.testing.assert_allclose(got["stats"][s], ref["stats"][s], rtol=1e-12)
        np.testing.assert_allclose(got["image"], ref["image"], rtol=1e-12)
    np.testing.assert_allclose(got["series"][:, 0], ref["series"][:, 0], rtol=1e-12)
    np.testing.assert_array_equal(got["series"][:, 1:], ref["series"][:, 1:])


@pytest.mark.parametrize("N", [64, 200, 333])
@pytest.mark.parametrize("k", ["device", 0, 1, 3])
def test_resume_every_state_kind_and_policy(tmp_path, N, k):
    """Save after k steps (k = 0 and the device reset: planes, no pre-state; 1: lattice + planes pre-state; 3: lattice +
    lattice), restore into a fresh world: the pre-state's outputs equal those before save, and M steps of every policy equal
    the uninterrupted run."""
    n = 300
    actions = np.random.RandomState(5).randint(9, size=(M, n))
    w = _world(N, n)
    _policy_setup(w)
    _start(w, N, n, k)
    has_pre = k not in ("device", 0)
    before = _pre_outputs(w, has_pre)
    w.save(str(tmp_path))
    for policy in POLICIES:
        ref = _world(N, n)
        _policy_setup(ref)
        _start(ref, N, n, k)
        exp = _continue(ref, policy, actions)
        got_w = _world(N, n)
        _policy_setup(got_w)
        got_w.restore(str(tmp_path))
        after = _pre_outputs(got_w, has_pre)
        assert after.keys() == before.keys()
        for key in before:
            if key == "stats":
                assert after[key] == before[key]
            else:
                np.testing.assert_array_equal(after[key], before[key], err_msg=key)
        _assert_same(_continue(got_w, policy, actions), exp)


def test_mlp_step_right_after_restore(tmp_path):
    """An MLP step reads the restored pre-state's observation: no extra step is needed first."""
    N, n = 200, 300
    w = _world(N, n)
    w.set_mlp(golden_mlp_params())
    _start(w, N, n, 4)
    w.save(str(tmp_path))
    w.step("mlp")
    ref = w.local_covers(), w.agents()
    x = _world(N, n)
    x.set_mlp(golden_mlp_params())
    x.restore(str(tmp_path))
    x.step("mlp")
    np.testing.assert_array_equal(x.local_covers(), ref[0])
    for a, b in zip(x.agents(), ref[1]):
        np.testing.assert_array_equal(a, b)


def _release(worlds):
    """Destroy the bands of a finished phase now, while no band of this process steps: dwt_destroy frees device and
    page-locked memory, which waits for the whole device."""
    import gc
    worlds.clear()
    gc.collect()


def _banded_continue(worlds, streams, policy="greedy"):
    """M steps on every band (step by step, as a banded world runs) and the results merged like _continue's."""
    def fn(w):
        series = w.run_series(M, policy, seed=17)
        done_at, ada = w.lifespans()
        xy, st = w.agents()
        return dict(series=series, covers=w.local_covers(), xy=xy, st=st, done_at=done_at, ada=ada, first=w.first_done_step,
                    step=w.step_count, L=w.L, checksum=w.cover_checksum(), obs=w.observe(), stats=w.diag_stats("temp"),
                    image=w.image("temp", 16))

    res = _run_bands(worlds, streams, fn)
    out = dict(res[0])
    out["covers"] = np.concatenate([r["covers"] for r in res], axis=1)
    # cover_checksum() sums over the ranks only with torch.distributed; the in-process bands return their own parts
    out["checksum"] = [sum(c) % (1 << 64) for c in zip(*(r["checksum"] for r in res))]
    for r in res[1:]:
        for key in ("xy", "st", "ada", "obs", "image", "series"):
            np.testing.assert_array_equal(r[key], res[0][key])
        assert r["stats"] == res[0]["stats"]
    return out


@pytest.mark.parametrize("save_on,restore_on", [((1, "local"), (3, "nccl")), ((1, "local"), (4, "p2p")),
                                                ((4, "p2p"), (1, "local")), ((4, "p2p"), (3, "nccl"))])
def test_reband(tmp_path, save_on, restore_on):
    """N = 333: 3 bands of 111 rows, 4 unequal bands of 83 / 83 / 83 / 84; agents clustered on the first band boundary
    too. Every combination equals the single-band uninterrupted run; no peer barrier times out. A peer-memory band refuses
    to save while the last step's agents are unfinished; save() finishes them first."""
    from therldaisyworld_b200 import DaisyWorldError
    _release([])                                         # earlier tests' handles, before any band of this one steps
    N, n, k = 333, 300, 3
    light, dark, ai, st = state(N, 4, n=n)
    ref = _world(N, n)
    ref.load_state(light, dark, ai, st)
    ref.run(k, "greedy")
    exp = _continue(ref, "greedy", None)

    def start(w):
        w.load_state(light, dark, ai, st)
        w.run(k - 1, "greedy")
        w.step("greedy")
        if w.mode == "p2p":                              # the agents of that step are finished by the next step or a flush
            with pytest.raises(DaisyWorldError, match="dwt_save_state.*not finished"):
                w.band.save_state()
        w.save(str(tmp_path))

    def banded(bands, mode):
        if bands == 1:
            return [_world(N, n)], None
        return _bands(N, n, bands, mode)

    worlds, streams = banded(*save_on)
    if streams is None:
        start(worlds[0])
    else:
        _run_bands(worlds, streams, start)
    _release(worlds)
    worlds, streams = banded(*restore_on)
    if streams is None:
        worlds[0].restore(str(tmp_path))
        got = _continue(worlds[0], "greedy", None)
    else:
        _run_bands(worlds, streams, lambda w: w.restore(str(tmp_path)))
        got = _banded_continue(worlds, streams)
    _release(worlds)
    _assert_same(got, exp, exact=restore_on[0] == 1)


def test_branching_in_peer_memory_mode(tmp_path):
    """One snapshot restored three times into the same 3-band peer-memory world, each branch with another policy: each
    equals a fresh uninterrupted single-band run of that policy, so nothing of the previous branch (series rows, claims,
    look-ahead decisions, lifespans) leaks into the next."""
    _release([])
    N, n, k = 200, 300, 4
    light, dark, ai, st = state(N, 3, n=n)
    one = _world(N, n)
    one.load_state(light, dark, ai, st)
    one.run(k, "greedy")
    one.save(str(tmp_path))
    worlds, streams = _bands(N, n, 3, "p2p")
    for policy in ("greedy", "random", "antigreedy"):
        ref = _world(N, n)
        ref.load_state(light, dark, ai, st)
        ref.run(k, "greedy")
        exp = _continue(ref, policy, None)
        _run_bands(worlds, streams, lambda w: w.restore(str(tmp_path)))
        _assert_same(_banded_continue(worlds, streams, policy), exp, exact=False)


def test_refusals_and_integrity(tmp_path):
    from therldaisyworld_b200 import DaisyWorldError
    from therldaisyworld_b200._lib import DwtBandState
    N, n = 200, 50
    w = _world(N, n)
    _start(w, N, n, 3)
    w.save(str(tmp_path))
    # another N or n: refused before any device call
    for dim, agents in ((256, n), (N, n + 1)):
        x = _world(dim, agents)
        calls = []
        for name in ("restore_state", "set_params", "set_agents", "set_clock"):
            setattr(x.band, name, lambda *a, _name=name: calls.append(_name))
        with pytest.raises(ValueError, match="does not fit"):
            x.restore(str(tmp_path))
        assert not calls
    b = w.band
    # agents of a step open, and a chunk open
    b.decide("greedy")
    b.move_graze()
    with pytest.raises(DaisyWorldError, match="dwt_save_state.*not finished"):
        b.save_state()
    b.finish_agents()
    b.stencil(0)
    b.halo_wrap()
    with pytest.raises(DaisyWorldError, match="dwt_save_state.*chunk is open"):
        b.save_state()
    w._pending += 1
    w.end_chunk()
    b.save_state()
    # bad representations
    rows = np.zeros((N + 2, N), dtype=np.uint32)
    p = rows.ctypes.data
    for cur, pre in ((7, 0), (2, 9), (1, 1), (1, 2), (0, 0), (-1, 0)):
        m = DwtBandState(cur_rep=cur, pre_rep=pre, L_last=1.0, done_at=0)
        assert b._lib.dwt_restore_state(b._h, C.byref(m), p, p, None) == -1, (cur, pre)
    assert b._lib.dwt_restore_state(b._h, C.byref(DwtBandState(cur_rep=2, pre_rep=2)), p, None, None) == -1
    # one flipped word of a shard: the whole-world checksum refuses it (current state, then pre-state)
    x = _world(N, n)
    x.restore(str(tmp_path))
    for which, name in (("cur", "cover_checksum"), ("pre", "pre_checksum")):
        f = tmp_path / f"{which}.rows-0000000-0000200.npy"
        a = np.load(f, mmap_mode="r+")
        a[17, 5] ^= np.uint32(1 << 16)
        a.flush()
        with pytest.raises(DaisyWorldError, match=name):
            x.restore(str(tmp_path))
        a[17, 5] ^= np.uint32(1 << 16)
        a.flush()
    x.restore(str(tmp_path))
