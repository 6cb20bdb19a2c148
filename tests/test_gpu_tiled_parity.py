"""GPU parity of the single-giant-grid path (TMA-tiled stencil kernel + parallel agent kernels, dwt_* C-ABI) against the
full-torus C oracle at reduced N, on one band and on several bands of one GPU (exchanges done in-process)."""
import numpy as np
import pytest

from band_helpers import ThreadComm, full_oracle, make_state, run_threads

pytestmark = pytest.mark.gpu


def _world(N, n, **kw):
    from therldaisyworld_b200.banded import BandedDaisyWorld
    return BandedDaisyWorld(N, n, **kw)


def _compare(worlds, ref, done_at, ada, full_grid=True):
    covers = np.concatenate([w.local_covers() for w in worlds], axis=1)
    np.testing.assert_array_equal(covers[0], ref.grid[0, 1])
    np.testing.assert_array_equal(covers[1], ref.grid[0, 2])
    for w in worlds:
        xy, st = w.agents()
        np.testing.assert_array_equal(xy, ref.agent_indices[0])
        np.testing.assert_array_equal(st, ref.agent_states[0, :, 0])
        d, a = w.lifespans()
        assert d == int(done_at[0])
        np.testing.assert_array_equal(a, ada[0, :, 0])
    if full_grid:
        grid = np.concatenate([w.local_grid() for w in worlds], axis=1)
        np.testing.assert_array_equal(grid, ref.grid[0])


@pytest.mark.parametrize("N,n,policy,steps,clustered", [
    (64, 8, "greedy", 70, True), (128, 37, "greedy", 60, False), (128, 64, "antigreedy", 33, True),
    (256, 300, "replay", 40, True), (192, 0, "none", 25, False), (128, 16, "none", 20, False), (64, 5, "greedy", 1, True)])
def test_single_band_matches_oracle(N, n, policy, steps, clustered):
    light, dark, ai, st = make_state(N, n, seed=N + n, clustered=clustered)
    w = _world(N, n)
    w.load_state(light, dark, ai, st)
    ref = full_oracle(w, light, dark, ai, st)
    acts = np.random.RandomState(1).randint(9, size=(steps, n)) if policy == "replay" else None
    w.run(steps, policy, actions=acts, chunk=16)
    _, done_at, ada = ref.run(steps, policy, actions=None if acts is None else acts[:, None, :])
    assert w.step_count == steps and w.L == ref.L
    _compare([w], ref, done_at, ada)


def test_single_band_to_death_and_non_default_params():
    """Neutral-ish albedos, faster ramp: the whole life of a 64x64 world through the tiled kernel, step by step phases."""
    N, n = 64, 6
    light, dark, ai, st = make_state(N, n, seed=11)
    w = _world(N, n, ramp_period=96)
    w.albedo_light, w.albedo_dark, w.gamma = 0.7, 0.3, 0.3
    w.load_state(light, dark, ai, st)
    ref = full_oracle(w, light, dark, ai, st)
    steps, done_at, ada = ref.run(100000, "greedy", stop_all_done=True)
    for _ in range(steps):
        w.step("greedy")
    assert w.lifespans()[0] == int(done_at[0]) and w.first_done_step == steps
    _compare([w], ref, done_at, ada)


@pytest.mark.parametrize("bands,policy", [(2, "greedy"), (4, "antigreedy"), (4, "replay")])
def test_bands_on_one_gpu_match_oracle(bands, policy):
    """Band ownership, ghost rows, replicated agents: `bands` handles on one GPU stepping in lock-step threads."""
    N, n, steps = 256, 200, 30
    light, dark, ai, st = make_state(N, n, seed=7, clustered=True)
    ai[n // 2:, 0] = (ai[n // 2:, 0] + N // bands) % N          # second cluster on the first interior band boundary
    shared = ThreadComm.Shared(bands)
    worlds = [_world(N, n, rank=r, world_size=bands, comm=ThreadComm(r, bands, shared)) for r in range(bands)]
    ref = full_oracle(worlds[0], light, dark, ai, st)
    acts = np.random.RandomState(2).randint(9, size=(steps, n)) if policy == "replay" else None

    def go(w):
        w.load_state(light, dark, ai, st)
        w.run(steps, policy, actions=acts, chunk=8)

    run_threads(worlds, go)
    _, done_at, ada = ref.run(steps, policy, actions=None if acts is None else acts[:, None, :])
    _compare(worlds, ref, done_at, ada)


@pytest.mark.parametrize("bands,policy,n", [(2, "greedy", 200), (4, "antigreedy", 200), (4, "replay", 200), (2, "none", 200),
                                            (2, "greedy", 900), (4, "antigreedy", 1500), (2, "greedy", "sms+1")])
def test_peer_memory_mode_bands_on_one_gpu(bands, policy, n):
    """dwt_step_p2p: owners publish decisions / gains into every band's exchange vector, edge rows are pushed into the
    neighbours' ghost rows, bands meet at device-side flag barriers. Here the 'peers' are bands of one process on one GPU,
    each on its own stream (the IPC variant of the same code path runs in tools/banded_nccl_check.py)."""
    import torch
    N, steps = 256, 30               # n > 256: several blocks in the agent kernels (grid barrier of k_band_fmc_graze)
    if n == "sms+1":                 # one block more than there are SMs: move/claim and graze as two launches on the lattice
        n = 256 * torch.cuda.get_device_properties(0).multi_processor_count + 1
    light, dark, ai, st = make_state(N, n, seed=17, clustered=True)
    ai[n // 2:, 0] = (ai[n // 2:, 0] + N // bands) % N
    shared = ThreadComm.Shared(bands)
    worlds = [_world(N, n, rank=r, world_size=bands, comm=ThreadComm(r, bands, shared), mode="p2p") for r in range(bands)]
    streams = [torch.cuda.Stream() for _ in range(bands)]
    tables = [w.band.peer_buffers() for w in worlds]
    for r, w in enumerate(worlds):
        w.band.set_stream(streams[r].cuda_stream)
        w.band.attach_peers(r, tables)
    ref = full_oracle(worlds[0], light, dark, ai, st)
    acts = np.random.RandomState(4).randint(9, size=(steps, n)) if policy == "replay" else None
    out = {}

    def go(w):
        with torch.cuda.stream(streams[w.rank]):
            w.load_state(light, dark, ai, st)
            w.run(steps, policy, actions=acts, chunk=8)
            out[w.rank] = (w.local_covers(), w.agents(), w.lifespans(), w.local_grid(), w.band.peer_timed_out())

    run_threads(worlds, go)
    _, done_at, ada = ref.run(steps, policy, actions=None if acts is None else acts[:, None, :])
    assert not any(out[r][4] for r in range(bands)), "a peer barrier timed out"
    covers = np.concatenate([out[r][0] for r in range(bands)], axis=1)
    np.testing.assert_array_equal(covers[0], ref.grid[0, 1])
    np.testing.assert_array_equal(covers[1], ref.grid[0, 2])
    np.testing.assert_array_equal(np.concatenate([out[r][3] for r in range(bands)], axis=1), ref.grid[0])
    for r in range(bands):
        np.testing.assert_array_equal(out[r][1][0], ref.agent_indices[0])
        np.testing.assert_array_equal(out[r][1][1], ref.agent_states[0, :, 0])
        assert out[r][2][0] == int(done_at[0])
        np.testing.assert_array_equal(out[r][2][1], ada[0, :, 0])


def test_device_reset_is_banding_invariant_and_fast_path_is_used():
    """dwt_init_random keys the RNG by global cell index: 1 band and 2 bands draw and evolve the same world."""
    N, n, steps = 128, 50, 25
    one = _world(N, n)
    one.reset_on_device(seed=3)
    one.run(steps, "greedy")
    shared = ThreadComm.Shared(2)
    two = [_world(N, n, rank=r, world_size=2, comm=ThreadComm(r, 2, shared)) for r in range(2)]

    def go(w):
        w.reset_on_device(seed=3)
        w.run(steps, "greedy")

    run_threads(two, go)
    np.testing.assert_array_equal(np.concatenate([w.local_covers() for w in two], axis=1), one.local_covers())
    np.testing.assert_array_equal(two[0].agents()[1], one.agents()[1])
    np.testing.assert_array_equal(two[1].lifespans()[1], one.lifespans()[1])
    cov = one.local_covers()
    assert cov.max() > 0.05 and (cov * 1000 == np.rint(cov * 1000)).all()
    # the literal fallback must be the exception, not the rule
    assert one.band.slow_count() < 1e-3 * steps * N * N
