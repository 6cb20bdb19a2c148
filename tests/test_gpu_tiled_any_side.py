"""The giant world at sides and band heights that are not a multiple of 64 (masked instance of the tiled stencil kernel over
the partial tiles, padded lattice layout, bands of unequal height): exact parity with the full-torus C oracle on one band,
on bands of one GPU with NCCL-style exchanges and in peer-memory mode, the climate series against the NumPy oracle, and
the storage outside the band left untouched."""
import numpy as np
import pytest

from band_helpers import ThreadComm, full_oracle, make_state, run_threads
from test_gpu_tiled_series import _oracle_series

pytestmark = pytest.mark.gpu


def _world(N, n, **kw):
    from therldaisyworld_b200.banded import BandedDaisyWorld
    return BandedDaisyWorld(N, n, **kw)


def _check_exact(covers, agents, lifespans, grid, ref, done_at, ada):
    np.testing.assert_array_equal(covers[0], ref.grid[0, 1])
    np.testing.assert_array_equal(covers[1], ref.grid[0, 2])
    np.testing.assert_array_equal(grid, ref.grid[0])
    for (xy, st), (d, a) in zip(agents, lifespans):
        np.testing.assert_array_equal(xy, ref.agent_indices[0])
        np.testing.assert_array_equal(st, ref.agent_states[0, :, 0])
        assert d == int(done_at[0])
        np.testing.assert_array_equal(a, ada[0, :, 0])


def _acts(policy, steps, n, seed):
    return np.random.RandomState(seed).randint(9, size=(steps, n)) if policy == "replay" else None


def _ref_run(ref, steps, policy, acts):
    return ref.run(steps, policy, actions=None if acts is None else acts[:, None, :])


# partial tiles 1, 63, 2, 8 and 13 columns wide; N mod 4 = 1, 3, 2, 0, 1
SIDES = (65, 127, 130, 200, 333)


@pytest.mark.parametrize("N", SIDES)
@pytest.mark.parametrize("policy,n", [("greedy", 300), ("antigreedy", 300), ("replay", 300), ("none", 300), ("greedy", 0)])
def test_single_band_any_side_matches_oracle(N, policy, n):
    """Agents packed around the (0, 0) corner: their moves wrap into the partial tile column and the partial tile row."""
    steps = 24
    light, dark, ai, st = make_state(N, n, seed=N + n, clustered=True)
    w = _world(N, n)
    w.load_state(light, dark, ai, st)
    ref = full_oracle(w, light, dark, ai, st)
    acts = _acts(policy, steps, n, 1)
    w.run(steps, policy, actions=acts, chunk=10)
    _, done_at, ada = _ref_run(ref, steps, policy, acts)
    assert w.step_count == steps and w.L == ref.L
    _check_exact(w.local_covers(), [w.agents()], [w.lifespans()], w.local_grid(), ref, done_at, ada)


def test_whole_life_at_side_65_phase_by_phase():
    """A garbage cell of the partial tiles in the per-step maxima would keep grid_done false and move done_at."""
    N, n = 65, 6
    light, dark, ai, st = make_state(N, n, seed=11, clustered=True)
    w = _world(N, n, ramp_period=96)
    w.albedo_light, w.albedo_dark, w.gamma = 0.7, 0.3, 0.3
    w.load_state(light, dark, ai, st)
    ref = full_oracle(w, light, dark, ai, st)
    steps, done_at, ada = ref.run(100000, "greedy", stop_all_done=True)
    for _ in range(steps):
        w.step("greedy")
    assert w.lifespans()[0] == int(done_at[0]) and w.first_done_step == steps
    _check_exact(w.local_covers(), [w.agents()], [w.lifespans()], w.local_grid(), ref, done_at, ada)


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


def _second_cluster(ai, worlds):
    """Half of the agents around the first interior band boundary (band 1's first row)."""
    n = ai.shape[0]
    ai[n // 2:, 0] = (ai[n // 2:, 0] + worlds[1].row0) % worlds[0].dim


@pytest.mark.parametrize("mode", ["nccl", "p2p"])
@pytest.mark.parametrize("N,bands,policy,n", [(200, 3, "greedy", 200), (333, 4, "antigreedy", 200), (200, 4, "replay", 200),
                                              (333, 4, "greedy", 600)])
def test_uneven_bands_on_one_gpu_match_oracle(mode, N, bands, policy, n):
    """Bands of 66/67/67, 83/83/83/84 and 50 rows (shorter than one tile); n > 256: several agent blocks."""
    import torch
    steps = 24
    worlds, streams = _bands(N, n, bands, mode)
    heights = [w.rows for w in worlds]
    assert sum(heights) == N and max(heights) - min(heights) <= 1
    light, dark, ai, st = make_state(N, n, seed=7 + N, clustered=True)
    _second_cluster(ai, worlds)
    ref = full_oracle(worlds[0], light, dark, ai, st)
    acts = _acts(policy, steps, n, 2)
    out = {}

    def go(w):
        with torch.cuda.stream(streams[w.rank]):
            w.load_state(light, dark, ai, st)
            w.run(steps, policy, actions=acts, chunk=8)
            out[w.rank] = (w.local_covers(), w.agents(), w.lifespans(), w.local_grid(),
                           w.band.peer_timed_out() if mode == "p2p" else False)

    run_threads(worlds, go)
    _, done_at, ada = _ref_run(ref, steps, policy, acts)
    assert not any(out[r][4] for r in range(bands)), "a peer barrier timed out"
    _check_exact(np.concatenate([out[r][0] for r in range(bands)], axis=1), [out[r][1] for r in range(bands)],
                 [out[r][2] for r in range(bands)], np.concatenate([out[r][3] for r in range(bands)], axis=1), ref, done_at, ada)


def test_device_reset_is_banding_invariant_at_side_333():
    N, n, steps = 333, 120, 20
    one = _world(N, n)
    one.reset_on_device(seed=3)
    one.run(steps, "greedy")
    worlds, _ = _bands(N, n, 3, "nccl")

    def go(w):
        w.reset_on_device(seed=3)
        w.run(steps, "greedy")

    run_threads(worlds, go)
    np.testing.assert_array_equal(np.concatenate([w.local_covers() for w in worlds], axis=1), one.local_covers())
    for w in worlds:
        np.testing.assert_array_equal(w.agents()[0], one.agents()[0])
        np.testing.assert_array_equal(w.agents()[1], one.agents()[1])
        np.testing.assert_array_equal(w.lifespans()[1], one.lifespans()[1])
    total = [sum(c) % (1 << 64) for c in zip(*[w.band.cover_checksum() for w in worlds])]
    assert total == one.cover_checksum()
    assert one.local_covers().max() > 0.05


@pytest.mark.parametrize("N", [130, 200])
@pytest.mark.parametrize("bands,mode", [(1, "local"), (3, "nccl"), (3, "p2p")])
def test_series_any_side_matches_oracle(N, bands, mode):
    """Series mode of the masked kernel: only the band's cells add to the temperature and cover sums."""
    import torch
    n, steps, policy = 40, 20, "greedy"
    light, dark, ai, st = make_state(N, n, seed=31 + N, clustered=True)
    ref = _oracle_series(N, light, dark, ai, st, steps, policy)
    if bands == 1:
        w = _world(N, n)
        w.load_state(light, dark, ai, st)
        series = [w.run_series(steps, policy, chunk=8)]
        covers = w.local_covers()
    else:
        worlds, streams = _bands(N, n, bands, mode)
        out = {}

        def go(w):
            with torch.cuda.stream(streams[w.rank]):
                w.load_state(light, dark, ai, st)
                out[w.rank] = (w.run_series(steps, policy, chunk=8), w.local_covers(),
                               w.band.peer_timed_out() if mode == "p2p" else False)

        run_threads(worlds, go)
        assert not any(out[r][2] for r in range(bands)), "a peer barrier timed out"
        series = [out[r][0] for r in range(bands)]
        covers = np.concatenate([out[r][1] for r in range(bands)], axis=1)
    for s in series:                                     # every rank returns the whole world's series
        assert s.shape == ref.shape
        np.testing.assert_array_equal(s[:, 1:], ref[:, 1:])
        np.testing.assert_allclose(s[:, 0], ref[:, 0], rtol=1e-9)
    cref = full_oracle(_world(N, n), light, dark, ai, st)
    cref.run(steps, policy)
    np.testing.assert_array_equal(covers[0], cref.grid[0, 1])
    np.testing.assert_array_equal(covers[1], cref.grid[0, 2])


def test_non_default_d4_physics_at_a_partial_tile():
    from kernel_sets import set_kernels
    N, n, steps = 130, 50, 30
    light, dark, ai, st = make_state(N, n, seed=5, clustered=True)
    w = _world(N, n)
    set_kernels(w, "d4_heavy")
    w.load_state(light, dark, ai, st)
    ref = full_oracle(w, light, dark, ai, st)
    w.run(steps, "greedy")
    _, done_at, ada = ref.run(steps, "greedy")
    _check_exact(w.local_covers(), [w.agents()], [w.lifespans()], w.local_grid(), ref, done_at, ada)
    assert w.band.slow_count() < 1e-3 * steps * N * N


def _stored(band):
    """The whole lattice buffer the last step wrote: [stored rows, pitch] int32, read through a view of library memory."""
    import torch
    rows = -(-band.rows // 64) * 64 + 2
    t = band._view(band._ptrs().recv_top, (rows, band.pitch), "<i4")
    torch.cuda.synchronize()
    return t.cpu().numpy().astype(np.int64)


def _check_storage(band, N, covers):
    """Ghost columns are copies of columns N-1 and 0, the band's cells are its covers, padding words and rows are 0."""
    lat = _stored(band)
    R = band.rows
    assert lat.shape[1] == -(-N // 64) * 64 + 8
    cells = lat[1:R + 1]
    np.testing.assert_array_equal(cells[:, 3], cells[:, N + 3])
    np.testing.assert_array_equal(cells[:, N + 4], cells[:, 4])
    np.testing.assert_array_equal((cells[:, 4:N + 4] & 0xffff) / 1000.0, covers[0])
    np.testing.assert_array_equal((cells[:, 4:N + 4] >> 16) / 1000.0, covers[1])
    assert not lat[:, 0:3].any() and not lat[:, N + 5:].any(), "a padding word was written"
    assert not lat[R + 2:].any(), "a padding row was written"
    return lat


@pytest.mark.parametrize("N", [65, 130, 333])
def test_storage_outside_the_band_is_untouched(N):
    """The masked kernel stores nothing outside the band: without a memory checker this is the out-of-bounds check, on
    both lattice buffers (odd and even step counts) of one band and of the bands of a 3-way split."""
    n = 40
    light, dark, ai, st = make_state(N, n, seed=N, clustered=True)
    w = _world(N, n)
    w.load_state(light, dark, ai, st)
    for steps in (5, 6):
        w.run(steps, "greedy")
        lat = _check_storage(w.band, N, w.local_covers())
        np.testing.assert_array_equal(lat[0], lat[N])        # one band: the ghost rows close the torus
        np.testing.assert_array_equal(lat[N + 1], lat[1])
    worlds, _ = _bands(N, n, 3, "nccl")

    def go(b):
        b.load_state(light, dark, ai, st)
        b.run(7, "greedy")

    run_threads(worlds, go)
    lats = [_check_storage(b.band, N, b.local_covers()) for b in worlds]
    for r, b in enumerate(worlds):                       # ghost rows hold the neighbours' edge rows, padding included
        up, down = lats[(r - 1) % 3], lats[(r + 1) % 3]
        np.testing.assert_array_equal(lats[r][0], up[worlds[(r - 1) % 3].rows])
        np.testing.assert_array_equal(lats[r][b.rows + 1], down[1])


def test_create_refuses_sides_below_64_and_bands_outside_8_to_n():
    from therldaisyworld_b200 import DaisyWorldError
    from therldaisyworld_b200.banded import DeviceBand
    p = _world(64, 0)                                    # carrier of the constants
    for N, row0, rows in ((63, 0, 63), (128, 0, 7), (128, 0, 129)):
        with pytest.raises(DaisyWorldError, match="dwt_create.*N >= 64 and 8 <= rows <= N"):
            DeviceBand(p, N, 0, row0, rows, 1)
    with pytest.raises(DaisyWorldError, match="dwt_create"):
        _world(100, 4, rank=0, world_size=16, comm=object())   # 6-row bands
