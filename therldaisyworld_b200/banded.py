"""A single giant toroidal RLDaisyWorld (BASELINE config 5), row-banded over the ranks of one node.

The world is ONE batch element of the reference environment (``daisy/daisy_world_rl.py``, ``batch_size == 1``) whose
grid does not fit in shared memory: rank r owns rows ``[floor(r*N/R), floor((r+1)*N/R))`` on its GPU (a ``dwt_handle`` of
``include/daisyworld_b200_tiled.h``) plus a ghost row above and below.  Agents are replicated on every rank.

One env step = the phase sequence of the header, with exactly these exchanges between ranks (``torch.distributed``:
NCCL over NVLink on GPUs, gloo in the CPU tests -- plumbing only, the data path is the CUDA kernels):

  * ONE SUM all-reduce per step over ``[gain(j-1) | act(j)]``: only the owner band of a cell knows what was eaten there,
    only the owner band of an agent sees its neighbourhood (greedy / anti-greedy).  Finishing step j-1 (state += gain,
    clip, lifespan counter) is deferred until the decisions of step j exist, so both vectors travel together;
  * after the edge tile rows of the stencil: the band's first/last row goes to the upper/lower neighbour's ghost row
    (ring, toroidal) on a side stream while the interior tile rows are still being computed;
  * per chunk of steps: MAX all-reduce of the per-step cover maxima (lifespan bookkeeping, ``grid_done``), and in
    ``run_series`` a SUM all-reduce of the per-step temperature and cover sums next to it;
  * ``observe()`` and every ``policy="mlp"`` step: a SUM all-reduce of the bands' partial observations ``[n, 7, 3, 3]``
    (the band that owns a window cell's row evaluates it, every other band contributes 0). An MLP step then decides on
    every rank from the same observation and needs no act exchange: two collectives per step (gain, obs);
  * the diagnostics (``diag_stats``, ``cover_stats``, ``image``): one SUM all-reduce per call of the bands' device-reduced
    parts, so every rank returns the same value.

``world_size == 1`` needs none of them (``dwt_halo_wrap`` closes the torus locally).

``mode="p2p"`` (GPUs of one node) takes the collectives off the step path altogether: the ranks map each other's
exchange vectors, barrier flags and lattice buffers through CUDA IPC once, and a step is ``dwt_step_p2p`` -- the owner of
an agent / the winner of a graze stores straight into every rank's exchange vector over NVLink, edge rows are pushed
into the neighbours' ghost rows, ranks meet at device-side flag barriers.  Only the per-chunk MAX all-reduce remains.
"""
import ctypes as C
import json
import os

import numpy as np

from . import _lib
from ._lib import DwClock, DwtPtrs, DW_DIAG, DW_POLICY, DWT_FIELD, DWT_REP
from .env import RLDaisyWorld, make_clock_struct, make_config_struct, set_default_attributes, set_default_kernels

_WORLD_POLICIES = ("greedy", "antigreedy", "eps_greedy")      # decisions that (may) read the grid: need the act exchange


def band_rows(N, world_size, rank):
    """Rows [lo, hi) of rank's band; N must split into equal multiples of 64."""
    if N % (64 * world_size):
        raise ValueError(f"N={N} must be a multiple of 64*world_size={64 * world_size}")
    R = N // world_size
    return rank * R, (rank + 1) * R


def balanced_rows(N, world_size, rank):
    """Rows [lo, hi) of rank's band in the partition BandedDaisyWorld uses: [floor(rank*N/world_size),
    floor((rank+1)*N/world_size)), so that bands differ by at most one row. Equals band_rows wherever that succeeds."""
    if not 0 <= rank < world_size:
        raise ValueError(f"rank {rank} outside 0..{world_size - 1}")
    return rank * N // world_size, (rank + 1) * N // world_size


# ---- snapshots (BandedDaisyWorld.save / restore)
SNAPSHOT_FORMAT = 1
_REP_NAME = {v: k for k, v in DWT_REP.items()}
# the constants a snapshot carries: RLDaisyWorld's configuration plus the other dw_config scalars, and the arrays
_SNAPSHOT_CONSTANTS = RLDaisyWorld._CONFIG_KEYS + ("q", "q2", "dt", "ddL", "ramp_up_down")
_SNAPSHOT_ARRAYS = ("daisy_kernel", "local_albedo_kernel", "adjacent_albedo_kernel", "neighborhood")
_CLOCK_KEYS = ("L", "dL", "min_L", "max_L", "ddL", "step_count", "ramp_period", "ramp_up_down")


def _rep_layout(rep, rows, N):
    """(shape, dtype) of `rows` rows of a state in representation rep (a DWT_REP value); (None, None) for none."""
    if rep == DWT_REP["lattice"]:
        return (rows, N), np.uint32
    if rep == DWT_REP["planes"]:
        return (2, rows, N), np.float64
    return None, None


def shard_name(which, lo, hi):
    """File of a snapshot shard: the rows [lo, hi) of the current state ("cur") or pre-state ("pre")."""
    return f"{which}.rows-{lo:07d}-{hi:07d}.npy"


def shard_pieces(ranges, N, first, count):
    """[(k, a, b)]: world rows first .. first + count - 1 (toroidal), in order, as row slices [a, b) of the shards whose
    global rows are ranges[k] = (lo, hi). The ranges must tile [0, N)."""
    cover = sorted(ranges)
    if not cover or cover[0][0] != 0 or cover[-1][1] != N or any(p[1] != q[0] for p, q in zip(cover, cover[1:])):
        raise ValueError(f"the shards {cover} do not tile the rows 0..{N - 1}")
    out, g, left = [], first % N, count
    while left:
        k = next(k for k, (lo, hi) in enumerate(ranges) if lo <= g < hi)
        lo, hi = ranges[k]
        take = min(hi - g, left)
        out.append((k, g - lo, g - lo + take))
        g, left = (g + take) % N, left - take
    return out


class DistComm:
    """The three exchanges of a banded step over torch.distributed (NCCL on GPUs, gloo on CPU)."""

    def __init__(self, rank, world_size, group=None):
        import torch.distributed as dist
        self.dist, self.rank, self.world_size, self.group = dist, int(rank), int(world_size), group

    def all_reduce_sum(self, t):
        self.dist.all_reduce(t, op=self.dist.ReduceOp.SUM, group=self.group)

    def all_reduce_max(self, t):
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX, group=self.group)

    def exchange_halos(self, send_top, send_bottom, recv_top, recv_bottom):
        dist = self.dist
        up, down = (self.rank - 1) % self.world_size, (self.rank + 1) % self.world_size
        if self.group is not None:
            up, down = dist.get_global_rank(self.group, up), dist.get_global_rank(self.group, down)
        # tag 0: downward message (my last row -> lower neighbour's top ghost); tag 1: upward. Posting order matters for
        # NCCL when up == down (two ranks): the first send pairs with the peer's first receive.
        ops = [dist.P2POp(dist.isend, send_bottom, down, group=self.group, tag=0),
               dist.P2POp(dist.isend, send_top, up, group=self.group, tag=1),
               dist.P2POp(dist.irecv, recv_top, up, group=self.group, tag=0),
               dist.P2POp(dist.irecv, recv_bottom, down, group=self.group, tag=1)]
        for req in dist.batch_isend_irecv(ops):
            req.wait()


class _DevArray:
    """Minimal __cuda_array_interface__ carrier so torch can view library-owned device memory without a copy."""

    def __init__(self, ptr, shape, typestr):
        self.__cuda_array_interface__ = {"shape": tuple(shape), "typestr": typestr, "data": (int(ptr), False), "version": 2}


class DeviceBand:
    """One rank's band on its GPU (ctypes over the dwt_* C-ABI)."""

    def __init__(self, params, N, n_agents, row0, rows, n_ranks, device=0):
        import torch
        self._torch = torch
        self._lib = _lib.load()
        self.N, self.n, self.row0, self.rows, self.n_ranks, self.device = int(N), int(n_agents), int(row0), int(rows), int(n_ranks), int(device)
        cfg = make_config_struct(params, 1, N, n_agents, device)
        h = C.c_void_p()
        rc = self._lib.dwt_create(C.byref(cfg), self.rows, self.row0, self.n_ranks, C.byref(h))
        if rc != 0:
            msg = self._lib.dwt_last_error(None)
            raise _lib.DaisyWorldError(f"dwt_create failed (code {rc}): {msg.decode() if msg else ''}")
        self._h = h
        p = C.c_int32(0)
        self._check(self._lib.dwt_get_pitch(self._h, C.byref(p)), "dwt_get_pitch")
        self.pitch = int(p.value)          # words per stored row (whole tiles plus the ghost columns)
        self._views = {}
        self._side = None

    def __del__(self):
        try:
            if getattr(self, "_h", None):
                self._lib.dwt_destroy(self._h)
                self._h = None
        except Exception:
            pass

    def _check(self, rc, what):
        _lib.check_tiled(self._lib, self._h, rc, what)

    # ---- state
    def set_params(self, params):
        cfg = make_config_struct(params, 1, self.N, self.n, self.device)
        self._check(self._lib.dwt_set_config(self._h, C.byref(cfg)), "dwt_set_config")

    def set_clock(self, clk):
        self._check(self._lib.dwt_set_clock(self._h, C.byref(clk)), "dwt_set_clock")

    def set_epsilon(self, epsilon):
        self._check(self._lib.dwt_set_epsilon(self._h, float(epsilon)), "dwt_set_epsilon")

    def get_clock(self):
        clk = DwClock()
        self._check(self._lib.dwt_get_clock(self._h, C.byref(clk)), "dwt_get_clock")
        return clk

    def upload(self, light_rows, dark_rows, agent_indices, agent_states):
        """light_rows/dark_rows: [rows + 2, N] (band with its ghost rows); agents: all n, global coordinates."""
        pd = C.POINTER(C.c_double)
        l = np.ascontiguousarray(light_rows, dtype=np.float64)
        d = np.ascontiguousarray(dark_rows, dtype=np.float64)
        assert l.shape == d.shape == (self.rows + 2, self.N)
        self._check(self._lib.dwt_upload_covers(self._h, l.ctypes.data_as(pd), d.ctypes.data_as(pd)), "dwt_upload_covers")
        if self.n:
            ai = np.ascontiguousarray(agent_indices, dtype=np.int64).reshape(self.n, 2)
            st = np.ascontiguousarray(agent_states, dtype=np.float64).reshape(self.n)
            self._check(self._lib.dwt_upload_agents(self._h, ai.ctypes.data_as(C.POINTER(C.c_int64)), st.ctypes.data_as(pd)),
                        "dwt_upload_agents")
        self._views = {}

    def init_random(self, seed, params):
        self._check(self._lib.dwt_init_random(self._h, C.c_uint64(seed), params.light_proportion, params.dark_proportion,
                                              params.initial_al, params.initial_ad), "dwt_init_random")
        self._views = {}

    def set_agents(self, agent_indices, agent_states):
        """all n agents, global coordinates (dwt_upload_agents); the covers are left alone"""
        if self.n:
            ai = np.ascontiguousarray(agent_indices, dtype=np.int64).reshape(self.n, 2)
            st = np.ascontiguousarray(agent_states, dtype=np.float64).reshape(self.n)
            self._check(self._lib.dwt_upload_agents(self._h, ai.ctypes.data_as(C.POINTER(C.c_int64)),
                                                    st.ctypes.data_as(C.POINTER(C.c_double))), "dwt_upload_agents")

    # ---- snapshots (dwt_save_state / dwt_restore_state)
    def save_state(self, alloc=None):
        """(meta, cur, pre, agents_done_at): the band's own rows of its current state and of its pre-state in their
        representation -- lattice: uint32 [rows, N] packed words, planes: float64 [2, rows, N] --, pre None when there is
        no pre-state; meta {cur_rep, pre_rep, L_last, done_at} with DWT_REP names. alloc(which, shape, dtype) ("cur" /
        "pre") supplies the arrays to fill, e.g. memory maps of the files they go to; default np.empty."""
        alloc = alloc or (lambda which, shape, dtype: np.empty(shape, dtype=dtype))
        m = _lib.DwtBandState()
        self._check(self._lib.dwt_save_state(self._h, C.byref(m), None, None, None), "dwt_save_state")
        arrays = {}
        for which, rep in (("cur", m.cur_rep), ("pre", m.pre_rep)):
            shape, dtype = _rep_layout(rep, self.rows, self.N)
            arrays[which] = alloc(which, shape, dtype) if shape else None
        ada = np.zeros(max(self.n, 1), dtype=np.int64)
        ptr = lambda a: None if a is None else a.ctypes.data
        self._check(self._lib.dwt_save_state(self._h, C.byref(m), ptr(arrays["cur"]), ptr(arrays["pre"]),
                                             ada.ctypes.data_as(C.POINTER(C.c_int64))), "dwt_save_state")
        meta = dict(cur_rep=_REP_NAME[m.cur_rep], pre_rep=_REP_NAME[m.pre_rep], L_last=m.L_last, done_at=int(m.done_at))
        return meta, arrays["cur"], arrays["pre"], ada[:self.n]

    def restore_state(self, meta, cur_rows, pre_rows, agents_done_at):
        """Replace the band's state (dwt_restore_state): cur_rows / pre_rows hold the band's rows WITH both ghost rows
        (rows + 2), in the layout save_state returns; meta as save_state returns it."""
        m = _lib.DwtBandState(cur_rep=DWT_REP[meta["cur_rep"]], pre_rep=DWT_REP[meta["pre_rep"]], L_last=float(meta["L_last"]),
                              done_at=int(meta["done_at"]))
        keep = []

        def ptr(a, rep):
            shape, dtype = _rep_layout(DWT_REP.get(rep, -1), self.rows + 2, self.N)
            if a is None or not shape:
                return None
            a = np.ascontiguousarray(a, dtype=dtype)
            assert a.shape == shape, (a.shape, shape)
            keep.append(a)
            return a.ctypes.data

        ada = np.ascontiguousarray(agents_done_at, dtype=np.int64).reshape(self.n) if self.n else np.zeros(1, dtype=np.int64)
        self._check(self._lib.dwt_restore_state(self._h, C.byref(m), ptr(cur_rows, meta["cur_rep"]), ptr(pre_rows, meta["pre_rep"]),
                                                ada.ctypes.data_as(C.POINTER(C.c_int64))), "dwt_restore_state")

    def pre_checksum(self):
        out = (C.c_uint64 * 4)()
        self._check(self._lib.dwt_pre_checksum(self._h, out), "dwt_pre_checksum")
        return [int(v) for v in out]

    # ---- phases
    def _replay_ptr(self, policy, actions, K=None):
        """The host int8 actions of a replay as dwt_decide / dwt_step_p2p ([n]) or dwt_run (K steps: [K, n]) take them;
        None for every other policy."""
        if policy != "replay":
            return None
        if K is None:
            a = np.asarray(actions).reshape(self.n)
        else:
            a = np.asarray(actions).reshape(-1, self.n)[:K]
            assert a.shape[0] == K
        return np.ascontiguousarray(a, dtype=np.int8).ctypes.data_as(C.POINTER(C.c_int8))

    def decide(self, policy, actions_step=None, seed=0):
        self._check(self._lib.dwt_decide(self._h, DW_POLICY[policy], self._replay_ptr(policy, actions_step), C.c_uint64(seed)),
                    "dwt_decide")

    def move_graze(self):
        self._check(self._lib.dwt_move_graze(self._h), "dwt_move_graze")

    def observe(self):
        """The band's partial observation of the current state into the device buffer (dwt_observe)."""
        self._check(self._lib.dwt_observe(self._h), "dwt_observe")

    def obs_tensor(self):
        """The device observation buffer [n, 7, 3, 3] as a torch view (summed over the ranks in place by the caller)."""
        p = C.c_void_p()
        self._check(self._lib.dwt_get_obs_ptr(self._h, C.byref(p)), "dwt_get_obs_ptr")
        return self._view(p.value, (max(self.n, 1), 7, 3, 3), "<f8")[:self.n]

    def get_obs(self):
        out = np.zeros((self.n, 7, 3, 3))
        self._check(self._lib.dwt_get_obs(self._h, out.ctypes.data_as(C.POINTER(C.c_double))), "dwt_get_obs")
        return out

    def set_mlp(self, params):
        p = np.ascontiguousarray(params, dtype=np.float64).ravel()
        self._check(self._lib.dwt_set_mlp(self._h, p.ctypes.data_as(C.POINTER(C.c_double)), int(p.size)), "dwt_set_mlp")

    def finish_agents(self):
        self._check(self._lib.dwt_finish_agents(self._h), "dwt_finish_agents")

    def stencil(self, part=0):
        self._check(self._lib.dwt_stencil(self._h, int(part)), "dwt_stencil")

    def halo_wrap(self):
        self._check(self._lib.dwt_halo_wrap(self._h), "dwt_halo_wrap")

    def stencil_and_exchange(self, comm):
        """Edge tile rows, then the halo exchange on a side stream overlapped with the interior tile rows."""
        torch = self._torch
        if self._side is None:
            self._side = torch.cuda.Stream(device=self.device)
            self._edge_done = torch.cuda.Event()
        self.stencil(1)
        main = torch.cuda.current_stream(self.device)
        self._edge_done.record(main)
        with torch.cuda.stream(self._side):
            self._side.wait_event(self._edge_done)
            comm.exchange_halos(*self.halo_tensors())
        self.stencil(2)
        main.wait_stream(self._side)

    # ---- peer-memory mode
    def set_stream(self, cuda_stream):
        self._check(self._lib.dwt_set_stream(self._h, C.c_void_p(int(cuda_stream))), "dwt_set_stream")

    def ipc_export(self):
        buf = C.create_string_buffer(4 * 64)
        self._check(self._lib.dwt_ipc_export(self._h, buf), "dwt_ipc_export")
        return bytes(buf.raw)

    def set_peer_rows(self, rows):
        """Band heights of all ranks in rank order (dwt_set_peer_rows); default: BandedDaisyWorld's balanced partition."""
        if rows is None:
            rows = [hi - lo for lo, hi in (balanced_rows(self.N, self.n_ranks, r) for r in range(self.n_ranks))]
        arr = (C.c_int32 * len(rows))(*[int(r) for r in rows])
        self._check(self._lib.dwt_set_peer_rows(self._h, len(rows), arr), "dwt_set_peer_rows")

    def ipc_attach(self, rank, blobs, peer_rows=None):
        self.set_peer_rows(peer_rows)
        blob = b"".join(blobs)
        self._check(self._lib.dwt_ipc_attach(self._h, int(rank), len(blobs), C.create_string_buffer(blob, len(blob))), "dwt_ipc_attach")

    def peer_buffers(self):
        out = (C.c_void_p * 4)()
        self._check(self._lib.dwt_get_peer_buffers(self._h, out), "dwt_get_peer_buffers")
        return [int(v or 0) for v in out]

    def attach_peers(self, rank, tables, peer_rows=None):
        """Same-process peers: tables[r] = peer_buffers() of rank r."""
        self.set_peer_rows(peer_rows)
        flat = (C.c_void_p * (4 * len(tables)))(*[p for t in tables for p in t])
        self._check(self._lib.dwt_attach_peers(self._h, int(rank), len(tables), flat), "dwt_attach_peers")

    def step_p2p(self, policy, actions_step=None, seed=0):
        self._check(self._lib.dwt_step_p2p(self._h, DW_POLICY[policy], self._replay_ptr(policy, actions_step), C.c_uint64(seed)),
                    "dwt_step_p2p")

    def flush_p2p(self):
        self._check(self._lib.dwt_flush_p2p(self._h), "dwt_flush_p2p")

    def cover_checksum(self):
        out = (C.c_uint64 * 4)()
        self._check(self._lib.dwt_cover_checksum(self._h, out), "dwt_cover_checksum")
        return [int(v) for v in out]

    def time_stencil(self, reps=20):
        us = C.c_double(0.0)
        self._check(self._lib.dwt_debug_time_stencil(self._h, int(reps), C.byref(us)), "dwt_debug_time_stencil")
        return us.value

    def peer_timed_out(self):
        v = C.c_int32(0)
        self._check(self._lib.dwt_peer_status(self._h, C.byref(v)), "dwt_peer_status")
        return bool(v.value)

    def run_local(self, K, policy, actions=None, seed=0):
        """K steps without any exchange (a band that is the whole torus)."""
        self._check(self._lib.dwt_run(self._h, int(K), DW_POLICY[policy], self._replay_ptr(policy, actions, K), C.c_uint64(seed)),
                    "dwt_run")

    def set_series(self, on):
        """Series mode: every step also sums sqrt(g)*T and the new milli-covers of the band's cells (dwt_set_series)."""
        self._check(self._lib.dwt_set_series(self._h, 1 if on else 0), "dwt_set_series")

    def take_series(self, K):
        """[K, 3] of the open chunk: sum of T (kelvin), sum of milli-light, sum of milli-dark (after any all-reduce of
        series_tensor)."""
        out = np.zeros((int(K), 3))
        self._check(self._lib.dwt_get_series(self._h, int(K), out.ctypes.data_as(C.POINTER(C.c_double))), "dwt_get_series")
        return out

    def end_chunk(self, K):
        first = C.c_int32(-1)
        self._check(self._lib.dwt_end_chunk(self._h, int(K), C.byref(first)), "dwt_end_chunk")
        return int(first.value)

    # ---- exchange buffers as torch CUDA tensors (zero-copy views of library memory)
    def _ptrs(self):
        p = DwtPtrs()
        self._check(self._lib.dwt_get_ptrs(self._h, C.byref(p)), "dwt_get_ptrs")
        return p

    def _view(self, ptr, shape, typestr):
        key = (int(ptr), tuple(shape), typestr)
        t = self._views.get(key)
        if t is None:
            t = self._torch.as_tensor(_DevArray(ptr, shape, typestr), device=f"cuda:{self.device}")
            self._views[key] = t
        return t

    def exch_tensor(self, gain=True, act=True):
        """The exchange vector [gain[n] | act[n]] (or one half of it) as a torch view."""
        t = self._view(self._ptrs().gain, (2 * max(self.n, 1),), "<f8")
        return t[(0 if gain else self.n):(2 * self.n if act else self.n)]

    def stepmax_tensor(self, K):
        return self._view(self._ptrs().stepmax, (4096 * 2,), "<i4")[:2 * K]

    def series_tensor(self, K):
        """The first K rows of the device series buffer [4096, 3] (partial sums of this band, additive over bands)."""
        p = C.c_void_p()
        self._check(self._lib.dwt_get_series_ptr(self._h, C.byref(p)), "dwt_get_series_ptr")
        return self._view(p.value, (4096, 3), "<f8")[:K]

    def halo_tensors(self):
        """(send_top, send_bottom, recv_top, recv_bottom): whole stored rows (pitch words, ghost columns and padding
        included) of the lattice buffer the current step writes, as int32 views."""
        p = self._ptrs()
        return tuple(self._view(q, (self.pitch,), "<i4") for q in (p.send_top, p.send_bottom, p.recv_top, p.recv_bottom))

    # ---- getters
    def reset_lifespans(self):
        self._check(self._lib.dwt_reset_lifespans(self._h), "dwt_reset_lifespans")

    def lifespans(self):
        done_at = C.c_int64(0)
        ada = np.zeros((self.n,), dtype=np.int64)
        self._check(self._lib.dwt_get_lifespans(self._h, C.byref(done_at), ada.ctypes.data_as(C.POINTER(C.c_int64))), "dwt_get_lifespans")
        return int(done_at.value), ada

    def agents(self):
        ai = np.zeros((self.n, 2), dtype=np.int64)
        st = np.zeros((self.n,), dtype=np.float64)
        if self.n:
            self._check(self._lib.dwt_get_agents(self._h, ai.ctypes.data_as(C.POINTER(C.c_int64)), st.ctypes.data_as(C.POINTER(C.c_double))),
                        "dwt_get_agents")
        return ai, st

    def covers(self):
        out = np.empty((2, self.rows, self.N))
        pd = C.POINTER(C.c_double)
        self._check(self._lib.dwt_get_covers(self._h, out[0].ctypes.data_as(pd), out[1].ctypes.data_as(pd)), "dwt_get_covers")
        return out

    def grid(self):
        out = np.empty((7, self.rows, self.N))
        self._check(self._lib.dwt_get_grid(self._h, out.ctypes.data_as(C.POINTER(C.c_double))), "dwt_get_grid")
        return out

    # ---- fp32 mode (dwt_grid_f32 .. dwt_f32_stats)
    def grid_f32(self):
        """The band's grid [7, rows, N] as float32 (dwt_get_grid_f32): channels 0, 1, 2, 6 and the agent stamp the binary32
        roundings of grid()'s, temperatures evaluated with fp32 arithmetic (within 1e-5 relative)."""
        out = np.empty((7, self.rows, self.N), dtype=np.float32)
        self._check(self._lib.dwt_get_grid_f32(self._h, out.ctypes.data_as(C.POINTER(C.c_float))), "dwt_get_grid_f32")
        return out

    def grid_f32_tensor(self):
        """Launch the fp32 materialisation (dwt_grid_f32, on the handle's stream) and return the device buffer [7, rows, N]
        as a torch view; the next call overwrites it."""
        self._check(self._lib.dwt_grid_f32(self._h), "dwt_grid_f32")
        p = C.c_void_p()
        self._check(self._lib.dwt_get_grid_f32_ptr(self._h, C.byref(p)), "dwt_get_grid_f32_ptr")
        return self._view(p.value, (7, self.rows, self.N), "<f4")

    def f32_stats(self):
        """Tier counters of the fp32 materialisation: cells evaluated with fp32 arithmetic, cells whose bare fraction went on
        to the fp64 tier, cells that needed the literal cell (cumulative)."""
        out = (C.c_uint64 * 3)()
        self._check(self._lib.dwt_f32_stats(self._h, out), "dwt_f32_stats")
        return {"cells": int(out[0]), "fp64_tier": int(out[1]), "literal": int(out[2])}

    def time_materialise(self, fp32, reps=10):
        """Device microseconds per materialisation (dwt_debug_time_materialise): fp32 mode, or the fp64 grid without its
        download."""
        us = C.c_double(0.0)
        self._check(self._lib.dwt_debug_time_materialise(self._h, 1 if fp32 else 0, int(reps), C.byref(us)),
                    "dwt_debug_time_materialise")
        return us.value

    # ---- diagnostics and plot feed (the unrounded fields of the last forward; dwt_get_diag .. dwt_pool)
    def diag(self, name):
        """The band's field `name` (a DW_DIAG key) of the last forward: [rows, N], growth [2, rows, N] (dl, dd)."""
        out = np.empty((2, self.rows, self.N) if name == "growth" else (self.rows, self.N))
        self._check(self._lib.dwt_get_diag(self._h, DW_DIAG[name], out.ctypes.data_as(C.POINTER(C.c_double))), "dwt_get_diag")
        return out

    def diag_stats(self, name):
        """[count, mean, m2, min, max] of the field over the band's own cells, m2 about the band's mean."""
        out = np.zeros(5)
        self._check(self._lib.dwt_get_diag_stats(self._h, DW_DIAG[name], out.ctypes.data_as(C.POINTER(C.c_double))),
                    "dwt_get_diag_stats")
        return out

    def cover_stats(self):
        """[sum light, sum dark, max light, max dark] over the band's own cells of the current state."""
        out = np.zeros(4)
        self._check(self._lib.dwt_get_cover_stats(self._h, out.ctypes.data_as(C.POINTER(C.c_double))), "dwt_get_cover_stats")
        return out

    def pool(self, field, block):
        """Launch the block sums [H, H] of a DWT_FIELD field over the band's own cells (dwt_pool) and return the device
        buffer as a torch view (summed over the ranks in place by the caller)."""
        self._check(self._lib.dwt_pool(self._h, DWT_FIELD[field], int(block)), "dwt_pool")
        p, H = C.c_void_p(), C.c_int32(0)
        self._check(self._lib.dwt_get_pool_ptr(self._h, C.byref(p), C.byref(H)), "dwt_get_pool_ptr")
        return self._view(p.value, (H.value, H.value), "<f8")

    def get_pool(self):
        p, H = C.c_void_p(), C.c_int32(0)
        self._check(self._lib.dwt_get_pool_ptr(self._h, C.byref(p), C.byref(H)), "dwt_get_pool_ptr")
        out = np.zeros((H.value, H.value))
        self._check(self._lib.dwt_get_pool(self._h, out.ctypes.data_as(C.POINTER(C.c_double))), "dwt_get_pool")
        return out

    def last_L(self):
        L = C.c_double(0.0)
        self._check(self._lib.dwt_get_last_L(self._h, C.byref(L)), "dwt_get_last_L")
        return L.value

    def slow_count(self):
        c = C.c_uint64(0)
        self._check(self._lib.dwt_debug_slow_count(self._h, C.byref(c)), "dwt_debug_slow_count")
        return int(c.value)

    def synchronize(self):
        self._check(self._lib.dwt_synchronize(self._h), "dwt_synchronize")


class BandedDaisyWorld:
    """Host-side driver of one giant world over `world_size` bands.

    Carries the reference's public constants as attributes (same names as RLDaisyWorld; mutate them before reset()).
    `band_factory(params, N, n_agents, row0, rows, n_ranks)` builds this rank's band: DeviceBand on a GPU (default), an
    oracle-backed stand-in in the CPU tests."""

    def __init__(self, grid_dimension, n_agents, rank=0, world_size=1, group=None, device=0, band_factory=None, comm=None,
                 mode="nccl", **kwargs):
        set_default_attributes(self, grid_dimension=grid_dimension, n_agents=n_agents, **kwargs)
        set_default_kernels(self)
        self.batch_size = 1
        self.rank, self.world_size, self.device = int(rank), int(world_size), int(device)
        self.comm = comm if (comm is not None or self.world_size == 1) else DistComm(rank, world_size, group)
        self.row0, hi = balanced_rows(self.dim, self.world_size, self.rank)
        self.rows = hi - self.row0
        factory = band_factory or (lambda p, N, n, r0, R, nr: DeviceBand(p, N, n, r0, R, nr, device=self.device))
        self.band = factory(self, self.dim, self.n_agents, self.row0, self.rows, self.world_size)
        self.L = self.min_L
        self.dL = (self.max_L - self.min_L) / self.ramp_period
        self.step_count = 0
        self._pending = 0          # steps recorded since the last end_chunk
        self._gain_pending = False # multi-rank: gains of the last step not yet summed / applied
        self.first_done_step = None
        self._series = None        # run_series: [k, 3] sums of the chunks closed so far
        self.mode = mode if self.world_size > 1 else "local"
        if self.mode == "p2p" and comm is None:
            # one-off exchange of the CUDA IPC handles (any transport would do; torch.distributed is at hand)
            blobs = [None] * self.world_size
            self.comm.dist.all_gather_object(blobs, self.band.ipc_export(), group=group)
            self.band.ipc_attach(self.rank, blobs)

    # ---- reset
    def _reset_clock(self):
        self.L = self.min_L
        self.dL = (self.max_L - self.min_L) / self.ramp_period
        self.step_count = 0
        self.band.set_params(self)
        self.band.set_clock(make_clock_struct(self))
        self.band.reset_lifespans()
        self._pending = 0
        self._gain_pending = False
        self.first_done_step = None

    def load_state(self, light, dark, agent_indices, agent_states):
        """reset() from explicit GLOBAL arrays: light/dark [N,N] (may be off the 0.001 lattice), agents [n,2], [n]."""
        self._reset_clock()
        N = self.dim
        rows = np.arange(self.row0 - 1, self.row0 + self.rows + 1) % N
        self.band.upload(np.asarray(light)[rows], np.asarray(dark)[rows], agent_indices, agent_states)

    def reset_on_device(self, seed=0):
        """reset() with the state drawn on the device (same distribution as the reference, counter RNG keyed by the
        global cell index: identical for every banding)."""
        self._reset_clock()
        self.band.init_random(seed, self)

    def set_mlp(self, params):
        """MLP.set_parameters (daisy/agents/mlp.py) for policy="mlp": 1808 weights, flat layout of MLP.get_parameters."""
        self.band.set_mlp(params)

    # ---- snapshots: the whole world's state to a directory and back, exactly, on any banding
    def _sum_u64(self, words):
        """The sum over the ranks of each 64-bit word, mod 2^64, on every rank: one _table of 16-bit limbs (exact in fp64)."""
        limbs = [(int(w) >> (16 * j)) & 0xffff for w in words for j in range(4)]
        tot = self._table(limbs).sum(axis=0)
        return [sum(int(tot[4 * i + j]) << (16 * j) for j in range(4)) & ((1 << 64) - 1) for i in range(len(words))]

    def _band_checksums(self, cur_rep, pre_rep):
        """this band's dwt_cover_checksum of the current state and of the pre-state (zeros where not on the lattice)"""
        cur = self.band.cover_checksum() if cur_rep == "lattice" else [0] * 4
        pre = self.band.pre_checksum() if pre_rep == "lattice" else [0] * 4
        return cur + pre

    def save(self, path):
        """Write the world's state to the directory `path`, exactly: every rank its own rows of the current state and the
        pre-state (cur.rows-<lo>-<hi>.npy, pre.rows-...), rank 0 world.json (clock, counters, constants, checksums) and
        agents.npz. Collective when world_size > 1: every rank calls it. MLP weights and eps_greedy's epsilon are policy
        parameters, not world state, and are not saved. restore() takes the snapshot back on any banding of a world with the
        same N and n."""
        self.end_chunk()                             # pending gains applied, lifespans folded: the state of a whole step
        b = self.band
        lo, hi = self.row0, self.row0 + self.rows
        os.makedirs(path, exist_ok=True)
        meta, cur, pre, ada = b.save_state()
        # np.save of an array in memory: writing through a memory map of the file was measured slower (tools/tiled_bench.py)
        for which, a in (("cur", cur), ("pre", pre)):
            if a is not None:
                np.save(os.path.join(path, shard_name(which, lo, hi)), a)
        sums = self._sum_u64(self._band_checksums(meta["cur_rep"], meta["pre_rep"]))
        # (peer-memory mode: that collective also keeps the next step's halo push off the pre-state until every rank read it)
        if self.rank == 0:
            ai, st = b.agents()
            np.savez(os.path.join(path, "agents.npz"), indices=ai, states=st, agents_done_at=ada)
            clk = b.get_clock()
            world = dict(format=SNAPSHOT_FORMAT, N=self.dim, n_agents=self.n_agents,
                         writer=dict(world_size=self.world_size, mode=self.mode,
                                     rows=[list(balanced_rows(self.dim, self.world_size, r)) for r in range(self.world_size)]),
                         cur_rep=meta["cur_rep"], pre_rep=meta["pre_rep"], clock={k: getattr(clk, k) for k in _CLOCK_KEYS},
                         step_count=self.step_count, first_done_step=self.first_done_step, L_last=meta["L_last"],
                         done_at=meta["done_at"], cover_checksum=sums[:4] if meta["cur_rep"] == "lattice" else None,
                         pre_checksum=sums[4:] if meta["pre_rep"] == "lattice" else None,
                         constants={k: np.asarray(getattr(self, k)).item() for k in _SNAPSHOT_CONSTANTS},
                         arrays={k: np.asarray(getattr(self, k)).tolist() for k in _SNAPSHOT_ARRAYS})
            with open(os.path.join(path, "world.json"), "w") as f:
                json.dump(world, f, indent=1)
        if self.comm is not None:
            self._table([0.0])                       # the snapshot is whole on disk once save() returns on any rank

    @staticmethod
    def read_snapshot_meta(path):
        with open(os.path.join(path, "world.json")) as f:
            return json.load(f)

    def _snapshot_rows(self, path, world, which):
        """This band's rows with both ghost rows (rows + 2, toroidal) of the snapshot's current state or pre-state, gathered
        from whichever shards hold them; None when the snapshot has no such state."""
        rep = world[f"{which}_rep"]
        if rep == "none":
            return None
        ranges = [tuple(r) for r in world["writer"]["rows"]]
        shards = [np.load(os.path.join(path, shard_name(which, lo, hi)), mmap_mode="r") for lo, hi in ranges]
        shape, _ = _rep_layout(DWT_REP[rep], None, self.dim)
        for (lo, hi), s in zip(ranges, shards):
            want = tuple(hi - lo if d is None else d for d in shape)
            if s.shape != want:
                raise ValueError(f"snapshot shard {shard_name(which, lo, hi)} has shape {s.shape}, expected {want}")
        axis = 0 if rep == "lattice" else 1
        parts = [shards[k][a:b] if axis == 0 else shards[k][:, a:b]
                 for k, a, b in shard_pieces(ranges, self.dim, self.row0 - 1, self.rows + 2)]
        return np.concatenate(parts, axis=axis)

    def restore(self, path):
        """Replace the world's whole state by the snapshot in `path` (save()): covers, pre-state, agents, clock, lifespan
        counters and constants. Works on any world_size and mode with the same N and n; refuses another N, n or format
        before touching the device. Nothing of the world's earlier history remains, so one snapshot can be restored many
        times into the same world (branching). Verifies the whole-world checksums of the lattice states and raises
        DaisyWorldError on a mismatch (a corrupted shard, or shards of two saves). Collective when world_size > 1."""
        world = self.read_snapshot_meta(path)
        if world.get("format") != SNAPSHOT_FORMAT:
            raise ValueError(f"snapshot format {world.get('format')!r}, this version reads {SNAPSHOT_FORMAT}")
        if (world["N"], world["n_agents"]) != (self.dim, self.n_agents):
            raise ValueError(f"snapshot of N={world['N']}, n={world['n_agents']} does not fit this world (N={self.dim}, "
                             f"n={self.n_agents})")
        cur, pre = self._snapshot_rows(path, world, "cur"), self._snapshot_rows(path, world, "pre")
        with np.load(os.path.join(path, "agents.npz")) as z:
            ai, st, ada = z["indices"], z["states"], z["agents_done_at"]
        self._flush()
        if self.mode == "p2p":
            self._table([0.0])                       # no neighbour's last halo push may still land in this band's ghost rows
        for k, v in world["constants"].items():
            setattr(self, k, v)
        for k, v in world["arrays"].items():
            setattr(self, k, np.array(v, dtype=np.float64))
        self.band.set_params(self)
        self.band.restore_state(dict(cur_rep=world["cur_rep"], pre_rep=world["pre_rep"], L_last=world["L_last"],
                                     done_at=world["done_at"]), cur, pre, ada)
        self.band.set_agents(ai, st)
        for k, v in world["clock"].items():
            setattr(self, k, v)
        self.band.set_clock(make_clock_struct(self))
        self.step_count, self.first_done_step = world["step_count"], world["first_done_step"]
        self._pending, self._gain_pending = 0, False
        # also the closing collective: no rank steps while a neighbour still writes its rows
        sums = self._sum_u64(self._band_checksums(world["cur_rep"], world["pre_rep"]))
        for name, got in (("cover_checksum", sums[:4]), ("pre_checksum", sums[4:])):
            if world[name] is not None and got != world[name]:
                raise _lib.DaisyWorldError(f"restore({path!r}): the {name} of the restored world {got} differs from the snapshot's "
                                           f"{world[name]} (a corrupted shard, or shards of two saves); restore or reset again")

    # ---- stepping
    def step(self, policy="greedy", actions_step=None, seed=0):
        """One env step with a device policy ("greedy", "antigreedy", "eps_greedy", "random", "none", "mlp") or "replay"
        of actions_step [n]. "mlp" is not available in p2p mode (raises before the step)."""
        b, comm = self.band, self.comm
        if self.mode == "p2p":
            b.step_p2p(policy, actions_step, seed)
            self._gain_pending = bool(self.n_agents)
            self._pending += 1
            return
        if policy == "mlp":
            self._observe_device()                   # finishes step j-1 first; every rank then decides on the same obs
        b.decide(policy, actions_step, seed)
        if comm is None:
            b.move_graze()
            b.finish_agents()
            b.stencil(0)
            b.halo_wrap()
        else:
            need_act = bool(self.n_agents) and policy in _WORLD_POLICIES
            if self._gain_pending or need_act:
                comm.all_reduce_sum(b.exch_tensor(gain=self._gain_pending, act=need_act))
            if self._gain_pending:
                b.finish_agents()                    # step j-1, before its gz flags are overwritten
            b.move_graze()
            self._gain_pending = bool(self.n_agents)
            if hasattr(b, "stencil_and_exchange"):
                b.stencil_and_exchange(comm)
            else:
                b.stencil(0)
                comm.exchange_halos(*b.halo_tensors())
        self._pending += 1

    def _check_peers(self):
        """Peer-memory mode: a device-side flag barrier gives up after a bounded spin (csrc/dw_tiled.cuh, ~4 s or
        DW_PEER_TIMEOUT_MS) and the step then continues on stale ghost rows / exchange vectors. Every point where results
        leave the device goes through here, so a stalled peer raises instead of yielding silently wrong grids and lifespans."""
        if self.mode == "p2p" and self.band.peer_timed_out():
            raise _lib.DaisyWorldError(f"rank {self.rank}: a peer-memory barrier timed out (a peer rank stalled or died); the state of "
                                  "this world is not trustworthy -- reset() before continuing")

    def _flush(self):
        """Finish the last step's agents (multi-rank: the deferred gain all-reduce)."""
        if self._gain_pending:
            if self.mode == "p2p":
                self.band.flush_p2p()
                self._check_peers()
            else:
                self.comm.all_reduce_sum(self.band.exch_tensor(gain=True, act=False))
                self.band.finish_agents()
            self._gain_pending = False

    def _observe_device(self):
        """The whole observation of the current state in the band's device buffer, on every rank: the agents' states must
        be final (the stamp of ch4), then the partial observations are summed over the ranks."""
        self._flush()
        self.band.observe()
        if self.comm is not None:
            # p2p mode: the pre-state's ghost rows read here are overwritten by the neighbours' halo push of the NEXT step;
            # this all-reduce completes on every rank only after every rank's observation, and before any of them can
            # issue that step
            self.comm.all_reduce_sum(self.band.obs_tensor())

    def observe(self):
        """obs[1, n, 7, 3, 3] of the current state: what the reference's step() returned for it (the 3x3 windows around
        the agents, all channels, times the neighbourhood mask), or after a reset its observation of the reset state.
        Every rank returns the same array."""
        if not self.n_agents:
            return np.zeros((1, 0, 7, 3, 3))
        self._observe_device()
        obs = self.band.get_obs()[None]
        self._check_peers()
        return obs

    def env_step(self, action=None):
        """The reference's step(action) for batch 1: (obs [1, n, 7, 3, 3], reward, done, {}). action: n integers 0..8 as
        [n], [1, n] or [1, n, 1]; None is the reference's all-zero action. reward / done are [1, n, 1] (the agents' states,
        state < 0.1), or with no agents [1, 2] (any light / dark cover left, and its negation)."""
        n = self.n_agents
        if action is not None:
            a = np.asarray(action)
            if a.shape not in ((n,), (1, n), (1, n, 1)) or (a.size and not np.issubdtype(a.dtype, np.integer)):
                raise ValueError(f"action must be n={n} integers as [n], [1, n] or [1, n, 1]; got shape {a.shape}, dtype {a.dtype}")
            if a.size and (a.min() < 0 or a.max() > 8):
                raise ValueError("actions must be in 0..8")
            self.step("replay", a.reshape(n))
        else:
            self.step("none")
        obs = self.observe()
        if n:
            reward = self.band.agents()[1].reshape(1, n, 1).copy()
            reward = reward * (reward > 0)
        else:
            cs = self.cover_checksum()
            reward = np.array([[cs[0] > 0, cs[1] > 0]])
        return obs, reward, reward < 0.1, {}

    def end_chunk(self):
        """Fold the per-step cover maxima of the steps since the last call into the lifespan counter."""
        self._flush()
        K = self._pending
        if K == 0:
            return
        if self.comm is not None:
            self.comm.all_reduce_max(self.band.stepmax_tensor(K))
        if self._series is not None:
            if self.comm is not None:
                self.comm.all_reduce_sum(self.band.series_tensor(K))
            self._series.append(self.band.take_series(K))
        first = self.band.end_chunk(K)
        self._check_peers()
        if first >= 0 and self.first_done_step is None:
            self.first_done_step = self.step_count + first + 1      # 1-based count of steps at which grid_done first held
        self.step_count += K
        self._pending = 0
        clk = self.band.get_clock()
        self.L, self.dL, self.min_L, self.max_L = clk.L, clk.dL, clk.min_L, clk.max_L

    def run(self, K, policy="greedy", actions=None, seed=0, chunk=256):
        """K env steps. actions: [K, n] ints 0..8 for policy='replay'. Lifespan counters are folded every `chunk` steps."""
        if self.world_size == 1 and hasattr(self.band, "run_local"):
            done = 0
            while done < K:
                k = min(chunk, K - done)
                self.band.run_local(k, policy, None if actions is None else np.asarray(actions)[done:done + k], seed)
                self._pending += k
                self.end_chunk()
                done += k
            return K
        for j in range(K):
            self.step(policy, None if actions is None else np.asarray(actions)[j], seed)
            if self._pending >= chunk:
                self.end_chunk()
        self.end_chunk()
        return K

    def run_series(self, K, policy="greedy", actions=None, seed=0, chunk=256):
        """run() that also returns the per-step means of the whole world [K, 3] = (global mean temperature of that step's
        forward -- env.temp.mean() of the reference --, mean light cover, mean dark cover after the step), the layout of
        RLDaisyWorld.run_series. Reduced inside the stencil kernels (series mode) and summed over the ranks once per chunk;
        every rank returns the same array. Needs g > 0."""
        self.end_chunk()
        self.band.set_series(True)
        self._series = []
        try:
            self.run(K, policy, actions=actions, seed=seed, chunk=chunk)
            sums = np.concatenate(self._series) if self._series else np.zeros((0, 3))
        finally:
            self._series = None
            if self._pending == 0:
                self.band.set_series(False)
        cells = float(self.dim) * self.dim
        return sums / np.array([cells, 1000.0 * cells, 1000.0 * cells])

    # ---- results
    def lifespans(self):
        """(done_at, agents_done_at[n]) -- the notebook counters (greedy_longevity_abatement.ipynb cell 2)."""
        self.end_chunk()
        return self.band.lifespans()

    def agents(self):
        self._flush()
        return self.band.agents()

    def cover_checksum(self):
        """Exact position-weighted checksum of the WHOLE world's covers (this rank's part summed over the ranks mod 2^64):
        identical for every banding of the same world (dwt_cover_checksum)."""
        self._flush()
        cs = self.band.cover_checksum()
        if self.comm is not None and hasattr(self.comm, "dist"):
            # int64 all-reduce wraps mod 2^64 like the device sums; the four words travel as signed values
            import torch
            t = torch.tensor([c - (1 << 64) if c >= (1 << 63) else c for c in cs], dtype=torch.int64, device=f"cuda:{self.device}")
            self.comm.dist.all_reduce(t, group=self.comm.group)
            cs = [int(v) & ((1 << 64) - 1) for v in t.tolist()]
        return cs

    def local_covers(self):
        """[2, rows, N]: light and dark cover of this rank's band."""
        return self.band.covers()

    def local_grid(self):
        """[7, rows, N]: env.grid[0] restricted to this rank's rows."""
        self._flush()
        return self.band.grid()

    # ---- fp32 mode: the grid of local_grid() as float32, evaluated with fp32 arithmetic from the lattice
    def _fenced(self, fn):
        """fn() on the band after the last step's agents are finished; in peer-memory mode followed by the fence that keeps
        every rank's next step (its halo push into the pre-state this reads) behind every rank's call, as local_diag."""
        self._flush()
        out = fn()
        if self.mode == "p2p":
            self.band.synchronize()                  # the pre-state is read before this rank meets the others
            self._table([0.0])
        self._check_peers()
        return out

    def local_grid_f32(self):
        """[7, rows, N] float32: local_grid() in fp32 mode. Channels 0, 1, 2, 6 and the agent stamp on channel 4 equal
        local_grid().astype(np.float32); the temperatures are evaluated with fp32 arithmetic, within 1e-5 relative. Half the
        download of local_grid() and no fp64 scratch on the device. In peer-memory mode every rank must call it."""
        return self._fenced(self.band.grid_f32)

    def local_grid_f32_tensor(self):
        """local_grid_f32() as a torch.float32 CUDA tensor [7, rows, N] on the band's device, without leaving the device (the
        materialisation is complete when it returns). It aliases library memory: the next local_grid_f32() or
        local_grid_f32_tensor() overwrites it -- clone() what must outlive that. In peer-memory mode every rank must call it."""
        def grid():
            t = self.band.grid_f32_tensor()
            self.band.synchronize()
            return t
        return self._fenced(grid)

    def f32_stats(self):
        """Tier counters of fp32 mode summed over the ranks: {cells, fp64_tier, literal} (see DeviceBand.f32_stats).
        Collective when world_size > 1."""
        self._flush()
        s = self.band.f32_stats()
        tot = self._sum_u64([s["cells"], s["fp64_tier"], s["literal"]])
        self._check_peers()
        return dict(cells=tot[0], fp64_tier=tot[1], literal=tot[2])

    # ---- diagnostics and plot feed (DESIGN.md §0 row (f) N3): what the reference's notebook helpers read from
    # RLDaisyWorld (notebook_helpers.py:45-57,139-150,210-223), reduced on the device per band and merged over the ranks.
    # The fields are the unrounded side effects of the last step's forward, like RLDaisyWorld.temp / .growth.
    # Every call is collective when world_size > 1 (every rank calls it) and returns the same value on every rank.
    def _table(self, row):
        """Every rank's row of a [world_size, k] table, in rank order: one SUM all-reduce of a table in which each rank
        fills its own row (x + 0 is exact, so every rank gets every row's bits). In peer-memory mode it is also what keeps
        the next step's halo push off the pre-state until every rank has read it (see _observe_device)."""
        row = np.asarray(row, dtype=np.float64)
        if self.comm is None:
            return row[None]
        t = self.band.exch_tensor(gain=True, act=False).new_zeros((self.world_size, row.size))
        t[self.rank] = t.new_tensor(row)
        self.comm.all_reduce_sum(t)
        return t.cpu().numpy()

    @staticmethod
    def _merge_stats(rows):
        """Chan's pairwise merge of [count, mean, m2, min, max] rows, in row order -> (count, mean, m2, min, max)."""
        n, mean, m2 = rows[0, :3]
        for c, mu, q in rows[1:, :3]:
            tot = n + c
            d = mu - mean
            mean = mean + d * (c / tot)
            m2 = m2 + q + d * d * (n * c / tot)
            n = tot
        return n, mean, m2, rows[:, 3].min(), rows[:, 4].max()

    def local_diag(self, name):
        """[rows, N] ([2, rows, N] for growth): this rank's rows of the unrounded field `name` (temp, temp_light, temp_dark,
        temp_effective, beta, beta_l, beta_d, growth) of the last step's forward. In peer-memory mode every rank must call it."""
        if name not in DW_DIAG:
            raise ValueError(f"unknown diagnostic field {name!r}; one of {sorted(DW_DIAG)}")
        self._flush()
        out = self.band.diag(name)
        if self.mode == "p2p":
            self._table([0.0])                       # fence: no rank's next step before every rank has read its pre-state
        self._check_peers()
        return out

    def diag_stats(self, name):
        """{mean, std, min, max} of a diagnostic field over the whole world (growth: both planes), std the population std
        like np.std -- RLDaisyWorld.diag_stats for the giant world."""
        if name not in DW_DIAG:
            raise ValueError(f"unknown diagnostic field {name!r}; one of {sorted(DW_DIAG)}")
        self._flush()
        n, mean, m2, mn, mx = self._merge_stats(self._table(self.band.diag_stats(name)))
        self._check_peers()
        return dict(mean=mean, std=float(np.sqrt(m2 / n)), min=mn, max=mx)

    def cover_stats(self):
        """Mean and max light / dark cover of the current state over the whole world (RLDaisyWorld.cover_stats)."""
        self._flush()
        rows = self._table(self.band.cover_stats())
        self._check_peers()
        cells = float(self.dim) * self.dim
        return dict(mean_light=rows[:, 0].sum() / cells, mean_dark=rows[:, 1].sum() / cells, max_light=rows[:, 2].max(),
                    max_dark=rows[:, 3].max())

    def image(self, field, block=16):
        """[H, H] block means of a field over the whole world, H = ceil(N / block): block (i, j) averages rows and columns
        [i*block, min((i+1)*block, N)) x [j*block, ...) (edge blocks are smaller when block does not divide N). field: a
        diagnostic (growth gives [2, H, H]; growth_l / growth_d one plane) or a grid channel as local_grid() holds it --
        grid_bare, grid_light, grid_dark, grid_temp, grid_temp_dark (channels 0, 1, 2, 3, 5). Only the image leaves the
        device."""
        if field == "growth":
            return np.stack([self.image("growth_l", block), self.image("growth_d", block)])
        if field not in DWT_FIELD:
            raise ValueError(f"unknown image field {field!r}; one of {sorted(DWT_FIELD) + ['growth']}")
        self._flush()
        t = self.band.pool(field, block)
        self.band.synchronize()                      # the block sums exist (and the pre-state is read) before any exchange
        if self.comm is not None:
            self.comm.all_reduce_sum(t)
        sums = t.cpu().numpy()
        self._check_peers()
        H = sums.shape[0]
        edge = np.minimum(np.arange(1, H + 1) * int(block), self.dim) - np.arange(H) * int(block)
        return sums / np.outer(edge, edge)

    @property
    def dead_temp(self):
        """reference :406-407,416 -- bare-planet temperature at the L of the last forward, as RLDaisyWorld.dead_temp."""
        L = self.band.last_L()
        return np.array([((self.S * L * (1 - self.albedo_bare)) / self.sigma) ** (1 / 4)])

    def run_with_series(self, K, every=16, policy="greedy", seed=0, images=(), block=16):
        """K steps in chunks of `every`, recording after each chunk what the reference's plot helpers read
        (notebook_helpers.py:45-57), as RLDaisyWorld.run_with_series: step, L, temp_mean, temp_std, dead_temp, light,
        dark; plus images = {field: image(field, block)} for the requested fields."""
        series = []
        done = 0
        while done < K:
            k = min(every, K - done)
            self.run(k, policy=policy, seed=seed)
            done += k
            t, c = self.diag_stats("temp"), self.cover_stats()
            series.append(dict(step=self.step_count, L=self.L, temp_mean=t["mean"], temp_std=t["std"], dead_temp=float(self.dead_temp[0]),
                               light=c["mean_light"], dark=c["mean_dark"], images={f: self.image(f, block) for f in images}))
        return series
