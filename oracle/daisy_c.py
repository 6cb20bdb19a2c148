"""ctypes front for the C oracle (oracle/daisy_oracle.c) -- TEST INFRASTRUCTURE ONLY.

Same role and restrictions as oracle/daisy_numpy.py; exists because the NumPy oracle is too slow
for BASELINE-sized parity runs (1000 worlds x 64x64 x ~480 steps)."""
import ctypes as C
import os

import numpy as np

from .build_oracle import build
from .daisy_numpy import daisy_weights, neighborhood_mask


class Params(C.Structure):
    _fields_ = [("B", C.c_int32), ("N", C.c_int32), ("n_agents", C.c_int32), ("ch", C.c_int32)] + \
               [(k, C.c_double) for k in ("p", "g", "S", "sigma", "gamma", "q", "q2", "temp_optimal", "dt",
                                          "agent_gamma", "albedo_bare", "albedo_light", "albedo_dark")] + \
               [("mask", C.c_double * 9), ("w", C.c_double * 9), ("adj", C.c_double * 9)]


class Clock(C.Structure):
    _fields_ = [(k, C.c_double) for k in ("L", "dL", "min_L", "max_L", "ddL")] + \
               [("step_count", C.c_int64), ("ramp_period", C.c_int64), ("ramp_up_down", C.c_int32), ("pad", C.c_int32)]


_lib = None


def lib():
    global _lib
    if _lib is None:
        _lib = C.CDLL(build())
        assert _lib.dwo_sizeof_params() == C.sizeof(Params)
        assert _lib.dwo_sizeof_clock() == C.sizeof(Clock)
        _lib.dwo_run.restype = C.c_int64
    return _lib


def _p(a, t):
    return None if a is None else a.ctypes.data_as(C.POINTER(t))


class COracleWorld:
    """State container + step functions; parameters are taken from any env-like object
    (oracle.daisy_numpy.OracleDaisyWorld, or the product's RLDaisyWorld) by attribute name."""

    def __init__(self, env, grid=None, agent_indices=None, agent_states=None):
        g = env.grid if grid is None else grid
        self.grid = np.ascontiguousarray(g, dtype=np.float64).copy()
        B, ch, N, _ = self.grid.shape
        ai = env.agent_indices if agent_indices is None else agent_indices
        st = env.agent_states if agent_states is None else agent_states
        self.agent_indices = np.ascontiguousarray(ai, dtype=np.int64).copy()
        self.agent_states = np.ascontiguousarray(st, dtype=np.float64).copy()
        n = self.agent_indices.shape[1]
        self.P = Params(B=B, N=N, n_agents=n, ch=7, p=env.p, g=env.g, S=env.S, sigma=env.sigma, gamma=env.gamma,
                        q=env.q, q2=env.q2, temp_optimal=env.temp_optimal, dt=env.dt, agent_gamma=env.agent_gamma,
                        albedo_bare=env.albedo_bare, albedo_light=env.albedo_light, albedo_dark=env.albedo_dark)
        mask = getattr(env, "neighborhood", neighborhood_mask(1, "von_neumann"))
        w = getattr(env, "daisy_kernel", daisy_weights())
        adj = getattr(env, "adjacent_albedo_kernel", None)
        if adj is None:
            adj = np.full((3, 3), 0.125)
            adj[1, 1] = 0.0
        self.P.mask[:] = list(np.asarray(mask, dtype=np.float64).ravel())
        self.P.w[:] = list(np.asarray(w, dtype=np.float64).ravel())
        self.P.adj[:] = list(np.asarray(adj, dtype=np.float64).ravel())
        self.clk = Clock(L=env.L, dL=env.dL, min_L=env.min_L, max_L=env.max_L, ddL=env.ddL,
                         step_count=env.step_count, ramp_period=env.ramp_period,
                         ramp_up_down=int(bool(env.ramp_up_down)))
        self.B, self.N, self.n = B, N, n
        self._scratch = np.empty_like(self.grid)

    @property
    def L(self):
        return self.clk.L

    @property
    def step_count(self):
        return self.clk.step_count

    def get_obs(self):
        obs = np.zeros((self.B, self.n, 7, 3, 3))
        if self.n:
            lib().dwo_get_obs(C.byref(self.P), _p(self.grid, C.c_double), _p(self.agent_indices, C.c_int64),
                              _p(obs, C.c_double))
        return obs

    def forward_diag(self):
        """Unrounded fields of a forward pass at the current state: [B,9,N,N]
        (T, Tl, Td, Te, beta, beta_l, beta_d, dl, dd).  Does not advance the state."""
        diag = np.zeros((self.B, 9, self.N, self.N))
        g = self.grid.copy()
        lib().dwo_forward(C.byref(self.P), C.c_double(self.clk.L), _p(g, C.c_double),
                          _p(self.agent_indices, C.c_int64), _p(self.agent_states, C.c_double),
                          _p(self._scratch, C.c_double), _p(diag, C.c_double))
        return diag

    def step(self, action=None):
        n = self.n
        obs = np.zeros((self.B, n, 7, 3, 3))
        if n:
            reward = np.zeros((self.B, n, 1)); done = np.zeros((self.B, n, 1), dtype=np.uint8)
        else:
            reward = np.zeros((self.B, 2)); done = np.zeros((self.B, 2), dtype=np.uint8)
        ab = am = 0
        a = None
        if action is not None:
            a = np.ascontiguousarray(np.asarray(action)[..., 0], dtype=np.int64)
            ab, am = a.shape
        lib().dwo_step(C.byref(self.P), C.byref(self.clk), _p(self.grid, C.c_double), _p(self._scratch, C.c_double),
                       _p(self.agent_indices, C.c_int64), _p(self.agent_states, C.c_double), _p(a, C.c_int64),
                       ab, am, _p(obs, C.c_double), _p(reward, C.c_double), _p(done, C.c_uint8))
        if n == 0:
            reward = reward.astype(bool)
        return obs, reward, done.astype(bool), {}

    def run(self, K, policy="greedy", actions=None, stop_all_done=False):
        """K fused steps with an in-oracle policy; returns (steps_run, done_at[B], agents_done_at[B,n,1])."""
        code = {"none": 0, "greedy": 1, "antigreedy": 2, "replay": 3}[policy]
        done_at = np.zeros((self.B,), dtype=np.int64)
        agents_done_at = np.zeros((self.B, self.n, 1), dtype=np.int64)
        a = None
        if actions is not None:
            a = np.ascontiguousarray(np.asarray(actions).reshape(-1, self.B, self.n), dtype=np.int64)
            assert a.shape[0] >= K
        steps = lib().dwo_run(C.byref(self.P), C.byref(self.clk), _p(self.grid, C.c_double),
                              _p(self.agent_indices, C.c_int64), _p(self.agent_states, C.c_double), code,
                              _p(a, C.c_int64), C.c_int64(K), int(stop_all_done), _p(done_at, C.c_int64),
                              _p(agents_done_at, C.c_int64))
        return int(steps), done_at, agents_done_at
