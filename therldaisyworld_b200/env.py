"""Drop-in ``RLDaisyWorld`` whose simulation step runs on a B200 through the C-ABI.

Mirrors the Python surface of the reference class (``daisy/daisy_world_rl.py:13-501``): same constructor
kwargs, same mutable public attributes, same ``reset/step/forward/get_obs/update_agents/update_L``
signatures, array shapes and dtypes, same use of the process-global legacy ``np.random`` stream at
construction and ``reset()``.  Reference callers (``daisy/agents/greedy.py``, ``daisy/agents/mlp.py``,
``daisy/evo/sges.py``, the notebooks) keep working unchanged.

State lives on the device.  ``env.grid``, ``env.agent_indices``, ``env.agent_states`` are host mirrors:
reading one downloads it lazily; assigning one (or mutating the array you were handed) is detected and
uploaded before the next device operation.

Additions that the reference does not have (they do not change any reference behaviour):
``run(K, policy=...)`` / ``simulate_lifespan(policy=...)`` -- the fused multi-step path with an on-device
policy and the notebook's lifespan counters.
"""
import ctypes as C
import json
import os
import weakref

import numpy as np
import numpy.random as npr

from . import _lib
from ._lib import DwClock, DwConfig, DwRunResult, DW_DIAG, DW_E_UNSUPPORTED, DW_POLICY


def query_kwargs(key, default, **kwargs):
    """reference: daisy/helpers.py:3-8"""
    return kwargs[key] if key in kwargs else default


def make_neighborhood(radius=1, mode="moore"):
    """Observation masks (reference: daisy/nn/functional.py:51-103)."""
    ax = np.arange(-radius, radius + 1)
    xx, yy = np.meshgrid(ax, ax)
    if mode == "moore":
        rr = np.maximum(np.abs(xx), np.abs(yy))
    elif mode == "circular":
        rr = np.abs(np.sqrt(xx ** 2 + yy ** 2))
    else:
        if mode != "von_neumann":
            print(f"neighborhood mode {mode} not recognized, using von Neumann default")
        rr = np.abs(xx) + np.abs(yy)
    out = np.zeros((2 * radius + 1, 2 * radius + 1))
    out[rr <= radius] = 1.0
    return out


def canonical_actions8(actions):
    """int8 action codes for the device from ANY integers, read like the reference reads them (daisy_world_rl.py:190-212:
    a == 8 stays, else a % 4 moves (Python modulo), a > 4 grazes): 0..8 as they are, a > 8 -> 12 + a % 4, a < 0 -> a % 4."""
    a = np.asarray(actions).astype(np.int64, copy=False)
    return np.where((a >= 0) & (a <= 8), a, np.where(a > 8, 12 + a % 4, a % 4)).astype(np.int8)


def _ptr(a, ctype):
    return None if a is None else a.ctypes.data_as(C.POINTER(ctype))


def set_default_attributes(obj, **kwargs):
    """Constants and kwargs of RLDaisyWorld.__init__ (reference :15-79); shared with banded.BandedDaisyWorld."""
    self = obj
    self.ch = 7
    self.batch_size = 32                      # ctor kwarg is ignored like the reference (:20)
    self.kr = query_kwargs("kr", 1, **kwargs)
    self.neighborhood_mode = query_kwargs("neighborhood_mode", "von_neumann", **kwargs)
    self.neighborhood = make_neighborhood(self.kr, self.neighborhood_mode)
    self.dim = kwargs["grid_dimension"] if "grid_dimension" in kwargs else 16

    self.p = 1.00
    self.g = 0.003265
    self.S = 1000.0
    self.sigma = 5.67e-8
    self.gamma = 0.25
    self.q = 0.2 * self.S / self.sigma
    self.use_microclimate = True
    self.collision_mode = query_kwargs("collision_mode", 0, **kwargs)
    self.q2 = self.q / 8.0 if self.use_microclimate else 0.0
    self.Toptim = 295.5
    self.dt = 1.0
    self.ddL = 0.0
    self.agent_gamma = 0.05
    self.max_L = 1.5
    self.min_L = 0.75
    self.initial_L = self.min_L
    self.ramp_period = kwargs["ramp_period"] if "ramp_period" in kwargs else 512
    self.ramp_up_down = False
    self.albedo_bare = 0.5
    self.albedo_light = 0.75
    self.albedo_dark = 0.25
    self.temp_optimal = 295.5
    self.food_chain_penalty = 0.5
    self.initial_al = 0.2
    self.initial_ad = 0.2
    self.light_proportion = 0.33
    self.dark_proportion = 0.33
    self.n_agents = query_kwargs("n_agents", 4, **kwargs)


def set_default_kernels(obj):
    """initialize_neighborhood (reference :265-283): daisy-spread and albedo kernels."""
    obj.n_daisies = 2
    obj.daisy_kernel = np.ones((1, 1, 3, 3)) * np.exp(-1)
    obj.daisy_kernel[:, :, 1, 1] = 1.0
    obj.daisy_kernel[:, :, 0::2, 0::2] = np.exp(-2)
    obj.daisy_kernel /= obj.daisy_kernel.sum()
    obj.local_albedo_kernel = np.zeros((1, 1, 3, 3))
    obj.local_albedo_kernel[:, :, 1, 1] = 1.0
    obj.adjacent_albedo_kernel = np.ones((1, 1, 3, 3)) / 8.0
    obj.adjacent_albedo_kernel[:, :, 1, 1] = 0.0


def shared_cell_offsets(agent_indices, N):
    """collision_mode == 1 bookkeeping (reference :220-242): the reference draws one npr.rand(1, n, 1) per cell that holds
    more than one agent, world after world. Returns int32 offsets [B+1]: offsets[b] = number of such cells in worlds < b
    (so offsets[-1] draws are needed in total). Integer work on the post-move positions only."""
    pos = np.asarray(agent_indices)
    B, n = pos.shape[:2]
    offsets = np.zeros(B + 1, dtype=np.int32)
    if n > 1:
        key = np.sort(pos[:, :, 0] * N + pos[:, :, 1], axis=1)                 # [B, n]
        same = key[:, 1:] == key[:, :-1]
        # a shared cell = a run of equal keys: count the runs' first repeats
        first_repeat = same & ~np.concatenate([np.zeros((B, 1), dtype=bool), same[:, :-1]], axis=1)
        np.cumsum(first_repeat.sum(axis=1), out=offsets[1:])
    return offsets


def make_config_struct(obj, batch, dim, n_agents, device):
    """dw_config from the public attributes of an environment object."""
    c = DwConfig(batch=int(batch), dim=int(dim), n_agents=int(n_agents), device=int(device),
                 p=obj.p, g=obj.g, S=obj.S, sigma=obj.sigma, gamma=obj.gamma, q=obj.q, q2=obj.q2,
                 temp_optimal=obj.temp_optimal, dt=obj.dt, agent_gamma=obj.agent_gamma,
                 albedo_bare=obj.albedo_bare, albedo_light=obj.albedo_light, albedo_dark=obj.albedo_dark)
    c.daisy_kernel[:] = [float(v) for v in np.asarray(obj.daisy_kernel, dtype=np.float64).ravel()]
    c.adjacent_kernel[:] = [float(v) for v in np.asarray(obj.adjacent_albedo_kernel, dtype=np.float64).ravel()]
    mask = np.asarray(obj.neighborhood, dtype=np.float64)
    if mask.shape != (3, 3):
        raise ValueError("get_obs gathers a 3-wide window (reference :257-258): only kr=1 neighbourhoods work")
    c.obs_mask[:] = [float(v) for v in mask.ravel()]
    return c


def make_clock_struct(obj):
    return DwClock(L=float(obj.L), dL=float(obj.dL), min_L=float(obj.min_L), max_L=float(obj.max_L),
                   ddL=float(obj.ddL), step_count=int(obj.step_count), ramp_period=int(obj.ramp_period),
                   ramp_up_down=int(bool(obj.ramp_up_down)))


class _PinnedPool:
    """Page-locked host blocks for the packed outputs of step() (dw_step_packed): the device->host copy is then one DMA at
    PCIe rate straight into the arrays the caller receives. step() must return FRESH arrays like the reference, so a block
    goes back to the pool only when every array carved from it has been garbage-collected (weakref.finalize on the ctypes
    buffer that is their common base). Callers that keep every observation would pin memory without bound: beyond
    MAX_LIVE blocks in flight the outputs fall back to ordinary (pageable) memory."""
    MAX_LIVE = 16

    def __init__(self, lib):
        self._lib = lib
        self._free = {}         # nbytes -> [address]
        self._live = 0

    def take(self, nbytes):
        """A writable ctypes byte buffer of nbytes in page-locked memory, or None when too many are still referenced."""
        free = self._free.setdefault(nbytes, [])
        if free:
            addr = free.pop()
        else:
            if self._live >= self.MAX_LIVE:
                return None
            p = C.c_void_p()
            if self._lib.dw_host_alloc(C.c_uint64(nbytes), C.byref(p)) != 0 or not p.value:
                return None
            addr = p.value
        self._live += 1
        buf = (C.c_ubyte * nbytes).from_address(addr)
        fin = weakref.finalize(buf, self._give_back, nbytes, addr)
        fin.atexit = False
        return buf

    def _give_back(self, nbytes, addr):
        self._live -= 1
        self._free.setdefault(nbytes, []).append(addr)

    def drain(self):
        for lst in self._free.values():
            for addr in lst:
                self._lib.dw_host_free(C.c_void_p(addr))
        self._free = {}


# attributes whose assignment has to reach the device before the next device operation (dw_set_config / dw_set_clock)
_CFG_ATTRS = frozenset(("p", "g", "S", "sigma", "gamma", "q", "q2", "temp_optimal", "dt", "agent_gamma", "albedo_bare", "albedo_light",
                        "albedo_dark", "daisy_kernel", "adjacent_albedo_kernel", "neighborhood"))
_CLK_ATTRS = frozenset(("L", "dL", "min_L", "max_L", "ddL", "step_count", "ramp_period", "ramp_up_down"))


class _Mirror:
    """Host mirror of one device array with write detection."""
    __slots__ = ("pristine", "handed", "assigned")

    def __init__(self):
        self.pristine = None   # private copy of what the device holds (None = not downloaded)
        self.handed = None     # the array the user holds (may have been mutated)
        self.assigned = False  # user assigned a brand-new array

    def invalidate(self):
        self.pristine = None
        self.handed = None
        self.assigned = False

    def dirty(self):
        if self.assigned:
            return True
        if self.handed is None or self.pristine is None:
            return False
        return not (self.handed.shape == self.pristine.shape and np.array_equal(self.handed, self.pristine))


class RLDaisyWorld:
    _DIAG_ATTRS = ("temp", "temp_light", "temp_dark", "temp_effective", "beta", "beta_l", "beta_d", "growth")

    def __setattr__(self, name, value):
        # the constants and the luminosity clock are plain mutable attributes like the reference's; assigning one marks the
        # device copy stale (pushed by the next device operation) instead of re-sending everything on every step
        if name in _CFG_ATTRS:
            self.__dict__["_cfg_dirty"] = True
        elif name in _CLK_ATTRS:
            self.__dict__["_clk_dirty"] = True
        object.__setattr__(self, name, value)

    def __init__(self, **kwargs):
        self._cfg_dirty = self._clk_dirty = True
        self._arr_sig = None
        set_default_attributes(self, **kwargs)

        # additions (not in the reference)
        self.device = int(kwargs.get("device", os.environ.get("LOCAL_RANK", 0)))
        self._lib = _lib.load()
        self._h = None
        self._shape = None
        self._m = {"grid": _Mirror(), "agent_indices": _Mirror(), "agent_states": _Mirror()}
        self._diag_cache = {}
        self._dead_L = None
        self._pool = _PinnedPool(self._lib)
        self._layout = None

        self.initialize_neighborhood()
        self.initialize_agents()
        self.reset()

    # ------------------------------------------------------------------ handle / plumbing
    def __del__(self):
        try:
            if getattr(self, "_h", None):
                self._lib.dw_destroy(self._h)
                self._h = None
            if getattr(self, "_pool", None):
                self._pool.drain()
        except Exception:
            pass

    def _check(self, rc, what):
        _lib.check(self._lib, self._h, rc, what)

    def _config(self):
        return make_config_struct(self, self.batch_size, self.dim, self.n_agents, self.device)

    def _clock(self):
        return DwClock(L=float(self.L), dL=float(self.dL), min_L=float(self.min_L), max_L=float(self.max_L),
                       ddL=float(self.ddL), step_count=int(self.step_count), ramp_period=int(self.ramp_period),
                       ramp_up_down=int(bool(self.ramp_up_down)))

    def _adopt_clock(self, clk):
        """Mirror the clock the device has advanced (no dirty mark: host and device agree)."""
        self.__dict__.update(L=clk.L, dL=clk.dL, min_L=clk.min_L, max_L=clk.max_L, step_count=int(clk.step_count))

    def _pull_clock(self):
        clk = DwClock()
        self._check(self._lib.dw_get_clock(self._h, C.byref(clk)), "dw_get_clock")
        self._adopt_clock(clk)

    def _ensure_handle(self, shape):
        """(Re)create the device handle when batch_size / dim / n_agents changed (they are re-read at reset())."""
        if self._h is not None and self._shape == shape:
            return
        if self._h is not None:
            self._lib.dw_destroy(self._h)
            self._h = None
        saved = (self.batch_size, self.dim, self.n_agents)
        self.batch_size, self.dim, self.n_agents = shape
        cfg = self._config()
        self.batch_size, self.dim, self.n_agents = saved
        h = C.c_void_p()
        rc = self._lib.dw_create(C.byref(cfg), C.byref(h))
        if rc != 0:
            msg = self._lib.dw_last_error(None)
            raise _lib.DaisyWorldError(f"dw_create failed (code {rc}): {msg.decode() if msg else ''}")
        self._h = h
        self._shape = shape
        self._cfg_dirty = self._clk_dirty = True
        self._layout = None
        self._pool.drain()
        for m in self._m.values():
            m.invalidate()

    def _push(self):
        """Send host-side changes (config, clock, mutated mirrors) to the device before a device operation."""
        if self._h is None:
            raise _lib.DaisyWorldError("environment has no device state; call reset()")
        B, N, n = self._shape
        # in-place edits of the small kernel arrays (env.daisy_kernel[...] = x) bypass __setattr__: compare their bytes
        sig = (np.asarray(self.daisy_kernel).tobytes(), np.asarray(self.adjacent_albedo_kernel).tobytes(),
               np.asarray(self.neighborhood).tobytes())
        if self._cfg_dirty or sig != self._arr_sig:
            cfg = self._config()
            cfg.batch, cfg.dim, cfg.n_agents = B, N, n      # shapes of live state only change at reset()
            self._check(self._lib.dw_set_config(self._h, C.byref(cfg)), "dw_set_config")
            self._cfg_dirty = False
            self._arr_sig = sig
        if self._clk_dirty:
            clk = self._clock()
            self._check(self._lib.dw_set_clock(self._h, C.byref(clk)), "dw_set_clock")
            self._clk_dirty = False
        g = ai = st = None
        if self._m["grid"].dirty():
            g = np.ascontiguousarray(self._m["grid"].handed, dtype=np.float64)
            if g.shape != (B, self.ch, N, N):
                raise ValueError(f"env.grid must have shape {(B, self.ch, N, N)}, got {g.shape}")
        if n and self._m["agent_indices"].dirty():
            ai = np.ascontiguousarray(self._m["agent_indices"].handed, dtype=np.int64)
            if ai.shape != (B, n, 2):
                raise ValueError(f"env.agent_indices must have shape {(B, n, 2)}, got {ai.shape}")
        if n and self._m["agent_states"].dirty():
            st = np.ascontiguousarray(self._m["agent_states"].handed, dtype=np.float64).reshape(B, n)
        if g is not None or ai is not None or st is not None:
            self._check(self._lib.dw_upload_state(self._h, _ptr(g, C.c_double), _ptr(ai, C.c_int64), _ptr(st, C.c_double)),
                        "dw_upload_state")
            for name, arr in (("grid", g), ("agent_indices", ai), ("agent_states", st)):
                if arr is not None:
                    m = self._m[name]
                    m.pristine = np.array(m.handed, copy=True)
                    m.assigned = False

    def _state_changed(self):
        for m in self._m.values():
            m.invalidate()
        self._diag_cache = {}

    # ------------------------------------------------------------------ host mirrors
    def _get_mirror(self, name):
        m = self._m[name]
        if m.handed is not None:
            return m.handed
        B, N, n = self._shape
        if name == "grid":
            arr = np.empty((B, self.ch, N, N))
            self._check(self._lib.dw_get_grid(self._h, _ptr(arr, C.c_double)), "dw_get_grid")
        else:
            ai = np.zeros((B, n, 2), dtype=np.int64)
            st = np.zeros((B, n, 1))
            if n:
                self._check(self._lib.dw_get_agents(self._h, _ptr(ai, C.c_int64), _ptr(st, C.c_double)), "dw_get_agents")
            for nm, a in (("agent_indices", ai), ("agent_states", st)):
                mm = self._m[nm]
                if mm.handed is None:
                    mm.pristine = a.copy()
                    mm.handed = a
            return self._m[name].handed
        m.pristine = arr.copy()
        m.handed = arr
        return arr

    def _set_mirror(self, name, value):
        m = self._m[name]
        m.handed = np.asarray(value)
        m.assigned = True

    grid = property(lambda self: self._get_mirror("grid"), lambda self, v: self._set_mirror("grid", v))
    agent_indices = property(lambda self: self._get_mirror("agent_indices"),
                             lambda self, v: self._set_mirror("agent_indices", v))
    agent_states = property(lambda self: self._get_mirror("agent_states"),
                            lambda self, v: self._set_mirror("agent_states", v))

    # ------------------------------------------------------------------ diagnostics (unrounded, lazy)
    def _diag(self, name):
        if name not in self._diag_cache:
            B, N, _ = self._shape
            out = np.empty((B, 2 if name == "growth" else 1, N, N))
            self._check(self._lib.dw_get_diag(self._h, DW_DIAG[name], _ptr(out, C.c_double)), "dw_get_diag")
            self._diag_cache[name] = out
        return self._diag_cache[name]

    temp = property(lambda self: self._diag("temp"))
    temp_light = property(lambda self: self._diag("temp_light"))
    temp_dark = property(lambda self: self._diag("temp_dark"))
    temp_effective = property(lambda self: self._diag("temp_effective"))
    beta = property(lambda self: self._diag("beta"))
    beta_l = property(lambda self: self._diag("beta_l"))
    beta_d = property(lambda self: self._diag("beta_d"))
    growth = property(lambda self: self._diag("growth"))

    def diag_stats(self, name):
        """{mean, std, min, max} of a diagnostic field (temp, temp_light, ..., growth) over the whole ensemble, reduced on
        the device: what the notebooks compute with env.temp.mean() (notebook_helpers.py:50,145,218) without the download."""
        out = np.zeros(4)
        self._push()
        self._check(self._lib.dw_get_diag_stats(self._h, DW_DIAG[name], _ptr(out, C.c_double)), "dw_get_diag_stats")
        return dict(mean=out[0], std=out[1], min=out[2], max=out[3])

    def cover_stats(self):
        """Mean and max light / dark cover of the current state over the whole ensemble, reduced on the device."""
        out = np.zeros(4)
        self._push()
        self._check(self._lib.dw_get_cover_stats(self._h, _ptr(out, C.c_double)), "dw_get_cover_stats")
        return dict(mean_light=out[0], mean_dark=out[1], max_light=out[2], max_dark=out[3])

    def run_series(self, K, policy="greedy", actions=None, seed=0):
        """run() that also returns the per-step ensemble means [K, 3] = (global mean temperature of that step's forward --
        env.temp.mean() --, mean light cover, mean dark cover): reduced inside the persistent fused kernels where the device
        has a series mode for the shape and the constants (dw_run_series decides), sampled between one-step launches
        otherwise."""
        B, N, n = self._shape
        colliding = self.collision_mode == 1 and n      # noise from the caller's NumPy stream every step: host-driven loop
        a8 = None
        if policy == "replay":
            a8 = np.ascontiguousarray(canonical_actions8(np.asarray(actions).reshape(-1, B, n)[:K]))
        out = np.zeros((int(K), 3))
        if not colliding and 1 <= K <= 4096:             # dw_run_series takes up to DW_FUSED_MAX_STEPS steps per call
            self._push()
            rc = self._lib.dw_run_series(self._h, int(K), DW_POLICY[policy], _ptr(a8, C.c_int8), C.c_uint64(seed),
                                         _ptr(out, C.c_double))
            if rc != DW_E_UNSUPPORTED:                   # refused before any step has run: fall through to the loop
                self._check(rc, "dw_run_series")
                self._state_changed()
                self._pull_clock()
                self._dead_L = None
                return out
        # one fused step per sample, the same three means from the device-side reductions
        for t in range(int(K)):
            self.run(1, policy=policy, actions=None if a8 is None else a8[t:t + 1], seed=seed)
            c = self.cover_stats()
            out[t] = (self.diag_stats("temp")["mean"], c["mean_light"], c["mean_dark"])
        return out

    def run_with_series(self, K, every=16, policy="greedy", seed=0):
        """K steps in chunks of `every`, recording after each chunk the ensemble diagnostics the reference's plot helpers
        read per step (notebook_helpers.py:45-57): global mean temperature, covers, luminosity, bare-planet temperature."""
        series = []
        done = 0
        while done < K:
            k = min(every, K - done)
            self.run(k, policy=policy, seed=seed)
            done += k
            t, c = self.diag_stats("temp"), self.cover_stats()
            series.append(dict(step=self.step_count, L=self.L, temp_mean=t["mean"], temp_std=t["std"], dead_temp=float(self.dead_temp[0]),
                               light=c["mean_light"], dark=c["mean_dark"]))
        return series

    @property
    def dead_temp(self):
        """reference :406-407,416 -- bare-planet temperature at the L of the last forward."""
        if self._dead_L is None:
            last = C.c_double()
            self._check(self._lib.dw_get_last_L(self._h, C.byref(last)), "dw_get_last_L")
            self._dead_L = last.value
        L = self._dead_L
        return np.array([((self.S * L * (1 - self.albedo_bare)) / self.sigma) ** (1 / 4)])

    # ------------------------------------------------------------------ reference API
    def set_use_microclimate(self, use_microclimate=True):
        self.use_microclimate = use_microclimate
        self.q2 = self.q / 8.0 if self.use_microclimate else 0.0

    _CONFIG_KEYS = ("max_L", "min_L", "initial_L", "ramp_period", "dL", "p", "g", "S", "sigma", "gamma", "albedo_bare",
                    "albedo_light", "albedo_dark", "temp_optimal", "light_proportion", "dark_proportion", "initial_al",
                    "initial_ad", "n_agents", "agent_gamma")

    def make_config(self):
        """reference :94-119"""
        return {k: getattr(self, k) for k in self._CONFIG_KEYS}

    def save_config(self, filepath=None):
        if filepath is None:
            filepath = os.path.join("results", "default_model_config.json")
        with open(filepath, "w") as f:
            json.dump(self.make_config(), f)

    def _apply_config(self, config):
        for k in self._CONFIG_KEYS:
            setattr(self, k, config[k])

    def load_config(self, filepath=None):
        if filepath is None:
            filepath = os.path.join("results", "default_model_config.json")
        with open(filepath, "r") as f:
            return json.load(f)

    def restore_config(self, filepath=None):
        self._apply_config(self.load_config(filepath))

    def initialize_neighborhood(self):
        """reference :265-283"""
        set_default_kernels(self)

    def initialize_agents(self):
        """reference :173-179 (one randint draw; states = 1)."""
        ai = np.random.randint(self.dim, size=(self.batch_size, self.n_agents, 2))
        st = np.ones((self.batch_size, self.n_agents, 1))
        if self._h is not None and self._shape == (self.batch_size, self.dim, self.n_agents):
            self.agent_indices = ai
            self.agent_states = st
        else:
            self._pending_agents = (ai, st)   # constructor call before the first reset(): no device state yet

    def initialize_grid(self):
        """reference :285-324: RNG draw order (dark first), cover init on the host; temperatures on the device."""
        B, N = self.batch_size, self.dim
        dark_probability = np.random.rand(B, 2, N, N)
        light_probability = np.random.rand(B, 2, N, N)
        dark = 1.0 * (dark_probability[:, 0] < self.dark_proportion) * self.initial_ad * dark_probability[:, 1]
        light = 1.0 * (light_probability[:, 0] < self.light_proportion) * self.initial_al * light_probability[:, 1]
        self._ensure_handle((int(B), int(N), int(self.n_agents)))
        self._m["grid"].invalidate()
        self._push()
        # narrow upload: the step reads only the two cover planes; ch0 and the temperatures are filled on the device
        light = np.ascontiguousarray(light, dtype=np.float64)
        dark = np.ascontiguousarray(dark, dtype=np.float64)
        self._check(self._lib.dw_upload_covers(self._h, _ptr(light, C.c_double), _ptr(dark, C.c_double)), "dw_upload_covers")
        self._check(self._lib.dw_init_temperatures(self._h), "dw_init_temperatures")
        self._dead_L = self.L
        self._m["grid"].invalidate()
        self._diag_cache = {}

    def reset(self):
        """reference :327-338"""
        self.L = self.min_L
        self.dL = (self.max_L - self.min_L) / self.ramp_period
        self.step_count = 0
        self.initialize_grid()
        self.initialize_agents()
        self._pending_agents = None
        return self.get_obs(self.agent_indices)

    def update_agents(self, action):
        """reference :181-244."""
        a = self._action(action)
        self._push()
        if self._shape[2]:
            if self.collision_mode == 1:
                self._update_agents_colliding(a, -1, 0)
            else:
                self._check(self._lib.dw_update_agents(self._h, _ptr(a, C.c_int64), a.shape[0], a.shape[1]), "dw_update_agents")
        self._state_changed()

    def _update_agents_colliding(self, a, policy, seed):
        """update_agents with collision_mode == 1 (reference :220-242). The device moves and grazes the agents and hands
        back their positions; this side only counts, per world, the cells holding more than one agent and draws the
        reference's npr.rand(1, n, 1) per such cell from the GLOBAL stream in the reference's (world, x, y) scan order
        (consecutive draws of n doubles = one draw of [cells, n]); the device then resolves the collisions and clips."""
        B, N, n = self._shape
        pos = np.empty((B, n, 2), dtype=np.int64)
        rc = self._lib.dw_agents_begin(self._h, None if a is None else _ptr(a, C.c_int64), 0 if a is None else a.shape[0],
                                       0 if a is None else a.shape[1], int(policy), C.c_uint64(seed), _ptr(pos, C.c_int64))
        self._check(rc, "dw_agents_begin")
        offsets = shared_cell_offsets(pos, N)
        cells = int(offsets[-1])
        noise = np.ascontiguousarray(np.random.rand(cells, n)) if cells else None
        rc = self._lib.dw_agents_collide(self._h, None if noise is None else _ptr(noise, C.c_double),
                                         offsets.ctypes.data_as(C.POINTER(C.c_int32)), float(self.food_chain_penalty))
        self._check(rc, "dw_agents_collide")

    def _action(self, action):
        a = np.asarray(action)
        if a.ndim != 3:
            raise IndexError("action must be indexable as action[b, n, 0] (reference :186-189)")
        return np.ascontiguousarray(a[:, :, 0], dtype=np.int64)

    def get_obs(self, agent_indices=None):
        """reference :246-263"""
        ai = np.ascontiguousarray(np.asarray(agent_indices), dtype=np.int64)
        b, m = ai.shape[:2]
        obs = np.zeros((b, m, self.ch, self.kr * 2 + 1, self.kr * 2 + 1))
        self._push()
        if b and m:
            self._check(self._lib.dw_get_obs_at(self._h, _ptr(ai, C.c_int64), b, m, _ptr(obs, C.c_double)), "dw_get_obs_at")
        return obs

    def forward(self, grid):
        """reference :434-461; standalone-callable (tests/daisy/test_daisy_world_rl.py:18-19)."""
        g = np.asarray(grid)
        B, N, _ = self._shape
        if g.shape != (B, self.ch, N, N):
            raise ValueError(f"forward expects a grid of shape {(B, self.ch, N, N)}")
        work = np.ascontiguousarray(g, dtype=np.float64)
        out = np.empty_like(work)
        self._push()
        self._check(self._lib.dw_forward(self._h, _ptr(work, C.c_double), _ptr(out, C.c_double)), "dw_forward")
        if work is not g:
            g[:, 0] = work[:, 0]
        self._dead_L = self.L
        self._diag_cache = {}
        return out

    def update_L(self, L):
        """reference :463-473"""
        self.step_count += 1
        if self.ramp_up_down and self.step_count % self.ramp_period == 0:
            self.dL *= -1
            self.min_L -= self.ddL
            self.max_L += self.ddL
        L += self.dL
        return max([min([L, self.max_L]), self.min_L])

    def step(self, action=None):
        """reference :475-497"""
        B, N, n = self._shape
        a = None
        if action is not None and n:
            a = self._action(action)
        return self._step_collect(a, -1, 0)

    def _out_views(self, want_obs):
        """A fresh block for dw_step_packed and the arrays step() returns carved out of it (layout: dw_step_out_layout)."""
        B, N, n = self._shape
        if self._layout is None:
            lay = (C.c_int64 * 4)()
            self._check(self._lib.dw_step_out_layout(self._h, lay), "dw_step_out_layout")
            self._layout = tuple(int(v) for v in lay)
        r_off, d_off, o_off, total = self._layout
        nbytes = total if (want_obs and n) else o_off
        buf = self._pool.take(nbytes)
        if buf is None:                              # many earlier outputs still referenced: ordinary memory
            buf = np.empty(nbytes, dtype=np.uint8)
            ptr = buf.ctypes.data_as(C.c_void_p)
        else:
            ptr = C.c_void_p(C.addressof(buf))       # NOT ctypes.cast: it stores the source in its own _objects (a cycle), and
                                                     # the block would only return to the pool when the cyclic GC runs
        m = n if n else 2
        reward = np.frombuffer(buf, dtype=np.float64, count=B * m, offset=r_off).reshape((B, n, 1) if n else (B, 2))
        done = np.frombuffer(buf, dtype=np.uint8, count=B * m, offset=d_off).reshape(reward.shape).view(np.bool_)
        obs = None
        if want_obs:
            obs = (np.frombuffer(buf, dtype=np.float64, count=B * n * 63, offset=o_off) if n else np.empty(0)).reshape(B, n, self.ch, 3, 3)
        return ptr, obs, reward, done

    def _step_collect(self, a, policy, seed, want_obs=True):
        """One step and everything step() returns: one C call, one device->host copy, one synchronisation."""
        B, N, n = self._shape
        self._push()
        self._dead_L = self.L
        clk = DwClock()
        if self.collision_mode == 1 and n:
            self._update_agents_colliding(a, policy, seed)
            ptr, obs, reward, done = self._out_views(True)       # the collision step returns the observation even without want_obs
            self._check(self._lib.dw_step_tail_packed(self._h, 1, ptr, C.byref(clk)), "dw_step_tail_packed")
        else:
            ptr, obs, reward, done = self._out_views(want_obs)
            rc = self._lib.dw_step_packed(self._h, None if a is None else _ptr(a, C.c_int64), 0 if a is None else a.shape[0],
                                          0 if a is None else a.shape[1], int(policy), C.c_uint64(seed), int(bool(want_obs)), ptr,
                                          C.byref(clk))
            self._check(rc, "dw_step_packed")
        self._state_changed()
        self._adopt_clock(clk)
        if not n:
            reward = reward.astype(bool)
        return obs, reward, done, {}

    def __call__(self, grid):
        pass

    # ------------------------------------------------------------------ additions: fused path
    def step_policy(self, policy="greedy", seed=0, want_obs=True):
        """One step with the action chosen on the device (Greedy's deterministic branch, or the MLP of set_mlp, fused in).
        want_obs=False returns None for the observation and leaves it on the device (the policy reads it there; observe()
        fetches it later): the step's device->host traffic drops from 504 to 9 bytes per agent."""
        return self._step_collect(None, DW_POLICY[policy], seed, want_obs=want_obs)

    def set_epsilon(self, epsilon):
        """Greedy.epsilon (agents/greedy.py:8) for policy="eps_greedy": per step ONE coin for the whole ensemble decides
        between random and greedy actions, like the reference's single np.random.rand() per call (device counter RNG)."""
        self._check(self._lib.dw_set_epsilon(self._h, float(epsilon)), "dw_set_epsilon")

    def observe(self):
        """Observations of the current state for all agents (what the last step()/run() would have returned). After a
        fused run only the agents' windows are re-evaluated on the device; the full grid is not materialised."""
        B, N, n = self._shape
        obs = np.zeros((B, n, self.ch, 3, 3))
        self._push()
        self._check(self._lib.dw_get_obs(self._h, _ptr(obs, C.c_double)), "dw_get_obs")
        return obs

    def grid_f32(self):
        """env.grid as float32 -- the fp32 mode. Lattice-resident state (after run() / lattice-resident step()): materialised
        with fp32 arithmetic from the packed lattice (k_forward_f32): covers and bare fraction are the float32 roundings of
        the reference values, temperatures within 1e-5 relative (observed 3e-6). Otherwise: env.grid converted on the device
        (6e-8). Half the download either way."""
        B, N, n = self._shape
        out = np.empty((B, self.ch, N, N), dtype=np.float32)
        self._push()
        self._check(self._lib.dw_get_grid_f32(self._h, _ptr(out, C.c_float)), "dw_get_grid_f32")
        return out

    def observe_f32(self):
        """observe() as float32 (what an fp32 policy network consumes): the agents' windows of grid_f32()."""
        B, N, n = self._shape
        out = np.zeros((B, n, self.ch, 3, 3), dtype=np.float32)
        self._push()
        self._check(self._lib.dw_get_obs_f32(self._h, _ptr(out, C.c_float)), "dw_get_obs_f32")
        return out

    def f32_stats(self):
        """Tier counters of the fp32-arithmetic materialisation: cells evaluated, cells whose bare fraction went on to the fp64
        fast path (fp32 value within its error bound of a rounding tie), cells that needed the literal cell."""
        out = (C.c_uint64 * 3)()
        self._check(self._lib.dw_f32_stats(self._h, out), "dw_f32_stats")
        return {"cells": int(out[0]), "fp64_tier": int(out[1]), "literal": int(out[2])}

    def set_mlp(self, parameters):
        """Weights of the reference's MLP policy (daisy/agents/mlp.py: MLP.get_parameters()) for policy="mlp": the
        63-16-32-9 ReLU network is evaluated on the device between steps, on observations built on the device."""
        p = np.ascontiguousarray(np.asarray(parameters, dtype=np.float64).ravel())
        self._check(self._lib.dw_set_mlp(self._h, _ptr(p, C.c_double), int(p.size)), "dw_set_mlp")

    def reset_lifespans(self):
        self._check(self._lib.dw_reset_lifespans(self._h), "dw_reset_lifespans")

    def lifespans(self):
        B, N, n = self._shape
        done_at = np.zeros((B,), dtype=np.int64)
        agents_done_at = np.zeros((B, n, 1), dtype=np.int64)
        self._check(self._lib.dw_get_lifespans(self._h, _ptr(done_at, C.c_int64), _ptr(agents_done_at, C.c_int64)),
                    "dw_get_lifespans")
        return done_at, agents_done_at

    def run(self, K, policy="greedy", actions=None, seed=0, stop_all_done=False):
        """K steps on the device with an on-device policy; lifespan counters accumulate (see lifespans()).

        policy: "none" | "greedy" | "antigreedy" | "random" | "eps_greedy" (see set_epsilon) | "mlp" (see set_mlp) | "replay"
        (actions[K,B,n(,1)] ints 0..8).
        Returns (steps_run, worlds_alive, all_done_hit)."""
        B, N, n = self._shape
        a8 = None
        if policy == "replay":
            a8 = np.ascontiguousarray(canonical_actions8(np.asarray(actions).reshape(-1, B, n)[:K]))
            if a8.shape[0] < K:
                raise ValueError("replay needs at least K action frames")
        if self.collision_mode == 1 and n:
            return self._run_colliding(int(K), policy, a8, seed, stop_all_done)
        self._push()
        res = DwRunResult()
        rc = self._lib.dw_run(self._h, int(K), DW_POLICY[policy], _ptr(a8, C.c_int8), C.c_uint64(seed),
                              int(bool(stop_all_done)), C.byref(res))
        self._check(rc, "dw_run")
        self._state_changed()
        self._pull_clock()
        self._dead_L = None
        return int(res.steps_run), int(res.worlds_alive), bool(res.all_done_hit)

    def _run_colliding(self, K, policy, a8, seed, stop_all_done):
        """run() with collision_mode == 1: the collision noise comes from the caller's NumPy stream every step (reference
        :220-242), so the loop is driven from here, one materialising step at a time; policy decisions, moves, grazing,
        collisions, forward and the lifespan counters stay on the device."""
        steps, alive, hit = 0, self._shape[0], False
        count = C.c_int64(0)
        self._push()                 # once: inside the loop the clock lives on the device (a push would rewind it)
        for t in range(K):
            if a8 is None:
                self._update_agents_colliding(None, DW_POLICY[policy], seed)
            else:
                self._update_agents_colliding(np.ascontiguousarray(a8[t], dtype=np.int64), -1, seed)
            self._check(self._lib.dw_step_tail_counted(self._h, C.byref(count)), "dw_step_tail_counted")
            steps, alive = steps + 1, int(count.value)
            if stop_all_done and alive == 0:
                hit = True
                break
        self._state_changed()
        self._pull_clock()
        self._dead_L = None
        return steps, alive, hit

    def simulate_lifespan(self, policy="greedy", actions=None, seed=0, max_steps=100000):
        """The notebook's simulate_lifespan (greedy_longevity_abatement.ipynb cell 2) after a reset():
        returns (done_at[B], agents_done_at[B,n,1])."""
        self.reset_lifespans()
        self.run(max_steps, policy=policy, actions=actions, seed=seed, stop_all_done=True)
        return self.lifespans()

    def reset_on_device(self, seed=0, world_offset=0):
        """reset() with the initial state drawn ON THE DEVICE (counter RNG; same distribution as the reference's reset,
        different stream): for ensembles too large to draw with numpy. Does not touch the global numpy RNG."""
        self.L = self.min_L
        self.dL = (self.max_L - self.min_L) / self.ramp_period
        self.step_count = 0
        self._ensure_handle((int(self.batch_size), int(self.dim), int(self.n_agents)))
        for m in self._m.values():
            m.invalidate()
        self._push()
        self._check(self._lib.dw_set_world_offset(self._h, int(world_offset)), "dw_set_world_offset")
        self._check(self._lib.dw_init_random(self._h, C.c_uint64(seed), self.light_proportion, self.dark_proportion,
                                             self.initial_al, self.initial_ad), "dw_init_random")
        self._check(self._lib.dw_init_temperatures(self._h), "dw_init_temperatures")
        self._dead_L = self.L
        self._diag_cache = {}
        self._pending_agents = None

    def residency(self):
        """Where the live state sits on the device: dict(grid=, lattice=, cover_planes=, pre=) (dw_debug_state)."""
        f = (C.c_int32 * 4)()
        self._check(self._lib.dw_debug_state(self._h, f), "dw_debug_state")
        return dict(grid=bool(f[0]), lattice=bool(f[1]), cover_planes=bool(f[2]), pre=int(f[3]))

    def synchronize(self):
        self._check(self._lib.dw_synchronize(self._h), "dw_synchronize")
