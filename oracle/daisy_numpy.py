"""CPU oracle (NumPy) for the RLDaisyWorld simulation step -- TEST INFRASTRUCTURE ONLY.

This file restates, in plain NumPy, the algorithm of the reference environment
``daisy/daisy_world_rl.py`` (riveSunder/therldaisyworld).  It is the *checker* for the
CUDA path: only ``tests/``, ``__graft_entry__.smoke()`` and the ``cpu_baseline`` /
``--impl reference`` legs of ``bench.py`` may import it.  Nothing under
``therldaisyworld_b200/`` imports it; the product path has no CPU fallback.

Parity status: the reference ships NO golden vectors or known-answer tests for this path
(its tests are shape/sign smoke tests, SURVEY.md section 4).  The oracle is therefore pinned
against trajectories recorded from the live, unmodified reference by
``oracle/gen_golden.py`` (fixtures in ``tests/golden/*.npz``) -- see
``tests/test_oracle_golden.py``.

Two convolution modes:
  * ``conv="stencil"`` (default): the 3x3 toroidal stencil that the reference's FFT
    convolution (``daisy/nn/functional.py:12-49``) is mathematically equal to.  ``ft_convolve``
    multiplies the two spectra, so it is a true circular convolution, not a correlation:
    out[i,j] = sum w[a,b]*x[i+1-a, j+1-b].  The tap order below is the *canonical arithmetic
    order* that ``oracle/daisy_oracle.c`` and the CUDA materialising kernel reproduce operation
    for operation.
  * ``conv="fft"``: circular convolution through ``np.fft`` like the reference, used only as
    the CPU *baseline* (same cost profile as the reference's NumPy path).

Canonical arithmetic order (IEEE binary64, no FMA contraction), per cell:
  b   = (p - l) - d                                            # daisy_world_rl.py:381
  Al  = ((ab*b) + al*l) + ad*d                                 # :388-390
  conv(x, w) = sum over the neighbour offsets (di, dj), row-major from (-1,-1) to (+1,+1), of
               w[1-di, 1-dj]*x[i+di, j+dj], left to right; the centre term is skipped only when
               its tap is exactly 0.0 (the default adjacent-albedo kernel)
  A   = ((ab*conv(b, adj)) + al*conv(l, adj)) + ad*conv(d, adj)   # :391, :278-281
  rho(x) = conv(x, daisy_kernel)                               # :423-432, :270-273
  Te  = root4(((S*L)*(1-A))/sigma)                             # :403-404
  T   = root4(q*(A-Al) + pow4(Te))                             # :409
  Tl  = root4(q2*(Al-al) + pow4(T));  Td likewise with ad      # :411-412
  root4(x) = sqrt(sqrt(x)); pow4(x) = (x*x)*(x*x)
  beta_x = 1 - g*((Topt-T_x)*(Topt-T_x))                       # :342-344
  ab_ = (p - rho_l) - rho_d                                    # :361
  dl  = rho_l*(ab_*beta_l - gamma); dd likewise                # :367-368
  l'  = clip(l + dt*dl, 0, 1); d' likewise; b' = (p - l') - d' # :449-450
  every channel: rint(x*1000)/1000                             # :452
"""
import json

import numpy as np

DEFAULTS = dict(
    ch=7, batch_size=32, kr=1, neighborhood_mode="von_neumann", dim=16,
    p=1.0, g=0.003265, S=1000.0, sigma=5.67e-8, gamma=0.25, use_microclimate=True,
    collision_mode=0, Toptim=295.5, dt=1.0, ddL=0.0, agent_gamma=0.05,
    max_L=1.5, min_L=0.75, ramp_period=512, ramp_up_down=False,
    albedo_bare=0.5, albedo_light=0.75, albedo_dark=0.25, temp_optimal=295.5,
    food_chain_penalty=0.5, initial_al=0.2, initial_ad=0.2,
    light_proportion=0.33, dark_proportion=0.33, n_agents=4,
)


def neighborhood_mask(radius=1, mode="von_neumann"):
    """Observation mask (reference: daisy/nn/functional.py:51-103)."""
    r = np.arange(-radius, radius + 1)
    dx, dy = np.meshgrid(r, r)
    if mode == "moore":
        dist = np.maximum(np.abs(dx), np.abs(dy))
    elif mode == "circular":
        dist = np.sqrt(dx ** 2 + dy ** 2)
    else:  # "von_neumann" and the reference's fallback for unknown names
        dist = np.abs(dx) + np.abs(dy)
    return (dist <= radius).astype(np.float64)


def daisy_weights():
    """3x3 spread kernel (reference: daisy_world_rl.py:270-273)."""
    w = np.full((3, 3), np.exp(-1))
    w[1, 1] = 1.0
    w[0::2, 0::2] = np.exp(-2)
    return w / w.sum()


def _shift(x, di, dj):
    """x[i+di, j+dj] with toroidal wrap on the last two axes."""
    return np.roll(x, shift=(-di, -dj), axis=(-2, -1))


def stencil9(x, w):
    """Circular convolution like ft_convolve: sum over the offsets (di, dj), row-major, of w[1-di, 1-dj]*x[i+di, j+dj],
    accumulated left to right; a centre tap of exactly 0.0 is skipped."""
    acc = None
    for di in (-1, 0, 1):
        for dj in (-1, 0, 1):
            tap = w[1 - di, 1 - dj]
            if tap == 0.0 and (di, dj) == (0, 0):
                continue  # the default adjacent-albedo kernel skips its zero centre tap
            term = tap * _shift(x, di, dj)
            acc = term if acc is None else acc + term
    return acc


def fft_circular(x, w):
    """Same convolution through the FFT (cost profile of the reference's ft_convolve)."""
    n = x.shape[-1]
    k = np.zeros((n, n))
    for a in range(3):
        for b in range(3):
            k[(a - 1) % n, (b - 1) % n] += w[a, b]
    return np.real(np.fft.ifft2(np.fft.fft2(x, axes=(-2, -1)) * np.fft.fft2(k), axes=(-2, -1)))


def root4(x):
    return np.sqrt(np.sqrt(x))


def pow4(x):
    x2 = x * x
    return x2 * x2


def round3(x):
    return np.rint(x * 1000.0) / 1000.0


class OracleDaisyWorld:
    """NumPy restatement of RLDaisyWorld (reference: daisy/daisy_world_rl.py:13-501)."""

    def __init__(self, conv="stencil", **kwargs):
        for k, v in DEFAULTS.items():
            setattr(self, k, v)
        self.conv = conv
        # recognised constructor keys (reference :24-29,44,62,79); anything else is ignored
        self.kr = kwargs.get("kr", 1)
        self.neighborhood_mode = kwargs.get("neighborhood_mode", "von_neumann")
        self.dim = kwargs.get("grid_dimension", 16)
        self.collision_mode = kwargs.get("collision_mode", 0)
        self.ramp_period = kwargs.get("ramp_period", 512)
        self.n_agents = kwargs.get("n_agents", 4)
        self.q = 0.2 * self.S / self.sigma
        self.q2 = self.q / 8.0
        self.initial_L = self.min_L
        self.neighborhood = neighborhood_mask(self.kr, self.neighborhood_mode)
        self.daisy_kernel = daisy_weights()
        self.adjacent_albedo_kernel = np.full((3, 3), 0.125)    # the reference's attribute name (:278-281)
        self.adjacent_albedo_kernel[1, 1] = 0.0
        self.init_agents()
        self.reset()

    def set_use_microclimate(self, flag=True):
        self.use_microclimate = flag
        self.q2 = self.q / 8.0 if flag else 0.0

    # ---- initialisation (reference :173-179, :285-338) ------------------------------
    def init_agents(self):
        self.agent_indices = np.random.randint(self.dim, size=(self.batch_size, self.n_agents, 2))
        self.agent_states = np.ones((self.batch_size, self.n_agents, 1))

    def init_grid(self):
        B, N = self.batch_size, self.dim
        u_dark = np.random.rand(B, 2, N, N)     # dark is drawn first (:287)
        u_light = np.random.rand(B, 2, N, N)
        dark = 1.0 * (u_dark[:, 0] < self.dark_proportion) * self.initial_ad * u_dark[:, 1]
        light = 1.0 * (u_light[:, 0] < self.light_proportion) * self.initial_al * u_light[:, 1]
        grid = np.zeros((B, self.ch, N, N))
        grid[:, 0] = self.p - light - dark
        grid[:, 1] = light
        grid[:, 2] = dark
        f = self.fields(grid[:, 1], grid[:, 2])
        grid[:, 3], grid[:, 4], grid[:, 5] = f["T"], f["Tl"], f["Td"]   # unrounded (:314-323)
        self.grid = grid

    def reset(self):
        self.L = self.min_L
        self.dL = (self.max_L - self.min_L) / self.ramp_period
        self.step_count = 0
        self.init_grid()
        self.init_agents()
        return self.get_obs(self.agent_indices)

    # ---- physics (reference :340-432) -----------------------------------------------
    def _conv(self, x, w):
        w = np.asarray(w, dtype=np.float64).reshape(3, 3)    # (3, 3) or the reference's (1, 1, 3, 3)
        return stencil9(x, w) if self.conv == "stencil" else fft_circular(x, w)

    def fields(self, l, d):
        """All per-cell intermediate fields of one forward pass from daisy covers l, d [B,N,N]."""
        ab, al, ad = self.albedo_bare, self.albedo_light, self.albedo_dark
        b = self.p - l - d
        Al = ab * b + al * l + ad * d
        adj = self.adjacent_albedo_kernel
        A = ab * self._conv(b, adj) + al * self._conv(l, adj) + ad * self._conv(d, adj)
        rho_l = self._conv(l, self.daisy_kernel)
        rho_d = self._conv(d, self.daisy_kernel)
        SL = self.S * self.L
        Te = root4((SL * (1 - A)) / self.sigma)
        dead = root4((SL * (1 - self.albedo_bare)) / self.sigma)
        T = root4(self.q * (A - Al) + pow4(Te))
        T4 = pow4(T)
        Tl = root4(self.q2 * (Al - al) + T4)
        Td = root4(self.q2 * (Al - ad) + T4)
        dT, dTl, dTd = self.temp_optimal - T, self.temp_optimal - Tl, self.temp_optimal - Td
        beta = 1 - self.g * (dT * dT)
        beta_l = 1 - self.g * (dTl * dTl)
        beta_d = 1 - self.g * (dTd * dTd)
        bare = self.p - rho_l - rho_d
        dl = rho_l * (bare * beta_l - self.gamma)
        dd = rho_d * (bare * beta_d - self.gamma)
        return dict(b=b, Al=Al, A=A, rho_l=rho_l, rho_d=rho_d, Te=Te, dead=dead, T=T, Tl=Tl, Td=Td,
                    beta=beta, beta_l=beta_l, beta_d=beta_d, dl=dl, dd=dd)

    def forward(self, grid):
        """reference :434-461.  Mutates grid[:,0] like the reference (:381)."""
        l, d = grid[:, 1], grid[:, 2]
        f = self.fields(l, d)
        grid[:, 0] = f["b"]
        B, N = grid.shape[0], grid.shape[-1]
        # side-effect diagnostics, unrounded, reference shapes (:345-347,373,404,415-419)
        self.temp, self.temp_light, self.temp_dark = (f[k][:, None] for k in ("T", "Tl", "Td"))
        self.temp_effective = f["Te"][:, None]
        self.dead_temp = np.array([f["dead"]])
        self.beta, self.beta_l, self.beta_d = (f[k][:, None] for k in ("beta", "beta_l", "beta_d"))
        self.growth = np.stack([f["dl"], f["dd"]], axis=1)
        new = np.zeros_like(grid)
        new[:, 1] = np.clip(l + self.dt * f["dl"], 0, 1)
        new[:, 2] = np.clip(d + self.dt * f["dd"], 0, 1)
        new[:, 0] = self.p - new[:, 1] - new[:, 2]
        new[:, 3], new[:, 4], new[:, 5] = f["T"], f["Tl"], f["Td"]
        new = round3(new)
        for bb in range(self.batch_size if self.n_agents else 0):
            for nn in range(self.n_agents):      # last index wins, dead agents included (:454-459)
                x, y = self.agent_indices[bb, nn]
                new[bb, 4, x, y] = self.agent_states[bb, nn, 0]
        return new

    # ---- agents (reference :181-263) --------------------------------------------------
    def update_agents(self, action):
        self.agent_states = self.agent_states - self.agent_gamma
        N = self.dim
        for bb in range(action.shape[0]):
            for nn in range(action.shape[1]):
                if not self.agent_states[bb, nn, 0] > 0.0:
                    continue                      # dead agents neither move nor graze
                a = int(action[bb, nn, 0])
                if a != 8:
                    axis, step = ((1, -1), (0, -1), (0, 1), (1, 1))[a % 4]
                    self.agent_indices[bb, nn, axis] += step
                self.agent_indices %= N           # reference wraps the whole array here (:208)
                if a > 4:                          # 5,6,7 move+graze; 8 graze in place; 4 moves only
                    x, y = self.agent_indices[bb, nn]
                    self.agent_states[bb, nn, 0] += self.grid[bb, 1, x, y] + self.grid[bb, 2, x, y]
                    self.grid[bb, 1:3, x, y] *= 0.0
        if self.collision_mode == 1:
            self.resolve_collisions()
        self.agent_states = np.clip(self.agent_states, 0.0, 1.0)

    def resolve_collisions(self):
        """reference :220-242 (next row N4). The reference scans every cell (xx, yy) of every world in row-major order and,
        where more than one agent sits, draws npr.rand(1, n, 1) from the GLOBAL stream: tie-break noise for all n agents of
        the world. The resident with the largest state + 0.01 * noise gains food_chain_penalty * (sum of the other
        residents' states, unclipped, dead agents included); the losers are NOT zeroed (the reference's last statement
        assigns into a fancy-indexed copy, :242). Only occupied cells can hold residents, so visiting the occupied cells in
        sorted (xx, yy) order consumes the stream exactly like the full scan."""
        n = self.agent_states.shape[1]
        for bb in range(self.agent_indices.shape[0]):
            cells = sorted({(int(x), int(y)) for x, y in self.agent_indices[bb]})
            for xx, yy in cells:
                residents = (self.agent_indices[bb, :, 0] == xx) & (self.agent_indices[bb, :, 1] == yy)
                if residents.sum() > 1:
                    noise = np.random.rand(1, n, 1)[0, :, 0]
                    temp = 1.0 * self.agent_states[bb, :, 0] + 0.01 * noise
                    winner_value = temp[residents].max()
                    losers = residents & (temp != winner_value)
                    eat = np.sum(self.agent_states[bb, :, 0][losers])        # NumPy's summation order (see sum_like_numpy)
                    self.agent_states[bb, temp == winner_value, 0] += self.food_chain_penalty * eat

    def get_obs(self, agent_indices):
        B, n = agent_indices.shape[:2]
        N = self.dim
        obs = np.zeros((B, n, self.ch, 3, 3))
        win = np.arange(-1, 2)
        for bb in range(B):
            for nn in range(n):
                x, y = agent_indices[bb, nn]
                rows = (x + win) % N
                cols = (y + win) % N
                obs[bb, nn] = self.grid[bb][:, rows][:, :, cols]
        return obs * self.neighborhood

    def update_L(self, L):
        self.step_count += 1
        if self.ramp_up_down and self.step_count % self.ramp_period == 0:
            self.dL *= -1
            self.min_L -= self.ddL
            self.max_L += self.ddL
        L += self.dL
        return max(min(L, self.max_L), self.min_L)

    def step(self, action=None):
        if action is None and self.n_agents:
            action = np.zeros((self.batch_size, self.n_agents, 1))
        if action is not None:
            self.update_agents(action)
        self.grid = self.forward(self.grid)
        obs = self.get_obs(self.agent_indices)
        if self.n_agents:
            reward = 1.0 * self.agent_states
        else:
            reward = self.grid[:, 1:3].sum(axis=(-2, -1)) > 0
        reward = reward * (reward > 0)
        done = reward < 0.1
        self.L = self.update_L(self.L)
        return obs, reward, done, {}


class OracleGreedy:
    """NumPy restatement of the Greedy policy (reference: daisy/agents/greedy.py:5-36)."""

    NEIGHBOURS = (3, 1, 7, 5)   # flat 3x3 indices of (y-1, x-1, x+1, y+1)  -> actions 4..7

    def __init__(self, epsilon=0.0, greedy=True):
        self.epsilon = epsilon
        self.greedy = greedy

    def __call__(self, obs):
        B, n = obs.shape[:2]
        food = (obs[..., 1, :, :] + obs[..., 2, :, :]).reshape(B, n, 9)[:, :, list(self.NEIGHBOURS)]
        if np.random.rand() > self.epsilon:      # ONE draw for the whole batch (:23)
            pick = np.argmax(food, axis=-1) if self.greedy else np.argmin(food, axis=-1)
            return (4 + pick).reshape(B, n, 1)
        return np.random.randint(9, size=(B, n, 1, 1)).reshape(B, n, 1)


class OracleMLP:
    """NumPy restatement of the MLP policy (reference: daisy/agents/mlp.py:12-147): 63 -> 16 -> 32 -> 9, no biases,
    relu(x) = x * (x > 0) (:20), action = argmax of the raw logits (:106-116); flat parameter layout of
    get_parameters / set_parameters (:122-147): the three weight matrices row-major, in order."""

    SHAPES = ((63, 16), (16, 32), (32, 9))
    N_PARAMS = sum(a * b for a, b in SHAPES)

    def __init__(self, parameters):
        p = np.asarray(parameters, dtype=np.float64).ravel()
        assert p.size == self.N_PARAMS
        self.layers, k = [], 0
        for a, b in self.SHAPES:
            self.layers.append(p[k:k + a * b].reshape(a, b))
            k += a * b

    def logits(self, obs):
        x = obs.reshape(*obs.shape[:-3], 63)
        for w in self.layers[:-1]:
            x = np.matmul(x, w)
            x = x * (x > 0.0)
        return np.matmul(x, self.layers[-1])

    def __call__(self, obs):
        return np.argmax(self.logits(obs), axis=-1, keepdims=True)


def es_get_fitness(env, agent, adversary, max_steps=768):
    """NumPy restatement of SimpleGaussianES.get_fitness (reference: daisy/evo/sges.py:144-181): one member (first half of
    every world's agents) against an adversary (second half) on a freshly reset env; returns (fitness, total_steps,
    done_at, steps_run)."""
    obs = env.reset()
    half = obs.shape[1] // 2
    all_done = False
    done_at = np.zeros((*obs.shape[:2], 1), dtype=int)
    total_steps = np.zeros((*obs.shape[:2], 1), dtype=int)
    sum_reward = 0.0
    while not all_done and env.step_count < max_steps:
        action = np.append(agent(obs[:, :half]), adversary(obs[:, half:]), axis=1)
        obs, reward, done, info = env.step(action)
        all_done = (np.ones_like(done).sum() - done.sum()) == 0
        done_at += (1 - 1 * done)
        sum_reward += (reward[:, :half]).mean()
        total_steps += (1 - 1 * done)
    return sum_reward / (obs.shape[0] * obs.shape[1]), total_steps, done_at, env.step_count


def lifespan_loop(env, agent, max_steps=100000):
    """The README lifespan metric (notebooks/greedy_longevity_abatement.ipynb cell 2).

    Assumes env.reset() has been called by the caller if a fresh world is wanted; returns
    (done_at[B], agents_done_at[B,n,1], steps_run)."""
    obs = env.get_obs(env.agent_indices)
    B, n = obs.shape[:2]
    done_at = np.zeros((B,), dtype=np.int64)
    agents_done_at = np.zeros((B, n, 1), dtype=np.int64)
    steps = 0
    while steps < max_steps:
        action = agent(obs) if agent is not None else None
        obs, reward, done, _ = env.step(action)
        steps += 1
        grid_done = env.grid[:, 1:3].max(axis=(1, 2, 3)) <= 0.005
        done_at += 1 - 1 * grid_done
        if n:
            agents_done_at += 1 - 1 * done
        if grid_done.all():
            break
    return done_at, agents_done_at, steps


def env_from_golden(z, conv="stencil"):
    """Rebuild an oracle env in the exact post-reset state recorded in a golden fixture."""
    meta = json.loads(str(z["meta"]))
    state = np.random.get_state()
    env = OracleDaisyWorld(conv=conv, **meta["ctor"])
    np.random.set_state(state)                     # constructing the oracle must not disturb callers
    for k, v in meta["attrs"].items():
        if k == "use_microclimate":
            env.set_use_microclimate(v)
        else:
            setattr(env, k, v)
    env.L = env.min_L
    env.dL = (env.max_L - env.min_L) / env.ramp_period
    env.step_count = 0
    env.grid = z["init_grid"].copy()
    env.agent_indices = z["init_agent_indices"].copy()
    env.agent_states = z["init_agent_states"].copy()
    return env, meta
