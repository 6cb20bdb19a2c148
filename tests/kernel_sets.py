"""Stencil kernels and physics constants beyond the reference's defaults, shared by the oracle and GPU kernel tests.

KERNEL_SETS maps a name to (daisy_kernel, adjacent_albedo_kernel), both (3, 3), as an env holds them:
  default     the reference's kernels (daisy_world_rl.py:270-273, :278-281)             -> fused path
  daisy_asym  9 distinct positive seeded taps, normalised: no symmetry of the square maps it to itself
                                                                                           -> materialising path
  adj_asym    reference daisy kernel; adjacent kernel of distinct taps, zero centre, sum 1 -> materialising path
  adj_centre  reference daisy kernel; adjacent kernel of distinct taps, non-zero centre, sum 1
                                                                                           -> materialising path
  d4_custom   D4 daisy kernel (centre 0.5, edge 0.1, corner 0.025); uniform adjacent 0.1 (sum 0.8)
                                                                                           -> fused, other coefficients
  d4_heavy    the reference daisy kernel scaled to sum 1.25 (densities can exceed 1)      -> fused

constant_draws() gives seeded physics constants in the ranges of tools/fuzz_fast_path.py::draw, plus p in [0.8, 1.0],
microclimate off in about a quarter of the draws, a short ramp_up_down period, and one draw with g = 0 (off the fast
path)."""
import numpy as np


def _reference_daisy():
    w = np.full((3, 3), np.exp(-1))
    w[1, 1] = 1.0
    w[0::2, 0::2] = np.exp(-2)
    return w / w.sum()


def _reference_adjacent():
    a = np.full((3, 3), 0.125)
    a[1, 1] = 0.0
    return a


def _distinct(rng, zero_centre):
    while True:
        t = rng.uniform(0.2, 1.0, size=9)
        if zero_centre:
            t[4] = 0.0
        if len(np.unique(t)) == 9:
            return (t / t.sum()).reshape(3, 3)


def _d4(centre, edge, corner):
    w = np.full((3, 3), edge)
    w[1, 1] = centre
    w[0::2, 0::2] = corner
    return w


def _kernel_sets():
    rng = np.random.RandomState(20261020)
    ref_w, ref_a = _reference_daisy(), _reference_adjacent()
    uniform = np.full((3, 3), 0.1)
    uniform[1, 1] = 0.0
    return {
        "default": (ref_w, ref_a),
        "daisy_asym": (_distinct(rng, zero_centre=False), ref_a),
        "adj_asym": (ref_w, _distinct(rng, zero_centre=True)),
        "adj_centre": (ref_w, _distinct(rng, zero_centre=False)),
        "d4_custom": (_d4(0.5, 0.1, 0.025), uniform),
        "d4_heavy": (ref_w * 1.25, ref_a),
    }


KERNEL_SETS = _kernel_sets()
ASYMMETRIC = ("daisy_asym", "adj_asym", "adj_centre")      # outside the fast path: the materialising kernels run them


def is_d4(w):
    return all(np.array_equal(w, v) for v in (w[::-1], w[:, ::-1], w.T))


def set_kernels(env, name):
    """Put kernel set `name` on an env (product or oracle) in the env's own shape."""
    w, a = KERNEL_SETS[name]
    env.daisy_kernel = w.reshape(np.shape(env.daisy_kernel)).copy()
    env.adjacent_albedo_kernel = a.reshape(np.shape(env.adjacent_albedo_kernel)).copy()


def constant_draws(count=5, seed=31):
    """`count` seeded constant sets (dicts of env attributes); the last one has g = 0."""
    rng = np.random.RandomState(seed)
    out = []
    for c in range(count):
        a = dict(albedo_bare=rng.uniform(0.3, 0.7), S=rng.uniform(700, 1300), g=10 ** rng.uniform(-3, -2),
                 gamma=rng.uniform(0.05, 0.45), dt=float(rng.choice([0.25, 0.5, 1.0])), temp_optimal=rng.uniform(280, 310),
                 agent_gamma=rng.uniform(0.01, 0.1), min_L=rng.uniform(0.5, 0.9), initial_al=rng.uniform(0.05, 0.6),
                 initial_ad=rng.uniform(0.05, 0.6), light_proportion=rng.uniform(0.1, 0.9),
                 dark_proportion=rng.uniform(0.1, 0.9), p=rng.uniform(0.8, 1.0))
        a["albedo_light"] = a["albedo_bare"] + rng.uniform(0.0, 0.3)
        a["albedo_dark"] = a["albedo_bare"] - rng.uniform(0.0, 0.3)
        a["max_L"] = a["min_L"] + rng.uniform(0.3, 1.2)
        a["use_microclimate"] = c % 4 != 1
        if c % 2 == 0:
            a.update(ramp_up_down=True, ramp_period=int(rng.choice([6, 10, 16])), ddL=float(rng.choice([0.0, 0.02])))
        if c == count - 1:
            a["g"] = 0.0
        out.append(a)
    return out


DRAWS = constant_draws()


def apply_draw(env, attrs):
    """Set a constant draw on an env before its reset(): q follows S like the reference's constructor (:43)."""
    for k, v in attrs.items():
        if k != "use_microclimate":
            setattr(env, k, v)
    env.q = 0.2 * env.S / env.sigma
    env.set_use_microclimate(attrs["use_microclimate"])


# (N, B, n) -> kernel family of the fused path (csrc/dw_run.inl::fused_kernel)
SHAPES = {
    (64, 6, 4): "64x64 persistent", (16, 9, 4): "sub-64", (8, 70, 3): "sub-64, partial CTA group", (20, 5, 3): "4x4 tile",
    (13, 4, 3): "padded tile", (33, 3, 5): "padded tile, odd N", (5, 3, 2): "generic", (2, 2, 1): "degenerate wrap",
    (1, 2, 1): "degenerate wrap",
}


# Shocks that move a cover by thousands of milli-covers in one step. The low word of the lattice kernels' rounding sum holds
# x + 0.5 (x = 1000 (l + dt dl), milli-cover) with only 12 integer bits, exact for x + 0.5 in [-2048, 2048); the kernels take
# the value from both words (csrc/dw_fused.cuh, DESIGN.md section 2). Far from T_opt, beta = 1 - g (T_opt - T)^2 is strongly
# negative. Every scenario leaves the 12-bit window and stays inside the tile loops' 16-bit one (window_crossings counts
# both). Every scenario is reached through plain attributes:
#   ctor    constructor keywords          attrs   attributes set before reset()
#   grow    steps before the shocked one  shock   attributes set right before the shocked step, put back after it
#   settle  steps after it                crosses whether the shocked step leaves the window (window_crossings proves it)
# A luminosity shock is not put back: the clock carries on from it (update_L clamps it into [min_L, max_L]).
# heat_step needs no shock: ramp_period=1 puts L at max_L after the literal first step, so step 2, the first step of the fast
# path, runs at max_L.
SCENARIOS = {
    "heat_step": dict(ctor=dict(ramp_period=1), attrs=dict(max_L=2.5), grow=1, shock={}, settle=20, crosses=True),
    "heat_graze": dict(ctor=dict(ramp_period=1), attrs=dict(max_L=2.0), grow=1, shock={}, settle=20, crosses=True),
    "heat_pulse": dict(ctor={}, attrs={}, grow=40, shock=dict(L=2.5), settle=20, crosses=True),
    "cold_pulse": dict(ctor={}, attrs={}, grow=40, shock=dict(L=0.1), settle=20, crosses=True),
    "upper_edge": dict(ctor={}, attrs={}, grow=40, shock=dict(dt=12.0, gamma=0.0), settle=20, crosses=True),
}
WINDOW = 2048.0          # |x + 0.5| bound of the fast path's low rounding word alone (12 integer bits), milli-cover
WIDE_WINDOW = 32768.0    # |x + 0.5| bound of the tile loops' rounding (funnel shift of both words, 16 bits)


def make_env(cls, name, N, B, n, seed):
    """An env of class `cls` (product or NumPy oracle) reset into scenario `name`'s starting state."""
    sc = SCENARIOS[name]
    np.random.seed(seed)
    env = cls(grid_dimension=N, n_agents=n, **sc["ctor"])
    env.batch_size = B
    for k, v in sc["attrs"].items():
        setattr(env, k, v)
    env.reset()
    return env


def apply_shock(name, *envs):
    """Set scenario `name`'s shock on every env (product, oracle or COracleWorld); returns the values to put back."""
    saved = []
    for env in envs:
        old = {}
        for k, v in SCENARIOS[name]["shock"].items():
            if hasattr(env, "clk") and hasattr(env, "P"):            # oracle.daisy_c.COracleWorld: clock and parameter structs
                target = env.clk if k == "L" else env.P
            else:
                target = env
            old[k] = getattr(target, k)
            setattr(target, k, v)
        saved.append(old)
    return saved


def undo_shock(name, saved, *envs):
    """Put back what apply_shock changed, except the luminosity, which the clock has moved on from."""
    for env, old in zip(envs, saved):
        for k, v in old.items():
            if k == "L":
                continue
            setattr(env.P if hasattr(env, "clk") and hasattr(env, "P") else env, k, v)


def window_crossings(name, N=64, B=4, n=4, seed=1, actions=None, state=None):
    """Run scenario `name` on the NumPy oracle up to its shocked step and
    return (below, above, wide, finite): how many cover updates of that step have 1000 (l + dt dl) + 0.5 below -WINDOW, at or
    above +WINDOW, and outside [-WIDE_WINDOW, WIDE_WINDOW), and whether every field of the step is finite. Counted from the
    unrounded fields(), so it holds whatever the kernels do. Agents: greedy, or actions[t] ([K, B, n] replay), or
    actions(obs) (a policy); state = (light, dark, agent_indices, agent_states) of one world replaces the reset state.
    """
    from oracle.daisy_numpy import OracleDaisyWorld, OracleGreedy
    sc = SCENARIOS[name]
    env = make_env(OracleDaisyWorld, name, N, B, n, seed)
    if state is not None:
        light, dark, ai, st = state
        env.batch_size = 1
        env.grid = np.zeros((1, 7, N, N))
        env.grid[0, 1], env.grid[0, 2] = light, dark
        env.agent_indices, env.agent_states = np.array(ai)[None].copy(), np.array(st, dtype=float)[None, :, None].copy()
    agent = OracleGreedy()
    obs = env.get_obs(env.agent_indices)

    def act(t, obs):
        if actions is None:
            return agent(obs)
        return actions(obs) if callable(actions) else np.asarray(actions[t]).reshape(env.batch_size, -1, 1)

    for t in range(sc["grow"]):
        obs, _, _, _ = env.step(act(t, obs))
    saved = apply_shock(name, env)
    seen = {}
    forward = env.forward

    def spy(grid):
        seen["f"] = env.fields(grid[:, 1].copy(), grid[:, 2].copy())
        seen["l"], seen["d"] = grid[:, 1].copy(), grid[:, 2].copy()
        return forward(grid)

    env.forward = spy
    try:
        env.step(act(sc["grow"], obs))
    finally:
        del env.forward
    f = seen["f"]
    x = np.stack([1000.0 * (seen["l"] + env.dt * f["dl"]), 1000.0 * (seen["d"] + env.dt * f["dd"])]) + 0.5
    undo_shock(name, saved, env)
    finite = all(np.isfinite(v).all() for v in f.values())
    return int((x < -WINDOW).sum()), int((x >= WINDOW).sum()), int(((x < -WIDE_WINDOW) | (x >= WIDE_WINDOW)).sum()), finite


def update_bound(L, dt=1.0, gamma=0.25, g=0.003265, S=1000.0, sigma=5.67e-8, p=1.0, ab=0.5, al=0.75, ad=0.25, Topt=295.5,
                 microclimate=True):
    """Upper bound of |x - k| (milli-cover) over every lattice state, for one step at luminosity L with the reference's kernels:
    rho (milli) <= 1000, |rho_b| <= dt max(p, 2 - p), and beta >= 1 - g (T_opt - T)^2 over the temperatures the fast path's
    linear form of T^4 reaches with covers in [0, 1000] and neighbour sums in [0, 8000]. inf when T^4 can reach 0."""
    q = 0.2 * S / sigma
    q2 = q / 8.0 if microclimate else 0.0
    a, cl, cd, cL = 0.125, (al - ab) / 1000.0, (ad - ab) / 1000.0, S * L / sigma
    x0 = cL + (q - cL) * ab * p * 8 * a + (q2 - q) * ab * p - q2 * al
    terms = ((q2 - q) * cl * 1000, (q2 - q) * cd * 1000, (q - cL) * a * cl * 8000, (q - cL) * a * cd * 8000)
    lo, hi = x0 + sum(min(0.0, t) for t in terms), x0 + sum(max(0.0, t) for t in terms)
    xdd = q2 * (al - ad)
    lo, hi = min(lo, lo + xdd), max(hi, hi + xdd)
    if lo <= 0:
        return np.inf
    dev = max(abs(Topt - lo ** 0.25), abs(Topt - hi ** 0.25))
    beta = max(1.0, g * dev * dev - 1.0)
    return 1000.0 * (abs(dt) * max(p, 2 - p) * beta + abs(dt * gamma))
