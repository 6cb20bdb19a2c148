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
