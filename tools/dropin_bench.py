"""The drop-in step() path as a reference caller uses it (daisy/agents/greedy.py:39-89, daisy/evo/sges.py:152-175): one
env.step(action) per iteration with a host policy, observation / reward / done downloaded every step -- against
step_policy (action chosen on the device) with and without the observation download. The state stays lattice-resident
(K = 1 launches of the fused kernel)."""
import json, os, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np


def host_greedy(obs):
    food = (obs[..., 1, :, :] + obs[..., 2, :, :]).reshape(*obs.shape[:2], 9)[:, :, [3, 1, 7, 5]]
    return (4 + np.argmax(food, axis=-1))[..., None]


def measure(B, N, n=4, iters=200, warm=20, device=0):
    """ms per call of the three single-step modes on one (B, N) ensemble."""
    from therldaisyworld_b200 import RLDaisyWorld
    np.random.seed(13)
    env = RLDaisyWorld(grid_dimension=N, n_agents=n, device=device)
    env.batch_size = B
    obs = env.reset()
    out = {"worlds": B, "grid": N, "n_agents": n, "iters": iters}
    modes = {"step_host_greedy": lambda o: env.step(host_greedy(o)),
             "step_policy_device_greedy": lambda o: env.step_policy("greedy"),
             "step_policy_no_obs": lambda o: env.step_policy("greedy", want_obs=False)}
    for name, fn in modes.items():
        obs = env.reset()
        for _ in range(warm):
            obs = fn(obs)[0]
        t0 = time.perf_counter()
        for _ in range(iters):
            obs = fn(obs)[0]
        dt = (time.perf_counter() - t0) / iters
        out[name] = {"ms_per_step": dt * 1e3, "env_steps_per_s": B / dt, "cell_updates_per_s": B * N * N / dt}
    out["residency"] = env.residency()
    return out


if __name__ == "__main__":
    for B, N in ((32, 16), (1000, 8), (32, 64), (1000, 64), (10000, 64)):
        r = measure(B, N)
        print(json.dumps(r), flush=True)
