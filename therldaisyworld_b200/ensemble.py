"""Multi-rank lifespan ensembles: worlds are independent, so an ensemble shards contiguously across ranks with NO
data-path collective.  The only exchanges are (1) an AND all-reduce (MIN over 64 bit flags) of the "every world of my
shard was grid_done at step j" mask per 64-step segment -- the notebook's loop stops at the first step where ALL worlds are
done (notebooks/greedy_longevity_abatement.ipynb cell 2) -- and (2) one SUM all-reduce of the 8-double lifespan
statistics vector at the end.  One process per GPU; torch.distributed is only plumbing (NCCL on GPUs, gloo in the
CPU tests, where an oracle-backed shard stands in for the device).
"""
import ctypes as C

import numpy as np

from ._lib import DW_POLICY


def shard_range(total, world_size, rank):
    """Contiguous [lo, hi) slice of `total` worlds owned by `rank` (sizes differ by at most one)."""
    base, rem = divmod(total, world_size)
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)


class DeviceShard:
    """The worlds of one rank, living in a therldaisyworld_b200.RLDaisyWorld handle on that rank's GPU."""

    def __init__(self, env, world_offset=0):
        self.env = env
        env._check(env._lib.dw_set_world_offset(env._h, int(world_offset)), "dw_set_world_offset")

    def begin(self):
        self.env._push()
        self.env.reset_lifespans()

    def checkpoint_save(self):
        self.env._check(self.env._lib.dw_checkpoint_save(self.env._h), "dw_checkpoint_save")

    def checkpoint_restore(self):
        self.env._check(self.env._lib.dw_checkpoint_restore(self.env._h), "dw_checkpoint_restore")

    def trim_supported(self, policy):
        """True when the next chunk can run 'masked': past the stopping step without a checkpoint, the surplus taken out of
        the agents' lifespan counters afterwards (dw_run_chunk_masked / dw_trim_lifespans)."""
        yes = C.c_int32(0)
        self.env._check(self.env._lib.dw_trim_supported(self.env._h, DW_POLICY[policy], C.byref(yes)), "dw_trim_supported")
        return bool(yes.value)

    def suggest_segment(self):
        """Segment length for trimmed runs. Overshooting the stopping step costs segment/2 steps on average, a segment boundary a
        launch, a read-back and (multi-rank) two small all-reduces. Measured on a B200 (tools/segment_bench.py, whole lives of
        64x64 worlds, greedy; profiles/r02_segment_bench.txt): 100 000 worlds -- 64: 649 ms, 32: 611 ms, 16: 696 ms (checkpoint +
        replay with 64: 688 ms); 2000 worlds -- 13.9 / 13.6 / 15.6 ms (14.8 ms)."""
        return 32

    def trim(self, j):
        self.env._check(self.env._lib.dw_trim_lifespans(self.env._h, int(j)), "dw_trim_lifespans")

    def run_chunk(self, K, policy, actions=None, seed=0, masked=False):
        env = self.env
        B, N, n = env._shape
        a8 = None
        if policy == "replay":
            a8 = np.ascontiguousarray(np.asarray(actions).reshape(-1, B, n)[:K], dtype=np.int8)
        mask = C.c_uint64()
        fn = env._lib.dw_run_chunk_masked if masked else env._lib.dw_run_chunk
        rc = fn(env._h, int(K), DW_POLICY[policy], None if a8 is None else a8.ctypes.data_as(C.POINTER(C.c_int8)),
                C.c_uint64(seed), C.byref(mask))
        env._check(rc, "dw_run_chunk_masked" if masked else "dw_run_chunk")
        env._state_changed()
        env._pull_clock()
        return int(mask.value)

    def stats(self, like):
        """Local {count, sum life, sum life^2, n_agents_total, sum agent_life, sum agent_life^2, 0, 0} written into
        `like` (a torch CUDA float64 tensor of 8 elements) on the device, ready for an NCCL all-reduce."""
        self.env._check(self.env._lib.dw_lifespan_stats_device(self.env._h, C.c_void_p(like.data_ptr())),
                        "dw_lifespan_stats_device")
        return like

    def lifespans(self):
        return self.env.lifespans()


def _and_reduce(mask, group, dist, device, nbits=64):
    """Bitwise AND of a 64-bit mask over the ranks. NCCL has no BAND, so the mask travels as 64 {0,1} flags and is
    reduced with MIN (works on NCCL and gloo alike)."""
    import torch
    if dist is None or not dist.is_initialized() or dist.get_world_size(group) == 1:
        return mask
    bits = torch.tensor([(mask >> j) & 1 for j in range(nbits)], dtype=torch.int32, device=device)
    dist.all_reduce(bits, op=dist.ReduceOp.MIN, group=group)
    return sum(int(b) << j for j, b in enumerate(bits.tolist()))


def simulate_lifespan(shard, policy="greedy", actions=None, seed=0, max_steps=100000, group=None, device="cpu", segment=None):
    """Run the notebook's lifespan experiment on a sharded ensemble; returns a dict with global statistics.

    Every rank calls this with its own shard. `actions` (replay policy) is this rank's slice [K, B_local, n].
    segment: steps per launch (<= 64); None = 64, or the shard's suggestion (the same on every rank: MIN-reduced) once the
    segments run trimmed."""
    import torch
    try:
        import torch.distributed as dist
        if not dist.is_available():
            dist = None
    except Exception:       # pragma: no cover
        dist = None
    shard.begin()
    if actions is not None:
        max_steps = min(max_steps, len(actions))      # replay: cannot run past the recorded actions
    steps = 0
    hit = False
    can_trim = getattr(shard, "trim_supported", None)
    auto = segment is None
    short = 64
    if auto and hasattr(shard, "suggest_segment"):
        short = shard.suggest_segment()
        if dist is not None and dist.is_initialized() and dist.get_world_size(group) > 1:
            t = torch.tensor([short], dtype=torch.int32, device=device)
            dist.all_reduce(t, op=dist.ReduceOp.MIN, group=group)
            short = int(t[0])
    trimmed_before = False
    while steps < max_steps:
        seg = (short if trimmed_before else 64) if auto else segment
        k = min(seg, max_steps - steps)
        # Statistics only: when every rank's shard supports it, the segment runs 'masked' -- no checkpoint copy, and if the
        # stopping step falls inside it the surplus is trimmed out of the agents' counters instead of rewinding and replaying
        # (the rewind costs a full segment of steps per experiment: overshoot + replay = segment). Decided per segment by all
        # ranks together (same AND-reduce as the done mask).
        masked = bool(_and_reduce(1 if (can_trim is not None and can_trim(policy)) else 0, group, dist, device, nbits=1))
        trimmed_before = masked           # the first segment (off-lattice reset state) is never trimmed; the rest follow it
        if not masked:
            shard.checkpoint_save()
        a = None if actions is None else actions[steps:steps + k]
        mask = _and_reduce(shard.run_chunk(k, policy, a, seed, masked=True) if masked else shard.run_chunk(k, policy, a, seed),
                           group, dist, device)
        if mask:
            j = (mask & -mask).bit_length() - 1           # first step at which every world of every rank was done
            if j < k - 1:
                if masked:
                    shard.trim(j)
                else:
                    shard.checkpoint_restore()
                    shard.run_chunk(j + 1, policy, a, seed)
            steps += j + 1
            hit = True
            break
        steps += k
    s = shard.stats(torch.zeros(8, dtype=torch.float64, device=device))
    if dist is not None and dist.is_initialized() and dist.get_world_size(group) > 1:
        dist.all_reduce(s, op=dist.ReduceOp.SUM, group=group)
    s = s.tolist()
    count, n_ag = s[0], s[3]
    mean = s[1] / count
    var = max(s[2] / count - mean * mean, 0.0)
    out = {"steps": steps, "all_done": hit, "worlds": int(count), "biosphere_lifespan_mean": mean,
           "biosphere_lifespan_sem": (var ** 0.5) / count ** 0.5}
    if n_ag:
        am = s[4] / n_ag
        av = max(s[5] / n_ag - am * am, 0.0)
        # the notebook divides the agent std by sqrt(number of worlds) (cell 16)
        out.update(agent_lifespan_mean=am, agent_lifespan_sem=(av ** 0.5) / count ** 0.5)
    return out
