/*
 * daisyworld_b200.h -- C ABI of the B200-native RLDaisyWorld simulation step.
 *
 * The reference (riveSunder/therldaisyworld) has no FFI: its boundary is the Python surface of
 * class RLDaisyWorld (daisy/daisy_world_rl.py:13-501).  Each entry point below names the reference
 * method / attribute it stands in for.  The Python drop-in (therldaisyworld_b200/env.py) binds these
 * symbols with ctypes; INTEGRATION.md shows the binding a reference maintainer would add.
 *
 * Conventions
 *   - every call returns 0 on success, <0 on error (DW_E_*); text via dw_last_error().
 *   - the caller owns every host buffer; the library owns all device memory.
 *   - state-changing calls are enqueued on the handle's CUDA stream (dw_set_stream; default: the
 *     legacy default stream) and return without waiting; getters synchronise that stream.
 *   - a handle is bound to one CUDA device, is not thread-safe; distinct handles are independent.
 *   - no host RNG, no global state, no CPU fallback: if no CUDA device is usable dw_create fails.
 *   - array layouts are the reference's: grid[B,7,N,N] f64 (channels: 0 bare, 1 light, 2 dark,
 *     3 T, 4 T_light/agent stamp, 5 T_dark, 6 unused), agent_indices[B,n,2] i64 (x = axis -2,
 *     y = axis -1), agent_states[B,n] f64, obs[B,n,7,3,3] f64.
 */
#ifndef DAISYWORLD_B200_H
#define DAISYWORLD_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DW_ABI_VERSION 3

enum {
    DW_OK = 0,
    DW_E_INVALID = -1,      /* bad argument / shape */
    DW_E_CUDA = -2,         /* CUDA runtime error (message has the CUDA string) */
    DW_E_UNSUPPORTED = -3,  /* configuration outside what the kernels implement */
    DW_E_STATE = -4         /* call not valid in the current state */
};

/* Policies executed on the device inside dw_step_packed / dw_run. */
enum {
    DW_POLICY_NONE = 0,       /* step(None): all-zero action when n_agents>0 (daisy_world_rl.py:477-478) */
    DW_POLICY_GREEDY = 1,     /* Greedy(eps=0), argmax branch (daisy/agents/greedy.py:16-30) */
    DW_POLICY_ANTIGREEDY = 2, /* Greedy(greedy=False), argmin branch (greedy.py:27-28) */
    DW_POLICY_REPLAY = 3,     /* actions[K,B,n] supplied by the caller (stochastic policies replayed) */
    DW_POLICY_RANDOM = 4,     /* uniform 0..8 per agent-step from a device counter RNG (throughput runs;
                                 not stream-compatible with numpy's MT19937) */
    DW_POLICY_EPS_GREEDY = 5, /* Greedy(epsilon=eps) (greedy.py:23-32): ONE coin per step for the whole ensemble (the
                                 reference draws one np.random.rand() per call): random actions if it lands below eps
                                 (dw_set_epsilon), greedy otherwise. Counter RNG like DW_POLICY_RANDOM. */
    DW_POLICY_MLP = 6         /* MLP.get_action (daisy/agents/mlp.py:97-116): 63-16-32-9 ReLU network on the agent's
                                 masked 7x3x3 observation, argmax of the logits; weights from dw_set_mlp. The
                                 observation is built on the device from the state the last step started from. */
};
#define DW_MLP_PARAMS 1808    /* 63*16 + 16*32 + 32*9, flat layout of MLP.get_parameters (mlp.py:122-147) */

/* dw_get_diag selectors: unrounded side-effect attributes of the last forward
   (daisy_world_rl.py:345-347,373,404,415-419). Each is [B,1,N,N] except growth [B,2,N,N]. */
enum {
    DW_DIAG_TEMP = 0, DW_DIAG_TEMP_LIGHT = 1, DW_DIAG_TEMP_DARK = 2, DW_DIAG_TEMP_EFFECTIVE = 3,
    DW_DIAG_BETA = 4, DW_DIAG_BETA_L = 5, DW_DIAG_BETA_D = 6, DW_DIAG_GROWTH = 7
};

/* Model constants: the mutable public attributes of RLDaisyWorld (daisy_world_rl.py:32-77) that the
   step reads.  batch/dim/n_agents fix the shapes of a handle (the reference re-reads them at reset();
   the Python front re-creates the handle there). */
typedef struct dw_config {
    int32_t batch;        /* env.batch_size (worlds owned by this handle / rank) */
    int32_t dim;          /* env.dim  (grid side N) */
    int32_t n_agents;     /* env.n_agents */
    int32_t device;       /* CUDA device ordinal */
    double p, g, S, sigma, gamma, q, q2, temp_optimal, dt, agent_gamma;
    double albedo_bare, albedo_light, albedo_dark;
    /* Both kernels are given as the env holds them, row-major 3x3. The step convolves with them like ft_convolve
       (daisy/nn/functional.py:12-49): out[i][j] = sum over a, b of k[a][b] * x[i+1-a][j+1-b], toroidal. */
    double daisy_kernel[9];     /* env.daisy_kernel (daisy_world_rl.py:270-273) */
    double adjacent_kernel[9];  /* env.adjacent_albedo_kernel (daisy_world_rl.py:278-281) */
    double obs_mask[9];         /* env.neighborhood for kr=1 (daisy/nn/functional.py:93-103) */
} dw_config;

/* Luminosity clock: env.L, dL, min_L, max_L, ddL, step_count, ramp_period, ramp_up_down
   (daisy_world_rl.py:329-332, 463-473). Shared by every world of the handle. */
typedef struct dw_clock {
    double L, dL, min_L, max_L, ddL;
    int64_t step_count, ramp_period;
    int32_t ramp_up_down, _pad;
} dw_clock;

/* Result of dw_run. */
typedef struct dw_run_result {
    int64_t steps_run;        /* env steps executed */
    int64_t worlds_alive;     /* worlds with max(grid[:,1:3]) > 0.005 after the last step */
    int32_t all_done_hit;     /* 1 if the run stopped because every world was grid_done in one step */
    int32_t _pad;
} dw_run_result;

/* Launch accounting of a handle since dw_set_profiling(h, 1). fused_ms is device time of the fused lattice kernel
   measured with CUDA events on the handle's stream. */
typedef struct dw_profile {
    uint64_t kernel_launches;      /* every kernel this library launched */
    uint64_t fused_launches;       /* launches of the fused lattice kernel */
    uint64_t fused_cell_updates;   /* cell-updates those launches performed */
    double fused_ms;               /* their summed duration */
} dw_profile;

typedef struct dw_handle dw_handle;

int dw_abi_version(void);
const char *dw_last_error(const dw_handle *h);   /* h may be NULL: error of the last failed dw_create */

/* RLDaisyWorld.__init__ shapes + constants (daisy_world_rl.py:15-83). Fails if no CUDA device. */
int dw_create(const dw_config *cfg, dw_handle **out);
int dw_destroy(dw_handle *h);
/* attribute mutation after construction (env.albedo_dark = ..., env.dt = ...); shapes must not change */
int dw_set_config(dw_handle *h, const dw_config *cfg);
int dw_set_clock(dw_handle *h, const dw_clock *clk);
int dw_get_clock(dw_handle *h, dw_clock *clk);
/* luminosity the last forward pass used (the L behind env.temp / env.dead_temp, daisy_world_rl.py:403-416) */
int dw_get_last_L(dw_handle *h, double *L);
int dw_set_stream(dw_handle *h, void *cuda_stream);
/* Greedy.epsilon for DW_POLICY_EPS_GREEDY (0 = always greedy, 1 = always random; README's "half-random" is 0.5) */
int dw_set_epsilon(dw_handle *h, double epsilon);
/* MLP.set_parameters (daisy/agents/mlp.py:130-147) for DW_POLICY_MLP: host double[DW_MLP_PARAMS] */
int dw_set_mlp(dw_handle *h, const double *parameters, int32_t n_parameters);
/* ES fitness rollout, SimpleGaussianES.get_fitness (daisy/evo/sges.py:144-181), for a whole population at once: the batch
   is n_members contiguous blocks of batch/n_members worlds; in block m the first half of every world's agents acts with
   members[m], the second half with members[adversary_index] (DW_POLICY_MLP on both).  members: host
   double[n_members][DW_MLP_PARAMS]. */
int dw_set_mlp_population(dw_handle *h, const double *members, int32_t n_members, int32_t adversary_index);
/* Runs the rollout from the uploaded reset state until every member's loop has ended (all its agents done, or
   max_steps): per step the member's sum_reward += mean(reward[:, :half]) while its loop is alive. */
int dw_run_population(dw_handle *h, int64_t max_steps, int64_t *steps_run);
/* fitness[m] = sum_reward / (worlds_per_member * n_agents); member_steps[m] = env.step_count when member m's loop ended;
   total_steps[B, n] = per-agent (1 - done) counts up to that step (== done_at of get_fitness) */
int dw_get_population_results(dw_handle *h, double *fitness, int64_t *member_steps, int64_t *total_steps);

/* env.grid / env.agent_indices / env.agent_states assignment (any of the pointers may be NULL = keep).
   Host -> device; pinned host memory makes the copy asynchronous. */
int dw_upload_state(dw_handle *h, const double *grid, const int64_t *agent_indices, const double *agent_states);

/* initialize_grid's cover assignment (daisy_world_rl.py:304-312): grid = 0, ch1 = light[B,N,N], ch2 = dark[B,N,N]
   (host planes).  The narrow upload the reset()/ensemble paths use: the step reads nothing else of the grid. */
int dw_upload_covers(dw_handle *h, const double *light, const double *dark);

/* Device-side synthetic reset for ensembles too large to draw on the host: same distribution as initialize_grid /
   initialize_agents (daisy_world_rl.py:285-302,173-179) from a counter RNG keyed by (seed, global world index, cell);
   not stream-compatible with numpy. Channels 3..5 stay 0 until dw_init_temperatures. */
int dw_init_random(dw_handle *h, uint64_t seed, double light_proportion, double dark_proportion, double initial_al,
                   double initial_ad);

/* initialize_grid's field fill (daisy_world_rl.py:304-324): ch0 = p-l-d and ch3..5 = UNROUNDED T, T_light,
   T_dark of the uploaded covers at the current clock L. Called by reset() after dw_upload_state. */
int dw_init_temperatures(dw_handle *h);

/* RLDaisyWorld.step(action) (daisy_world_rl.py:475-497): update_agents -> forward -> get_obs -> reward/done -> update_L,
   all on the device, with ALL of its return values brought to the host by one copy.
   policy < 0: action is host int64 [ab,am] (ab<=B, am<=n), or NULL for step(None). Action values: ANY integer, read like
   the reference does (a == 8 stays, else a % 4 moves, a > 4 grazes; daisy_world_rl.py:190-212). Otherwise the action is
   chosen on the device by DW_POLICY_* (Greedy.__call__ or MLP.get_action fused in) and `action` is ignored.
   The state stays where the fused kernels keep it (packed 0.001 lattice, or the lean cover planes right after a reset)
   whenever the fast path covers the physics: one K = 1 launch of the fused kernel; the fp64 grid[B,7,N,N], the
   diagnostics and the observation windows are rebuilt on demand from the state the step started from. Partial actions
   (ab < B or am < n) and non-D4-symmetric kernels run the materialising kernels (64 B per cell).
   `out` receives the device's output block [reward f64 B*m | done u8 B*m, padded to a multiple of 8 | obs f64 B*n*63]
   (m = n, or 2 when n_agents == 0); byte offsets from dw_step_out_layout: layout[4] = {reward, done, obs, total bytes}.
   want_obs == 0 stops after the reward/done part (device policies do not need the observation on the host: at B = 1000,
   n = 4 it is 2 MB of the 2.04 MB). With `out` from dw_host_alloc (page-locked) the copy is a single DMA at PCIe rate.
   clk (may be NULL) receives the advanced clock. */
int dw_step_out_layout(dw_handle *h, int64_t *layout /*[4]*/);
int dw_step_packed(dw_handle *h, const int64_t *action, int32_t ab, int32_t am, int32_t policy, uint64_t seed,
                   int32_t want_obs, void *out, dw_clock *clk);
int dw_host_alloc(uint64_t bytes, void **out);
int dw_host_free(void *p);

/* Pieces of step(), exposed because callers use them standalone:
   RLDaisyWorld.update_agents(action) (:181-244) */
int dw_update_agents(dw_handle *h, const int64_t *action, int32_t ab, int32_t am);
/* collision_mode == 1 (daisy_world_rl.py:220-242, default off): where several agents share a cell after the moves, the
   reference draws npr.rand(1, n, 1) from the caller's GLOBAL NumPy stream per shared cell, in (world, x, y) scan order.
   The stream stays with the caller, so the step is split around the draws:
     dw_agents_begin    pay agent_gamma, move, graze (no clip yet); returns the post-move agent_indices [B,n,2] so that the
                        caller can count the shared cells of every world (integer bookkeeping only) and draw.
                        action, policy and seed as in dw_step_packed.
     dw_agents_collide  noise [cells, n] (the draws, in order), cell_offsets [B+1] (first draw of each world, [0] = 0):
                        resolves the collisions on the device (winner = resident with the largest state + 0.01 * noise,
                        gains food_chain_penalty * np.sum(other residents' states), losers keep theirs like :242) and
                        clips. Fails with DW_E_INVALID if a world's shared-cell count differs from the device's.
     dw_step_tail_packed   the rest of step(): forward, stamp, obs, reward/done, update_L; want_obs, out and clk as in
                        dw_step_packed.
   Every other stepping call returns DW_E_STATE between dw_agents_begin and dw_agents_collide. */
int dw_agents_begin(dw_handle *h, const int64_t *action, int32_t ab, int32_t am, int32_t policy, uint64_t seed,
                    int64_t *agent_indices);
int dw_agents_collide(dw_handle *h, const double *noise, const int32_t *cell_offsets, double food_chain_penalty);
int dw_step_tail_packed(dw_handle *h, int32_t want_obs, void *out, dw_clock *clk);
/* same tail for multi-step loops with collisions: advances the lifespan counters of dw_run (notebook cell 2) instead of
   collecting the outputs; *worlds_alive = worlds with max(grid[:,1:3]) > 0.005 after the step */
int dw_step_tail_counted(dw_handle *h, int64_t *worlds_alive);
/* RLDaisyWorld.forward(grid) (:434-461) on a caller grid (host in, host out) with the handle's agents/L;
   writes the mutated ch0 back into grid_in like the reference (:381). Does not advance the state. */
int dw_forward(dw_handle *h, double *grid_in, double *grid_out);
/* RLDaisyWorld.get_obs(agent_indices) (:246-263) at caller-supplied positions [b,m,2] -> obs[b,m,7,3,3] */
int dw_get_obs_at(dw_handle *h, const int64_t *agent_indices, int32_t b, int32_t m, double *obs);

/* Getters (device -> host, synchronise). */
int dw_get_grid(dw_handle *h, double *grid);                              /* env.grid */
/* fp32 mode (BASELINE.json north_star: "1e-5 in fp32 mode"): env.grid / the observations as binary32.
   Lattice-resident state (after fused steps / lattice-resident step()) with the fast path's constants: the grid is
   materialised with fp32 ARITHMETIC straight from the packed lattice (k_forward_f32: FFMA + MUFU.RSQ temperatures, 32 B of
   HBM traffic per cell instead of 64+). The covers (ch 1, 2) and the bare fraction (ch 0; fp32 evaluation screened by its
   error bound, fp64 fast path, then the literal cell) are the fp32 roundings of the reference's values; the temperatures
   (ch 3..5) are within ~5e-7 relative plus a possible 0.001 K rounding flip (3e-6). Any other state: the fp64
   materialisation converted to binary32 (2^-24 relative). Replaces reading RLDaisyWorld.grid (daisy_world_rl.py:434-461) /
   get_obs (:246-263) in a float32 pipeline. */
int dw_get_grid_f32(dw_handle *h, float *grid);                           /* [B,7,N,N] */
int dw_get_obs_f32(dw_handle *h, float *obs);                             /* [B,n,7,3,3] */
/* out[0] = cells materialised by the fp32-arithmetic path so far, out[1] = of those, cells whose bare fraction went on to the
   fp64 tier, out[2] = cells that needed the literal cell */
int dw_f32_stats(dw_handle *h, uint64_t *out /*[3]*/);
/* measurement hook: device time (CUDA events) of `reps` materialisations of the current lattice-resident state, fp32 != 0:
   k_forward_f32 (+ stamp), else the fp64 k_forward (+ stamp) */
int dw_debug_time_materialise(dw_handle *h, int32_t fp32, int32_t reps, double *ms_per_call);
int dw_get_agents(dw_handle *h, int64_t *agent_indices, double *agent_states);
int dw_get_obs(dw_handle *h, double *obs);                                /* obs of the last step / current state */
int dw_get_diag(dw_handle *h, int32_t which, double *out);                /* env.temp, env.beta_l, env.growth ... */
/* Ensemble statistics of one diagnostic field reduced on the device (what the notebooks compute with env.temp.mean(),
   notebook_helpers.py:50,145,218): out = {mean, population std, min, max} over all worlds and cells (both channels for
   DW_DIAG_GROWTH). Nothing but four doubles leaves the device. */
int dw_get_diag_stats(dw_handle *h, int32_t which, double *out /*[4]*/);
/* The same for the daisy covers of the current state: out = {mean light, mean dark, max light, max dark}. */
int dw_get_cover_stats(dw_handle *h, double *out /*[4]*/);

/* K fused steps with an on-device policy and the notebook lifespan counters
   (notebooks/greedy_longevity_abatement.ipynb cell 2): done_at[b] += !grid_done, agents_done_at[b,i] += !done.
   actions: host int8 [K,B,n] for DW_POLICY_REPLAY, else NULL.  stop_all_done: stop after the first step in
   which every world of this handle is grid_done (the notebook's loop condition). */
int dw_run(dw_handle *h, int64_t K, int32_t policy, const int8_t *actions, uint64_t seed, int32_t stop_all_done,
           dw_run_result *res);
/* Statistics-only variant of dw_run_chunk for lifespan ensembles (notebook cell 2 run for its counters only): the chunk may run
   past the stopping step; the kernels record per agent in which steps of the chunk it was not done, and
   dw_trim_lifespans(h, j) takes the steps after step j (0-based, the first step at which every world of every rank was
   grid_done) back out of agents_done_at. done_at needs no correction (every world stays done). No checkpoint, no replay; the
   lattice/agents/clock are left where the chunk ended. dw_trim_supported: *yes = 1 when the NEXT chunk can run this way
   (lattice-resident state, persistent kernel families, built-in policies); otherwise use dw_checkpoint_save + dw_run_chunk +
   dw_checkpoint_restore. */
int dw_trim_supported(dw_handle *h, int32_t policy, int32_t *yes);
int dw_run_chunk_masked(dw_handle *h, int32_t K, int32_t policy, const int8_t *actions, uint64_t seed, uint64_t *done_mask);
int dw_trim_lifespans(dw_handle *h, int32_t j);
/* Multi-rank variant: run exactly `K` (<=64) steps and return, per step, whether every world of THIS handle
   was grid_done (bit j of *done_mask = step j); the caller ANDs masks across ranks and decides. */
int dw_run_chunk(dw_handle *h, int32_t K, int32_t policy, const int8_t *actions, uint64_t seed, uint64_t *done_mask);
/* dw_run that also returns, for every step, the ensemble means the reference's plot helpers read (notebook_helpers.py:
   45-57): out[K][3] = {global mean of the unrounded temperature of that step's forward (env.temp.mean()), mean light cover,
   mean dark cover after the step}, reduced inside the fused kernel. K <= 4096. Shapes and configurations without an
   in-kernel series (see dw_run_series in csrc/dw_run.inl) fail with DW_E_UNSUPPORTED before any step has run. */
int dw_run_series(dw_handle *h, int64_t K, int32_t policy, const int8_t *actions, uint64_t seed, double *out);
int dw_reset_lifespans(dw_handle *h);
int dw_get_lifespans(dw_handle *h, int64_t *done_at /*[B]*/, int64_t *agents_done_at /*[B,n]*/);
/* Ensemble statistics of the lifespan counters on the DEVICE, for an NCCL all-reduce by the caller:
   out_dev (device pointer, 8 doubles) = {count, sum life, sum life^2, n_agents_total, sum agent_life,
   sum agent_life^2, worlds_alive, 0}. */
int dw_lifespan_stats_device(dw_handle *h, double *out_dev);

/* Device-side state checkpoint (grid/lattice, agents, clock, counters): used to rewind a chunk and by the
   benchmark to restart from the same initial state without host traffic. */
int dw_checkpoint_save(dw_handle *h);
int dw_checkpoint_restore(dw_handle *h);

int dw_synchronize(dw_handle *h);

/* Multi-rank ensembles: global index of this handle's first world (only feeds the DW_POLICY_RANDOM counter RNG). */
int dw_set_world_offset(dw_handle *h, uint32_t world0);

int dw_set_profiling(dw_handle *h, int32_t on);      /* resets the counters */
int dw_get_profile(dw_handle *h, dw_profile *out);

/* Diagnostics of the fused path (tests / profiling): number of cells recomputed in literal order because the fast
   path landed within the tie filter; and the fast fourth root evaluated on the device (host in, host out). */
int dw_debug_slow_count(dw_handle *h, uint64_t *count, int32_t reset);
/* where the live state currently resides: flags[4] = {fp64 grid[B,7,N,N] valid, packed lattice valid, lean reset planes
   valid, kind of the recorded pre-state (0 none, 1 grid, 2 lattice, 3 cover planes)}. Tests use it to check that step()
   stays lattice-resident. */
int dw_debug_state(dw_handle *h, int32_t *flags /*[4]*/);
int dw_debug_root4(dw_handle *h, const double *x, double *y, int32_t n);
/* test hook of the screened materialising kernels: over a host grid [B,7,N,N] (channels 1,2 read) at the handle's clock,
   out[0..2] = largest |screened - literal| * 1000 of the unrounded new covers, bare fraction and temperatures over the
   cells inside the screened range, out[3..5] = the tie-filter half-widths they must stay below */
int dw_debug_screen_error(dw_handle *h, const double *grid, double *out);
/* number of integers k in [-kmax,kmax] for which the division-free k/1000 used by the kernels differs from the IEEE
   quotient (must be 0) */
int dw_debug_markstein(dw_handle *h, uint32_t kmax, uint32_t *bad);
/* the binary32 twin used by the fp32 mode (dw_div1000f): integers |k| <= kmax whose division-free k/1000 differs from the
   correctly rounded quotient; exact up to 2^19 */
int dw_debug_markstein_f32(dw_handle *h, uint32_t kmax, uint32_t *bad);
/* Measured FP64 FMA peak of the handle's device (dependent DFMA chains, full occupancy): best of `reps` launches of
   `iters` x 8 FMAs per thread, in TFLOP/s (FMA = 2 flop).  Roofline denominator of the fused kernel. */
int dw_debug_fp64_peak(dw_handle *h, int32_t iters, int32_t reps, double *tflops_best, double *ms_best);

#ifdef __cplusplus
}
#endif
#endif /* DAISYWORLD_B200_H */
