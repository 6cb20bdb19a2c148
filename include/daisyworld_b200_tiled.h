/*
 * daisyworld_b200_tiled.h -- C ABI of the single-giant-grid path (BASELINE config 5): ONE toroidal N x N RLDaisyWorld
 * (batch_size == 1, daisy/daisy_world_rl.py:13-501) too large for shared memory, optionally split into row bands, one
 * band per GPU.  Same conventions as daisyworld_b200.h (return codes, ownership, stream semantics, no CPU fallback).
 *
 * A handle owns rows [row0, row0 + rows) of the world (rows == N: the whole torus on one GPU) plus one ghost row above
 * and below.  Agents are replicated: every rank holds all n agents (global coordinates) and runs the same agent
 * kernels; only the rank that owns a cell eats from it.
 *
 * One env step (daisy_world_rl.py:475-497) is the phase sequence below.  With several ranks the caller sums two small
 * device vectors across ranks between phases and copies two halo rows to the neighbours after the stencil
 * (therldaisyworld_b200/banded.py does this with torch.distributed: NCCL on GPUs, gloo in the CPU tests):
 *
 *   dwt_decide        Greedy.__call__ (agents/greedy.py:16-30) or replay/none/random, owner rank only -> act[n]
 *                     [ranks > 1 and greedy/antigreedy: all-reduce SUM of act]
 *   dwt_move_graze    update_agents (:181-216): pay agent_gamma, move, graze in agent-index order -> gain[n]
 *                     [ranks > 1: all-reduce SUM of gain]
 *   dwt_finish_agents state += gain, clip (:244), agents_done_at += !done; reward and done (:486-492) follow from
 *                     the states (dwt_get_agents)
 *   dwt_stencil       forward (:434-452) on the band -> new covers (ghost columns included); update_L (:463-473);
 *                     per-step species max. Parts 1 + 2 split it into edge tile rows and interior so that the
 *                     halo exchange can overlap the interior.
 *   ghost rows        toroidal wrap (dwt_halo_wrap, one rank) or the neighbours' edge rows (caller copies whole
 *                     stored rows of dwt_get_pitch words).
 * gain[n] and act[n] are adjacent in memory (gain first): finishing step j can be deferred until the decisions of
 * step j + 1 exist, so that ONE all-reduce per step carries both (therldaisyworld_b200/banded.py does that).
 *
 * Observations and DW_POLICY_MLP: once a step's agents are finished, dwt_observe writes the band's PARTIAL observation of
 * the current state, obs[n, 7, 3, 3] -- step()'s obs[0] (daisy_world_rl.py:494) for the window cells in rows this band
 * owns, 0 elsewhere -- into a device buffer (dwt_get_obs_ptr).  With several ranks the caller sums it across ranks (one
 * non-zero term per element, like act); with one rank it is already the whole observation.  dwt_decide(DW_POLICY_MLP)
 * then maps that buffer to every agent's action on every rank, so an MLP step needs no act exchange:
 *
 *   dwt_finish_agents (step j - 1) -> dwt_observe [ranks > 1: all-reduce SUM of obs] -> dwt_decide(DW_POLICY_MLP)
 *   -> dwt_move_graze -> dwt_stencil ...
 *
 * Peer-memory mode (dwt_step_p2p) refuses DW_POLICY_MLP; dwt_observe works there after dwt_flush_p2p.
 *
 * Diagnostics (dwt_get_diag, dwt_get_diag_stats, dwt_get_cover_stats, dwt_pool): the unrounded fields of the last step's
 * forward, their statistics and block sums for images, reduced on the device per band; see the section below.
 *
 * Snapshots (dwt_save_state, dwt_restore_state): a band's whole state out to the host and back, exactly, between steps; a
 * snapshot of one banding restores on any other, because the state is the same integer lattice whatever the banding. See
 * the section below.
 *
 * Constraints of the tiled kernels: N >= 64, 8 <= rows <= N, D4-symmetric kernels (the defaults). Bands may differ in
 * height; a side or band that is not a multiple of 64 runs a masked instance of the stencil kernel over its partial tiles.
 */
#ifndef DAISYWORLD_B200_TILED_H
#define DAISYWORLD_B200_TILED_H

#include "daisyworld_b200.h"

#ifdef __cplusplus
extern "C" {
#endif

typedef struct dwt_handle dwt_handle;

/* Device pointers a multi-rank driver needs (valid until the next dwt_stencil for the halo rows, for the life of the
   handle for the rest). Row pointers address a whole stored row of dwt_get_pitch packed u32 words (light milli-cover |
   dark << 16; words 4 .. N + 3 are the N columns, word 3 and word N + 4 the ghost columns, the rest is padding). */
typedef struct dwt_ptrs {
    double *act;            /* [n]   action + 1 per agent (0 = not decided here); act == gain + n */
    double *gain;           /* [n]   food eaten per agent on this rank */
    int32_t *stepmax;       /* [4096, 2] per-step max milli-cover of (light, dark) over this band */
    uint32_t *send_top;     /* band row 0 (whole stored row)              -> the rank above's bottom ghost */
    uint32_t *send_bottom;  /* band row rows-1                            -> the rank below's top ghost */
    uint32_t *recv_top;     /* ghost row above the band */
    uint32_t *recv_bottom;  /* ghost row below the band */
} dwt_ptrs;

const char *dwt_last_error(const dwt_handle *h);
/* cfg->dim = N, cfg->n_agents = n, cfg->batch must be 1; rows/row0: the band of this handle; n_ranks: number of bands */
int dwt_create(const dw_config *cfg, int32_t rows, int32_t row0, int32_t n_ranks, dwt_handle **out);
int dwt_destroy(dwt_handle *h);
/* New constants for the handle. Refuses with DW_E_UNSUPPORTED what dwt_create refuses (the tiled kernels need D4-symmetric
   kernels, a zero-centre uniform albedo kernel and g > 0) and keeps the old configuration then. */
int dwt_set_config(dwt_handle *h, const dw_config *cfg);
int dwt_set_clock(dwt_handle *h, const dw_clock *clk);
int dwt_get_clock(dwt_handle *h, dw_clock *clk);
int dwt_set_stream(dwt_handle *h, void *cuda_stream);
int dwt_set_epsilon(dwt_handle *h, double epsilon);       /* for DW_POLICY_EPS_GREEDY, see dw_set_epsilon */
int dwt_synchronize(dwt_handle *h);

/* reset(): cover planes of the band INCLUDING its two ghost rows, host fp64 [(rows + 2), N] each (row 0 = world row
   row0 - 1 with toroidal wrap); the state is off the 0.001 lattice until the first step (daisy_world_rl.py:299-302). */
int dwt_upload_covers(dwt_handle *h, const double *light, const double *dark);
/* all n agents, global coordinates: agent_indices[n,2] int64, agent_states[n] */
int dwt_upload_agents(dwt_handle *h, const int64_t *agent_indices, const double *agent_states);
/* device-side synthetic reset (distribution of initialize_grid/initialize_agents, counter RNG keyed by the global cell /
   agent index: every banding of the same world gets the same state) */
int dwt_init_random(dwt_handle *h, uint64_t seed, double light_proportion, double dark_proportion, double initial_al,
                    double initial_ad);

/* phases of one step (see the header comment). actions: host int8 [n] for DW_POLICY_REPLAY, else NULL.
   DW_POLICY_MLP reads the observation buffer: it needs dwt_set_mlp (else DW_E_STATE) and a dwt_observe since the last
   change of state -- step phase, upload, reset, dwt_set_config (else DW_E_STATE). */
int dwt_decide(dwt_handle *h, int32_t policy, const int8_t *actions, uint64_t seed);
int dwt_move_graze(dwt_handle *h);
int dwt_finish_agents(dwt_handle *h);
int dwt_stencil(dwt_handle *h, int32_t part);   /* 0: whole band; 1: edge tile rows, then 2: interior tile rows */
int dwt_halo_wrap(dwt_handle *h);      /* one rank: ghost rows from the band's own edge rows */
int dwt_get_ptrs(dwt_handle *h, dwt_ptrs *out);
/* words per stored row: 64 * ceil(N / 64) + 8 (N + 8 when N is a multiple of 64), a multiple of 16 bytes */
int dwt_get_pitch(const dwt_handle *h, int32_t *pitch);

/* ---- observations and the MLP policy (see the header comment) ---------------------------------------------------------
 * dwt_observe: the band's partial observation obs[n, 7, 3, 3] of the current state -> the device buffer, on the handle's
 * stream. The window is the 3x3 around each agent's current position, all 7 channels (ch4: the state of the highest-index
 * agent on the cell, dead agents included, after the step), times dw_config.obs_mask. Right after a reset, before any
 * step, it shows initialize_grid's unrounded fields at the current L with no agent stamp. DW_E_STATE before any state
 * exists, after dwt_debug_time_stencil (until the next step), and while a step's agents are not finished (between
 * dwt_move_graze and dwt_finish_agents; in peer-memory mode until dwt_flush_p2p). The buffer is allocated on first use. */
int dwt_observe(dwt_handle *h);
int dwt_get_obs_ptr(dwt_handle *h, double **obs /* device [n, 7, 3, 3] */);
int dwt_get_obs(dwt_handle *h, double *out /* host [n, 7, 3, 3] */);         /* synchronises */
/* MLP.set_parameters (daisy/agents/mlp.py:130-147) for DW_POLICY_MLP: host double[DW_MLP_PARAMS], as dw_set_mlp */
int dwt_set_mlp(dwt_handle *h, const double *parameters, int32_t n_parameters);

/* K whole steps on one rank (rows == N): the phases above back to back on the handle's stream, no host sync.
   DW_POLICY_MLP runs dwt_observe before each decision. */
int dwt_run(dwt_handle *h, int64_t K, int32_t policy, const int8_t *actions /*[K,n] or NULL*/, uint64_t seed);
/* Close a chunk of `K` steps whose per-step maxima sit in stepmax (all-reduced MAX over ranks by the caller when there
   are several): done_at += #steps whose max(light, dark) > 5 (notebook cell 2: grid_done = max <= 0.005);
   first_all_done = first step index of the chunk with the world done, or -1. Clears stepmax and the series rows. */
int dwt_end_chunk(dwt_handle *h, int32_t K, int32_t *first_all_done);
int dwt_reset_lifespans(dwt_handle *h);
int dwt_get_lifespans(dwt_handle *h, int64_t *done_at /*[1]*/, int64_t *agents_done_at /*[n]*/);

/* ---- climate series: per-step sums over the band's own cells, reduced inside the stencil kernels -----------------------
 * With series mode on, step j of a chunk adds to row j of a device buffer [4096, 3] (doubles):
 *   column 0: sum of sqrt(g) * T, T the unrounded global temperature of the step's forward (the reference's env.temp);
 *   columns 1, 2: sum of the new light / dark milli-covers (1000 * cover; integers, exact and order-independent in fp64).
 * Ghost rows and columns never count, so the rows are additive over the bands of a world: a multi-rank caller all-reduces
 * (SUM) the K rows of dwt_get_series_ptr before dwt_get_series. dwt_end_chunk, dwt_upload_covers and dwt_init_random clear
 * the rows. Switching series mode while a chunk is open fails with DW_E_STATE; it needs g > 0 (DW_E_UNSUPPORTED). */
int dwt_set_series(dwt_handle *h, int32_t on);
int dwt_get_series_ptr(dwt_handle *h, double **series /* device [4096, 3] */);
/* [K, 3] host: sum of T (kelvin), sum of milli-light, sum of milli-dark of the chunk's first K steps; call before
   dwt_end_chunk. Synchronises. */
int dwt_get_series(dwt_handle *h, int32_t K, double *out);

/* ---- peer-memory mode: one process per GPU, no collective on the step path -----------------------------------------
 * Every rank maps every other rank's exchange vector, barrier flags and lattice buffers (CUDA IPC over NVLink/NVSwitch).
 * The owner band of an agent / the winner of a graze stores its result straight into ALL ranks' exchange vectors
 * (exactly one writer per entry: nothing to reduce), a band pushes its edge rows into the neighbours' ghost rows, and
 * ranks meet at device-side flag barriers. dwt_step_p2p is one env step; every rank calls it in lock-step.
 * Setup: dwt_ipc_export on every rank -> all-gather the blobs (any transport) -> dwt_ipc_attach. */
#define DWT_IPC_HANDLE_BYTES 64
#define DWT_PEER_BUFFERS 4          /* lattice buffer 0, lattice buffer 1, exchange vector, barrier flags */
int dwt_ipc_export(dwt_handle *h, void *handles /* [DWT_PEER_BUFFERS][DWT_IPC_HANDLE_BYTES] */);
int dwt_ipc_attach(dwt_handle *h, int32_t rank, int32_t n_ranks, const void *all_handles /* [n_ranks][4][64] */);
/* same-process variant (several bands of one process, tests): raw device pointers [n_ranks][DWT_PEER_BUFFERS] */
int dwt_get_peer_buffers(dwt_handle *h, void **out /* [DWT_PEER_BUFFERS] */);
int dwt_attach_peers(dwt_handle *h, int32_t rank, int32_t n_ranks, void *const *table);
/* Both attach calls also allocate the fp64 reset planes (otherwise allocated by the first dwt_upload_covers /
   dwt_init_random), so that no band of a peer-memory world allocates device memory once any band may be stepping. */
/* rows[n_ranks]: the band height of every rank, in rank order (they add up to N). Needed before either attach call when
   the bands differ in height: a band writes its last row into the ghost row below its upper neighbour's band. Without
   it, attaching assumes equal bands and refuses with DW_E_STATE when rows * n_ranks != N. */
int dwt_set_peer_rows(dwt_handle *h, int32_t n_ranks, const int32_t *rows);
/* DW_POLICY_MLP: DW_E_UNSUPPORTED, before anything is launched */
int dwt_step_p2p(dwt_handle *h, int32_t policy, const int8_t *actions /* [n] or NULL */, uint64_t seed);
int dwt_flush_p2p(dwt_handle *h);                       /* finish the agents of the last step */
int dwt_peer_status(dwt_handle *h, int32_t *timed_out); /* 1 if a barrier gave up waiting for a peer */

/* getters (synchronise) */
int dwt_get_agents(dwt_handle *h, int64_t *agent_indices, double *agent_states);
int dwt_get_covers(dwt_handle *h, double *light, double *dark);                 /* band rows, [rows, N] each */
/* env.grid of the band: [7, rows, N] (channels as in the reference; ch4 carries the agent stamp), materialised by a
   literal forward from the post-graze state the last step started from. Needs at least one step. */
int dwt_get_grid(dwt_handle *h, double *grid);
/* Position-weighted checksum of the band's own cells, computed on the device with exact integer arithmetic (mod 2^64):
   out[4] = {sum kl, sum kd, sum kl*w, sum kd*w} over the milli-covers k = 1000 * cover, w = (global_row * 131 + column)
   % 977 + 1. Additive over bands: the sum over the ranks of a banded world equals the checksum of the same world on one
   GPU (bench.py prints it so that the 1/2/4/8-GPU runs can be compared; the reference quantity is env.grid[0, 1:3]). */
int dwt_cover_checksum(dwt_handle *h, uint64_t *out /*[4]*/);
int dwt_debug_slow_count(dwt_handle *h, uint64_t *count);
/* Measurement hook: average duration (microseconds, CUDA events) of `reps` back-to-back launches of the band's stencil
   kernel on the current state -- the compute floor of one step, against which bench.py states the per-step exchange /
   agent overhead. Overwrites the recorded pre-state (dwt_get_grid needs a new step afterwards). Always times the kernel
   with series mode off and records nothing into the series rows. */
int dwt_debug_time_stencil(dwt_handle *h, int32_t reps, double *us_per_launch);

/* ---- diagnostics and plot feed (what the reference's notebook helpers read: env.temp.mean(), the covers, images) ---------
 * The fields are the unrounded side effects of the last step's forward, as dw_get_diag defines them (DW_DIAG_* selectors),
 * evaluated like dwt_get_grid: a literal forward of the post-graze pre-state that step started from, at S * L of that step.
 * Nothing but the requested result is allocated: statistics and images are reduced on the device while the field is
 * evaluated (per-CTA partials, then one block, in a fixed order: the same banding returns the same bits on every call).
 * The results are the band's own part; a multi-rank caller merges them (banded.py: one SUM all-reduce per call).
 * DW_E_STATE without a pre-state (before the first step after an upload / reset, after dwt_debug_time_stencil) and while a
 * step's agents are not finished (as dwt_observe); DW_E_INVALID for a bad selector or block size.
 * Reading the pre-state races with the next step's halo push in peer-memory mode: a caller meets every rank (any
 * collective) after these calls and before the next dwt_step_p2p. */
/* dwt_pool field selectors: DW_DIAG_TEMP .. DW_DIAG_BETA_D, the two planes of DW_DIAG_GROWTH, and the grid channels
   0, 1, 2, 3, 5 of dwt_get_grid (rounded b', light, dark, rounded T, rounded T_d) */
enum {
    DWT_FIELD_TEMP = 0, DWT_FIELD_TEMP_LIGHT = 1, DWT_FIELD_TEMP_DARK = 2, DWT_FIELD_TEMP_EFFECTIVE = 3,
    DWT_FIELD_BETA = 4, DWT_FIELD_BETA_L = 5, DWT_FIELD_BETA_D = 6, DWT_FIELD_GROWTH_L = 7, DWT_FIELD_GROWTH_D = 8,
    DWT_FIELD_GRID_BARE = 9, DWT_FIELD_GRID_LIGHT = 10, DWT_FIELD_GRID_DARK = 11, DWT_FIELD_GRID_TEMP = 12,
    DWT_FIELD_GRID_TEMP_DARK = 13
};
/* the band's field [rows, N] (DW_DIAG_GROWTH: [2, rows, N], dl then dd) -> host; uses the dwt_get_grid scratch. Synchronises. */
int dwt_get_diag(dwt_handle *h, int32_t which, double *out);
/* out[5] = {count, mean, m2, min, max} of a DW_DIAG_* field over the band's own cells (growth: both planes, 2 * rows * N
   values), m2 = sum (x - mean)^2 about the band's mean. Synchronises. */
int dwt_get_diag_stats(dwt_handle *h, int32_t which, double *out);
/* out[4] = {sum light, sum dark, max light, max dark} over the band's own cells of the CURRENT state (also right after a
   reset); exact on the lattice (integer milli-covers). Synchronises. */
int dwt_get_cover_stats(dwt_handle *h, double *out);
/* Block sums of a DWT_FIELD_* field over the cells this band owns -> device buffer [H, H], H = ceil(N / block), 1 <= block
   <= N: entry (i, j) sums global rows and columns [i * block, min((i + 1) * block, N)) x [j * block, ...); every entry is
   written (0 where the band owns nothing), so the SUM over the ranks is the whole world's block sums. Dividing by the
   cells of each block (fewer at the edges when block does not divide N) gives the block-averaged image. On the handle's
   stream; the buffer is allocated on first use and grows with H. */
int dwt_pool(dwt_handle *h, int32_t field, int32_t block);
int dwt_get_pool_ptr(dwt_handle *h, double **pool /* device [H, H] */, int32_t *H);
int dwt_get_pool(dwt_handle *h, double *out /* host [H, H] */);               /* synchronises */
/* L of the last step's forward (the L of the reset before any step), for the bare-planet temperature; as dw_get_last_L */
int dwt_get_last_L(dwt_handle *h, double *L);

/* ---- fp32 mode: the band's grid as float32, evaluated with fp32 arithmetic from the lattice ------------------------------
 * The grid of dwt_get_grid, [7, rows, N] float32 (ch4: the agent stamp), the giant world's counterpart of dw_get_grid_f32:
 * the temperatures (channels 3..5) are evaluated in binary32 from the post-graze pre-state at S * L of the last step (within
 * 1e-5 relative of the fp64 grid), the bare fraction is screened against a proven fp32 error bound and otherwise finished by
 * the fp64 fast path and the literal cell, so channels 0, 1, 2 and 6 are the exact binary32 roundings of dwt_get_grid's.
 * 36 bytes of device memory traffic per cell against 64 or more for the fp64 grid, and no fp64 scratch. Right after the
 * first step of a reset or upload (the pre-state is the fp64 planes) the fp64 grid is converted, exactly
 * dwt_get_grid's values rounded to float32; those cells do not count in dwt_f32_stats.
 * DW_E_STATE without a pre-state (before the first step after an upload / reset / restore of a snapshot without one, after
 * dwt_debug_time_stencil), while a step's agents are not finished (between dwt_move_graze and dwt_finish_agents; in
 * peer-memory mode until dwt_flush_p2p) and after a failed dwt_restore_state; DW_E_INVALID for NULL pointers.
 * Reading the pre-state races with the next step's halo push in peer-memory mode: a caller meets every rank (any
 * collective) after these calls and before the next dwt_step_p2p. */
/* materialise into the device buffer float [7, rows, N] (allocated on first use, 28 bytes per band cell) on the handle's
   stream, without synchronising; the buffer is overwritten by the next call */
int dwt_grid_f32(dwt_handle *h);
int dwt_get_grid_f32_ptr(dwt_handle *h, float **grid /* device [7, rows, N] */);
int dwt_get_grid_f32(dwt_handle *h, float *out /* host [7, rows, N] */);     /* dwt_grid_f32 + download; synchronises */
/* out[3] = {cells evaluated with fp32 arithmetic, cells whose bare fraction went on to the fp64 tier, cells that needed the
   literal cell}, cumulative over the handle's life. Synchronises. */
int dwt_f32_stats(dwt_handle *h, uint64_t *out /*[3]*/);
/* Measurement hook: average device time (microseconds, CUDA events) of `reps` back-to-back materialisations after one
   warm-up: fp32 != 0 the work of dwt_grid_f32, fp32 == 0 that of dwt_get_grid without its download. Refuses like
   dwt_grid_f32. */
int dwt_debug_time_materialise(dwt_handle *h, int32_t fp32, int32_t reps, double *us_per_call);

/* ---- snapshots: a band's state out of and back into a handle, exactly --------------------------------------------------
 * A band's state is its current state, the pre-state the last step started from (observations, DW_POLICY_MLP and the
 * diagnostics read it), L_last, done_at and agents_done_at; the agents and the clock have their own getters and setters.
 * Each of the two states is held in one representation:
 *   DWT_REP_LATTICE  packed u32 words (light milli-cover | dark << 16), row by row, N words per row, no padding;
 *   DWT_REP_PLANES   fp64 covers [2][rows][N] (light plane, then dark): the off-lattice state of a reset or upload;
 *   DWT_REP_NONE     absent (the pre-state right after a reset or upload, and after dwt_debug_time_stencil).
 * The current state is planes until the first step and the lattice after it; the pre-state is none, then the planes after
 * the first step, then the lattice. None of it depends on the banding, so a snapshot taken on one partition of the world
 * can be restored on any other. */
enum { DWT_REP_NONE = 0, DWT_REP_PLANES = 1, DWT_REP_LATTICE = 2 };
typedef struct dwt_band_state {
    int32_t cur_rep, pre_rep;   /* DWT_REP_* of the current state and of the pre-state */
    double L_last;              /* dwt_get_last_L */
    int64_t done_at;            /* dwt_get_lifespans */
    uint64_t cur_bytes;         /* bytes of cur_rows of dwt_save_state (the band's own rows); 0 for DWT_REP_NONE */
    uint64_t pre_bytes;         /* bytes of pre_rows of dwt_save_state */
} dwt_band_state;
/* The band's state -> host. meta always receives the representations, L_last, done_at and the byte sizes, so a first call
   with NULL rows sizes the buffers. cur_rows / pre_rows (when not NULL) receive the band's OWN rows [rows][N] in their
   representation, agents_done_at (when not NULL) n counters. Staged through a page-locked buffer of the handle (about
   (rows + 2) * N * 4 bytes, allocated on first use). DW_E_STATE while the snapshot would not be a whole step: between
   dwt_move_graze and dwt_finish_agents, in peer-memory mode before dwt_flush_p2p, and while a chunk is open (call
   dwt_end_chunk first). Synchronises. */
int dwt_save_state(dwt_handle *h, dwt_band_state *meta, void *cur_rows, void *pre_rows, int64_t *agents_done_at);
/* Replaces the band's state. cur_rows / pre_rows hold the band's rows WITH both ghost rows, global rows row0 - 1 .. row0 +
   rows (toroidal), i.e. rows + 2 rows in the representation meta names (pre_rows is ignored for DWT_REP_NONE); the ghost
   columns are written on the device, so no exchange between bands is needed. Sets L_last, done_at and agents_done_at[n]
   (NULL: zero), drops any look-ahead decisions and observation, returns the claim arrays to idle and clears the per-step
   maxima and series rows. Keeps the lattice buffer parity (every rank of a peer-memory world must keep the same one).
   Allocates the fp64 planes when the snapshot holds planes. DW_E_INVALID for an unknown representation or a pair that
   cannot occur (the pre-state is at most one step behind); DW_E_STATE while a step's agents are not finished (as
   dwt_save_state). In peer-memory mode every rank meets every other (any collective) before and after this call. If it fails
   after its checks (a copy or an allocation), the band's old state is partly overwritten: every call that reads the state
   then fails with DW_E_STATE until dwt_upload_covers, dwt_init_random or a successful dwt_restore_state. Synchronises. */
int dwt_restore_state(dwt_handle *h, const dwt_band_state *meta, const void *cur_rows, const void *pre_rows,
                      const int64_t *agents_done_at);
/* dwt_cover_checksum of the pre-state when it is on the lattice (DW_E_STATE otherwise) */
int dwt_pre_checksum(dwt_handle *h, uint64_t *out /*[4]*/);

#ifdef __cplusplus
}
#endif
#endif /* DAISYWORLD_B200_TILED_H */
