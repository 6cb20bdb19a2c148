// C-ABI implementation (include/daisyworld_b200.h): handle management, state residency, launches.
// Build: nvcc -gencode arch=compute_100a,code=sm_100a -fmad=false -lineinfo (therldaisyworld_b200/build.py)
#include <cstdarg>
#include <cstdlib>
#include <cstdio>
#include <cstring>
#include <string>
#include <vector>

#include "dw_common.cuh"
#include "dw_generic.cuh"
#include "dw_fused.cuh"
#include "dw_f32.cuh"

static thread_local std::string g_create_error;

enum PreKind { PRE_NONE = 0, PRE_GRID = 1, PRE_LAT = 2, PRE_COV = 3 };

// What a fused launch does besides the steps: nothing, record the per-step series (dw_run_series), or run DW_POLICY_MLP
enum FusedMode { FUSED_PLAIN = 0, FUSED_SERIES = 1, FUSED_MLP = 2, FUSED_MODES = 3 };

// One fused kernel instance: a row of the table in fused_kernel (dw_run.inl)
struct FusedKernel {
    void (*kern)(const FusedArgs) = nullptr;   // nullptr: no fused kernel runs this mode at this shape
    int threads = 256;
    size_t smem = 0;                           // dynamic shared memory per CTA
    bool persistent = false;                   // resident CTAs share a (worlds, step chunk) queue; else one CTA per world
    int worlds = 1;                            // worlds per work item
    bool trim = false;                         // records alive_mask (dw_run_chunk_masked)
    int blocks = 0;                            // resident CTAs of a persistent kernel on the handle's device (resolve_fused)
};

struct dw_handle {
    dw_config cfg{};
    dw_clock clk{};
    cudaStream_t stream = nullptr;
    std::string err;
    size_t NN = 0;

    // fp64 materialised representation (allocated lazily: pure ensemble runs never need it)
    double *grid[2] = {nullptr, nullptr};
    int cur = 0;
    bool grid_valid = false;
    bool ch6_dirty[2] = {false, false};
    // lean reset state: fp64 cover planes [B,2,N,N] (light, dark), off the 0.001 lattice; the 7-channel grid of such a
    // state (ch0, initial temperatures) is only materialised when a caller asks for it
    double *cov = nullptr;
    bool cov_valid = false;
    double cov_L = 0.0;                 // luminosity of initialize_grid's temperature fill (dw_init_temperatures)
    // packed lattice representation [B,N,N]
    uint32_t *lat[2] = {nullptr, nullptr};
    int lcur = 0;
    bool lat_valid = false;
    // state the last forward started from (post-graze): source of diagnostics / lazy materialisation
    PreKind pre = PRE_NONE;
    const double *pre_grid = nullptr;   // points into grid[] or fwd scratch
    uint32_t *lat_pre = nullptr;
    double L_last = 0.0;

    int32_t *agent_xy = nullptr;
    long long *agent_idx64 = nullptr;   // staging of uploaded int64 agent_indices (converted on the device: no host sync)
    double *agent_state = nullptr;
    // step outputs in ONE device block, layout [reward f64 B*m | done u8 B*m (padded to 8) | obs f64 B*n*63], m = n or 2
    // when n_agents == 0: dw_step_packed brings all of step()'s return values to the host with a single copy. The
    // observation part is allocated on first use (ensembles that never ask for observations keep the block small).
    unsigned char *out_block = nullptr;
    bool out_full = false;
    double *obs = nullptr;
    bool obs_valid = false;
    double *reward = nullptr;
    uint8_t *done = nullptr;
    bool count_life = true;                    // fused / lean launches add their steps to the lifespan counters (dw_run); step() does not
    // diagnostics of a standalone dw_forward(grid) call (env.forward refreshes env.temp/beta/growth as a side effect)
    // live in their own slot: the pre-state of the LIVE state is not touched (the reference's forward leaves the env alone)
    bool fwd_diag = false;
    double fwd_L = 0.0;
    unsigned long long *world_max = nullptr;   // [B,2]
    int64_t *done_at = nullptr, *agents_done_at = nullptr;
    unsigned int *alive = nullptr;             // [64] per-step alive-world counters of a chunk
    int8_t *action_dev = nullptr;
    size_t action_cap = 0;
    double *scratch = nullptr;                 // diag / forward scratch
    size_t scratch_cap = 0;
    double *fwd_in = nullptr, *fwd_out = nullptr;
    unsigned int *slow_count = nullptr;        // [0] literal recomputations in fused runs, [1] scratch counter
    // fp32 mode (dw_f32.cuh): float [B,7,N,N] grid materialised with fp32 arithmetic, tier counters {fp64-tier cells, literal cells}
    float *grid32 = nullptr;
    unsigned long long *f32_stats = nullptr;
    unsigned long long f32_cells = 0;          // cells materialised by the fp32 path so far
    unsigned int world0 = 0;                   // global index of the first world (multi-rank ensembles)
    double epsilon = 0.0;                      // Greedy.epsilon of DW_POLICY_EPS_GREEDY
    // series mode of the fused kernel (dw_run_series)
    bool series_on = false;
    int64_t series_pos = 0;
    double *series_T = nullptr;
    unsigned long long *series_l = nullptr, *series_d = nullptr;
    double *mlp_dev = nullptr;                 // [DW_MLP_PARAMS] weights of DW_POLICY_MLP, or [n_members][DW_MLP_PARAMS]
    size_t mlp_cap = 0;
    bool mlp_set = false;
    // population mode (ES fitness rollouts): members own contiguous blocks of worlds
    int pop_members = 0, pop_adversary = 0;
    double *pop_sum = nullptr;                 // [members] sum_reward
    int *pop_done = nullptr;                   // [members] loop ended
    int64_t *pop_steps = nullptr, *pop_frozen = nullptr;   // [members] step count at the end; [B,n] frozen (1-done) counters
    unsigned int *pop_ndone = nullptr;
    unsigned char *pin = nullptr;              // pinned host staging of a step's explicit action bytes (stage_action)
    bool agents_open = false;                  // between dw_agents_begin and dw_agents_collide the agent states are unclipped
    StepCoef *sc_dev = nullptr;                // per-step coefficient table of a fused launch
    std::vector<dw_clock> sc_clk;              // clock before each step of the table on the device (+ the one after the last)
    int sc_policy = -1;                        // what the cached table was built for (launch_fused)
    uint64_t sc_seed = 0;
    double sc_eps = 0.0;
    dw_config sc_cfg{};
    unsigned int *persist_sync = nullptr;      // [1 + B] work queue + per-world progress of the persistent kernel
    FusedKernel fused[FUSED_MODES];            // kernel of each fused mode, resolved on the mode's first launch (resolve_fused)
    bool fused_ready[FUSED_MODES] = {};
    // statistics-only lifespan runs (dw_run_chunk_masked / dw_trim_lifespans): per-agent "not done" bits of the last chunk
    unsigned long long *alive_mask = nullptr;
    bool mask_on = false, mask_complete = false;
    double *pop_rew = nullptr;                 // [64][B*n] per-step agent states of a fused population segment (k_pop_post)
    bool pop_rew_on = false;
    // profiling (dw_set_profiling): kernel launch count, and device time of the fused kernel via events
    dw_profile prof{};
    bool profiling = false;
    cudaEvent_t ev[2] = {nullptr, nullptr};
    bool ev_pending = false;
    uint64_t ev_cells = 0;

    // checkpoint
    struct Ckpt {
        bool have = false, grid_valid = false, lat_valid = false;
        double *grid = nullptr, *cov = nullptr;
        bool cov_valid = false, have_cov = false;
        double cov_L = 0;
        uint32_t *lat = nullptr, *lat_pre = nullptr;
        int32_t *agent_xy = nullptr;
        double *agent_state = nullptr;
        int64_t *done_at = nullptr, *agents_done_at = nullptr;
        dw_clock clk{};
        PreKind pre = PRE_NONE;
        double L_last = 0;
        bool ch6_dirty_saved = false;   // of the buffer the checkpointed grid was copied from
    } ck[2];   // slot 0: dw_checkpoint_save/restore (caller), slot 1: dw_run's chunk rewind
};

#define DW_LAUNCHED(h) do { (h)->prof.kernel_launches += 1; DW_CUDA_TRY((h), cudaGetLastError()); } while (0)

static int dw_fail(dw_handle *h, int code, const char *what, const char *detail);
static int dw_fail(dw_handle *h, int code, const char *what, const char *detail) {
    std::string m = std::string(what) + ": " + detail;
    if (h) h->err = m; else g_create_error = m;
    return code;
}

static DevParams make_params_cfg(const dw_config &c) {
    DevParams P{};
    P.B = c.batch; P.N = c.dim; P.n_agents = c.n_agents;
    P.p = c.p; P.g = c.g; P.S = c.S; P.sigma = c.sigma; P.gamma = c.gamma; P.q = c.q; P.q2 = c.q2;
    P.temp_optimal = c.temp_optimal; P.dt = c.dt; P.agent_gamma = c.agent_gamma;
    P.ab = c.albedo_bare; P.al = c.albedo_light; P.ad = c.albedo_dark;
    // ft_convolve is a convolution, not a correlation: the neighbour at row-major position i takes the tap turned 180 degrees
    for (int i = 0; i < 9; ++i) { P.w[i] = c.daisy_kernel[8 - i]; P.adj[i] = c.adjacent_kernel[8 - i]; P.mask[i] = c.obs_mask[i]; }
    // Screened forward (dw_screened_cell): the fast evaluation differs from the literal one by the fast fourth root
    // (3e-12 relative, asserted in the tests) plus a few ulp. With T <= 400 K and |Topt - T| <= max(|Topt - 150|, |Topt - 400|)
    // (the kernel checks the range) and densities in [0, 1]: |d(1000 l')| <= 1000 dt 2 g |Topt - T| T 3e-12, b' twice that,
    // |d(1000 T)| <= 1000 * 400 * 3e-12. Filters are 4x the bounds.
    P.adj_sum = 0.0;
    for (int i = 0; i < 9; ++i) P.adj_sum += c.adjacent_kernel[i];
    const double dT = fmax(fabs(c.temp_optimal - 150.0), fabs(c.temp_optimal - 400.0));
    const double bound = 1000.0 * fabs(c.dt) * 2.0 * fabs(c.g) * dT * 400.0 * 3e-12;
    P.eps_c = fmax(4.0 * bound, 4e-6);
    P.eps_b = 2.0 * P.eps_c;
    P.eps_T = 4.0 * 1000.0 * 400.0 * 3e-12;
    P.xlo = 150.0 * 150.0 * 150.0 * 150.0;
    P.xhi = 400.0 * 400.0 * 400.0 * 400.0;
    P.screen = (P.eps_c < 0.05 && c.sigma > 0.0 && !getenv("DW_LITERAL_ONLY")) ? 1 : 0;   // NaN bounds fail the comparison too
    return P;
}
static DevParams make_params(const dw_handle *h) { return make_params_cfg(h->cfg); }

static inline int grid_for(size_t total, int block = 256) {
    size_t g = (total + block - 1) / block;
    const size_t cap = 148 * 64;   // grid-stride loops: a few waves of 148 SMs
    return (int)(g < 1 ? 1 : (g > cap ? cap : g));
}

// forward launches: two cells per thread when the world side is even (aligned 16-byte accesses), else one
template <class Src>
static void launch_forward(dw_handle *h, const DevParams &P, double SL, Src src, double *out, double *writeback_b0,
                           unsigned long long *world_max, int zero6);
template <class Src>
static void launch_forward_lattice(dw_handle *h, const DevParams &P, double SL, Src src, uint32_t *lat_out, unsigned long long *world_max);

static void update_L(dw_clock &c) {   // daisy_world_rl.py:463-473
    c.step_count += 1;
    if (c.ramp_up_down && c.ramp_period != 0 && c.step_count % c.ramp_period == 0) {
        c.dL *= -1;
        c.min_L -= c.ddL;
        c.max_L += c.ddL;
    }
    double L = c.L + c.dL;
    L = L < c.max_L ? L : c.max_L;
    c.L = L > c.min_L ? L : c.min_L;
}

template <class T>
static int dev_alloc(dw_handle *h, T **p, size_t count) {
    if (*p) return DW_OK;
    DW_CUDA_TRY(h, cudaMalloc((void **)p, (count ? count : 1) * sizeof(T)));
    DW_CUDA_TRY(h, cudaMemsetAsync(*p, 0, (count ? count : 1) * sizeof(T), h->stream));
    return DW_OK;
}

static int ensure_grid_buffers(dw_handle *h) {
    const size_t G = (size_t)h->cfg.batch * 7 * h->NN;
    for (int i = 0; i < 2; ++i) {
        int rc = dev_alloc(h, &h->grid[i], G);
        if (rc) return rc;
    }
    return DW_OK;
}

static int ensure_scratch(dw_handle *h, size_t count) {
    if (h->scratch_cap >= count) return DW_OK;
    if (h->scratch) cudaFree(h->scratch);
    h->scratch = nullptr;
    DW_CUDA_TRY(h, cudaMalloc((void **)&h->scratch, count * sizeof(double)));
    h->scratch_cap = count;
    return DW_OK;
}

static size_t out_m(const dw_handle *h) { return (size_t)h->cfg.batch * (h->cfg.n_agents ? h->cfg.n_agents : 2); }
static size_t out_done_off(const dw_handle *h) { return out_m(h) * sizeof(double); }
static size_t out_obs_off(const dw_handle *h) { return out_done_off(h) + ((out_m(h) + 7) & ~(size_t)7); }
static size_t out_total(const dw_handle *h) { return out_obs_off(h) + (size_t)h->cfg.batch * h->cfg.n_agents * 63 * sizeof(double); }

static int ensure_out_block(dw_handle *h, bool with_obs) {
    if (h->out_block && (h->out_full || !with_obs)) return DW_OK;
    const size_t bytes = with_obs ? out_total(h) : out_obs_off(h);
    unsigned char *blk = nullptr;
    DW_CUDA_TRY(h, cudaMalloc((void **)&blk, bytes ? bytes : 8));
    DW_CUDA_TRY(h, cudaMemsetAsync(blk, 0, bytes ? bytes : 8, h->stream));
    if (h->out_block) {            // growing: keep reward / done of the last step
        DW_CUDA_TRY(h, cudaMemcpyAsync(blk, h->out_block, out_obs_off(h), cudaMemcpyDeviceToDevice, h->stream));
        DW_CUDA_TRY(h, cudaStreamSynchronize(h->stream));
        cudaFree(h->out_block);
    }
    h->out_block = blk;
    h->out_full = with_obs;
    h->reward = reinterpret_cast<double *>(blk);
    h->done = blk + out_done_off(h);
    h->obs = with_obs ? reinterpret_cast<double *>(blk + out_obs_off(h)) : nullptr;
    h->obs_valid = false;
    return DW_OK;
}

// every operation that advances or replaces the live state ends the validity of what was derived from the old one
static void state_changed(dw_handle *h) {
    h->obs_valid = false;
    h->fwd_diag = false;
}

// ---- lazy conversions between the two state representations -----------------------------------------
static int launch_stamp(dw_handle *h, double *grid, bool counters, unsigned int *alive_slot, bool rewards) {
    const DevParams P = make_params(h);
    k_stamp_reward<<<(P.B + 127) / 128, 128, 0, h->stream>>>(
        P, grid, h->agent_xy, h->agent_state, (counters || P.n_agents == 0) ? h->world_max : nullptr,
        rewards ? h->reward : nullptr, rewards ? h->done : nullptr, counters ? h->done_at : nullptr,
        counters ? h->agents_done_at : nullptr, alive_slot);
    DW_LAUNCHED(h);
    return DW_OK;
}

// make grid[cur] hold the full reference grid of the current state
template <class Src>
static void launch_forward(dw_handle *h, const DevParams &P, double SL, Src src, double *out, double *writeback_b0,
                           unsigned long long *world_max, int zero6) {
    const size_t total = (size_t)P.B * h->NN;
    if ((P.N & 1) == 0)
        k_forward_x2<Src><<<grid_for(total / 2), 256, 0, h->stream>>>(P, SL, src, out, writeback_b0, world_max, zero6);
    else
        k_forward<Src><<<grid_for(total), 256, 0, h->stream>>>(P, SL, src, out, writeback_b0, world_max, zero6);
}
template <class Src>
static void launch_forward_lattice(dw_handle *h, const DevParams &P, double SL, Src src, uint32_t *lat_out, unsigned long long *world_max) {
    const size_t total = (size_t)P.B * h->NN;
    if ((P.N & 1) == 0)
        k_forward_lattice_x2<Src><<<grid_for(total / 2), 256, 0, h->stream>>>(P, SL, src, lat_out, world_max);
    else
        k_forward_lattice<Src><<<grid_for(total), 256, 0, h->stream>>>(P, SL, src, lat_out, world_max);
}

static int ensure_grid(dw_handle *h) {
    if (h->grid_valid) return DW_OK;
    if (!h->lat_valid && !h->cov_valid) return dw_fail(h, DW_E_STATE, "ensure_grid", "no state uploaded");
    int rc = ensure_grid_buffers(h);
    if (rc) return rc;
    const DevParams P = make_params(h);
    const size_t total = (size_t)P.B * h->NN;
    double *out = h->grid[h->cur];
    if (h->cov_valid) {
        // the reset state: covers from the lean planes, ch0 and the UNROUNDED initial temperatures (initialize_grid :304-324)
        k_cov_to_grid<<<grid_for(total), 256, 0, h->stream>>>(P.B, h->NN, h->cov, out);
        DW_LAUNCHED(h);
        k_init_fields<<<grid_for(total), 256, 0, h->stream>>>(P, h->cfg.S * h->cov_L, out);
        DW_LAUNCHED(h);
        h->ch6_dirty[h->cur] = false;
        h->pre = PRE_GRID;
        h->pre_grid = out;
        h->L_last = h->cov_L;
        h->grid_valid = true;
        return DW_OK;
    }
    if (h->pre == PRE_COV) {
        // the state is one lean step past the reset: literal forward from the post-graze cover planes
        SrcCov src{h->cov, h->NN};
        launch_forward(h, P, h->cfg.S * h->L_last, src, out, nullptr, nullptr, h->ch6_dirty[h->cur] ? 1 : 0);
        DW_LAUNCHED(h);
        h->ch6_dirty[h->cur] = false;
        rc = launch_stamp(h, out, false, nullptr, false);
        if (rc) return rc;
    } else if (h->pre == PRE_LAT) {
        // full literal forward from the post-graze lattice the last fused step started from: reproduces
        // b' (rounded from UNROUNDED l',d'), the temperatures of that step, and l',d' (== lat[lcur]).
        SrcLattice src{h->lat_pre, h->NN};
        launch_forward(h, P, h->cfg.S * h->L_last, src, out, nullptr, nullptr, h->ch6_dirty[h->cur] ? 1 : 0);
        DW_LAUNCHED(h);
        h->ch6_dirty[h->cur] = false;
        rc = launch_stamp(h, out, false, nullptr, false);
        if (rc) return rc;
    } else {
        return dw_fail(h, DW_E_STATE, "ensure_grid", "lattice state without a recorded pre-state");
    }
    h->grid_valid = true;
    return DW_OK;
}

// ---- API ------------------------------------------------------------------------------------------------
extern "C" int dw_abi_version(void) { return DW_ABI_VERSION; }

extern "C" const char *dw_last_error(const dw_handle *h) { return h ? h->err.c_str() : g_create_error.c_str(); }

static int validate_cfg(dw_handle *h, const dw_config *c) {
    if (!c) return dw_fail(h, DW_E_INVALID, "config", "NULL");
    if (c->batch < 1 || c->dim < 1 || c->n_agents < 0) return dw_fail(h, DW_E_INVALID, "config", "batch>=1, dim>=1, n_agents>=0 required");
    if ((size_t)c->dim >= (1u << 23)) return dw_fail(h, DW_E_INVALID, "config", "dim too large");
    return DW_OK;
}

extern "C" int dw_create(const dw_config *cfg, dw_handle **out) {
    if (!out) return dw_fail(nullptr, DW_E_INVALID, "dw_create", "out is NULL");
    *out = nullptr;
    int rc = validate_cfg(nullptr, cfg);
    if (rc) return rc;
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0)
        return dw_fail(nullptr, DW_E_CUDA, "dw_create", e != cudaSuccess ? cudaGetErrorString(e) : "no CUDA device (there is no CPU fallback)");
    if (cfg->device < 0 || cfg->device >= ndev) return dw_fail(nullptr, DW_E_INVALID, "dw_create", "bad device ordinal");
    e = cudaSetDevice(cfg->device);
    if (e != cudaSuccess) return dw_fail(nullptr, DW_E_CUDA, "cudaSetDevice", cudaGetErrorString(e));
    dw_handle *h = new dw_handle();
    h->cfg = *cfg;
    h->NN = (size_t)cfg->dim * cfg->dim;
    const size_t B = cfg->batch, n = cfg->n_agents;
    rc = dev_alloc(h, &h->agent_xy, B * n * 2);
    if (!rc) rc = dev_alloc(h, &h->agent_state, B * n);
    if (!rc) rc = ensure_out_block(h, false);
    if (!rc) rc = dev_alloc(h, &h->world_max, B * 2);
    if (!rc) rc = dev_alloc(h, &h->done_at, B);
    if (!rc) rc = dev_alloc(h, &h->agents_done_at, B * n);
    if (!rc) rc = dev_alloc(h, &h->alive, DW_FUSED_MAX_STEPS);
    if (rc) { g_create_error = h->err; dw_destroy(h); return rc; }
    h->clk.L = 0.75; h->clk.min_L = 0.75; h->clk.max_L = 1.5; h->clk.ramp_period = 512;
    h->clk.dL = (h->clk.max_L - h->clk.min_L) / 512.0;
    *out = h;
    return DW_OK;
}

extern "C" int dw_destroy(dw_handle *h) {
    if (!h) return DW_OK;
    cudaSetDevice(h->cfg.device);
    cudaStreamSynchronize(h->stream);
    void *ptrs[] = {h->grid[0], h->grid[1], h->cov, h->agent_idx64, h->lat[0], h->lat[1], h->lat_pre, h->agent_xy, h->agent_state, h->out_block, h->world_max, h->done_at, h->agents_done_at, h->alive, h->action_dev, h->scratch, h->fwd_in, h->slow_count, h->grid32, h->f32_stats, h->pop_rew, h->alive_mask, h->sc_dev, h->persist_sync, h->series_T, h->series_l, h->series_d, h->mlp_dev, h->pop_sum, h->pop_done, h->pop_steps, h->pop_frozen, h->pop_ndone,
                    h->fwd_out};
    for (void *p : ptrs) if (p) cudaFree(p);
    if (h->pin) cudaFreeHost(h->pin);
    for (auto &c : h->ck) {
        void *cp[] = {c.grid, c.cov, c.lat, c.lat_pre, c.agent_xy, c.agent_state, c.done_at, c.agents_done_at};
        for (void *p : cp) if (p) cudaFree(p);
    }
    delete h;
    return DW_OK;
}

extern "C" int dw_set_config(dw_handle *h, const dw_config *cfg) {
    if (!h) return DW_E_INVALID;
    int rc = validate_cfg(h, cfg);
    if (rc) return rc;
    if (cfg->batch != h->cfg.batch || cfg->dim != h->cfg.dim || cfg->n_agents != h->cfg.n_agents || cfg->device != h->cfg.device)
        return dw_fail(h, DW_E_INVALID, "dw_set_config", "shapes/device of a handle are fixed; create a new handle");
    h->cfg = *cfg;
    return DW_OK;
}

extern "C" int dw_set_clock(dw_handle *h, const dw_clock *clk) {
    if (!h || !clk) return DW_E_INVALID;
    h->clk = *clk;
    return DW_OK;
}
extern "C" int dw_get_clock(dw_handle *h, dw_clock *clk) {
    if (!h || !clk) return DW_E_INVALID;
    *clk = h->clk;
    return DW_OK;
}
extern "C" int dw_get_last_L(dw_handle *h, double *L) {
    if (!h || !L) return DW_E_INVALID;
    *L = h->fwd_diag ? h->fwd_L : h->L_last;
    return DW_OK;
}
extern "C" int dw_set_stream(dw_handle *h, void *s) {
    if (!h) return DW_E_INVALID;
    h->stream = (cudaStream_t)s;
    h->sc_clk.clear();                         // the cached coefficient table was uploaded in the old stream's order
    return DW_OK;
}
extern "C" int dw_set_epsilon(dw_handle *h, double epsilon) {
    if (!h || !(epsilon >= 0.0 && epsilon <= 1.0)) return DW_E_INVALID;
    h->epsilon = epsilon;
    return DW_OK;
}
extern "C" int dw_synchronize(dw_handle *h) {
    if (!h) return DW_E_INVALID;
    DW_CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    DW_CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    return DW_OK;
}

extern "C" int dw_upload_state(dw_handle *h, const double *grid, const int64_t *agent_indices, const double *agent_states) {
    if (!h) return DW_E_INVALID;
    DW_CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    const size_t B = h->cfg.batch, n = h->cfg.n_agents, NN = h->NN;
    if (agent_states) h->agents_open = false;      // a fresh agent state supersedes a pending collision pass
    if (grid) {
        int rc = ensure_grid_buffers(h);
        if (rc) return rc;
        DW_CUDA_TRY(h, cudaMemcpyAsync(h->grid[h->cur], grid, B * 7 * NN * sizeof(double), cudaMemcpyHostToDevice, h->stream));
        // channel 6 is "always 0" after any forward (new_grid = 0*grid, :445); only pay for zeroing it when
        // the caller actually put something there
        bool dirty = false;
        for (size_t b = 0; b < B && !dirty; ++b) {
            const double *c6 = grid + (b * 7 + 6) * NN;
            for (size_t i = 0; i < NN; ++i) if (c6[i] != 0.0) { dirty = true; break; }
        }
        h->ch6_dirty[h->cur] = dirty;   // cleaned (zeroed) the next time a forward writes this buffer
        h->grid_valid = true;
        h->cov_valid = false;
        h->lat_valid = false;
        h->pre = PRE_NONE;
        state_changed(h);
    }
    if (n && agent_indices) {
        // int64 -> wrapped int32 on the device: with pinned host memory the whole upload is asynchronous
        const size_t count = B * n * 2;
        int rc = dev_alloc(h, &h->agent_idx64, count);
        if (rc) return rc;
        DW_CUDA_TRY(h, cudaMemcpyAsync(h->agent_idx64, agent_indices, count * sizeof(long long), cudaMemcpyHostToDevice, h->stream));
        k_agent_indices_in<<<(unsigned)((count + 255) / 256), 256, 0, h->stream>>>(h->agent_idx64, count, h->cfg.dim, h->agent_xy);
        DW_LAUNCHED(h);
        state_changed(h);
    }
    if (n && agent_states) {
        DW_CUDA_TRY(h, cudaMemcpyAsync(h->agent_state, agent_states, B * n * sizeof(double), cudaMemcpyHostToDevice, h->stream));
        state_changed(h);
    }
    return DW_OK;
}

// initialize_grid's cover assignment (daisy_world_rl.py:304-312): channels 1,2 from host planes, the rest zero
extern "C" int dw_upload_covers(dw_handle *h, const double *light, const double *dark) {
    if (!h || !light || !dark) return DW_E_INVALID;
    DW_CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    const size_t B = h->cfg.batch, NN = h->NN;
    int rc = dev_alloc(h, &h->cov, B * 2 * NN);
    if (rc) return rc;
    DW_CUDA_TRY(h, cudaMemcpy2DAsync(h->cov, 2 * NN * sizeof(double), light, NN * sizeof(double), NN * sizeof(double), B,
                                     cudaMemcpyHostToDevice, h->stream));
    DW_CUDA_TRY(h, cudaMemcpy2DAsync(h->cov + NN, 2 * NN * sizeof(double), dark, NN * sizeof(double), NN * sizeof(double), B,
                                     cudaMemcpyHostToDevice, h->stream));
    h->cov_valid = true;
    h->cov_L = h->clk.L;
    h->grid_valid = false;
    h->lat_valid = false;
    h->pre = PRE_NONE;
    state_changed(h);
    return DW_OK;
}

// Device-side synthetic reset (same distribution as initialize_grid/initialize_agents, counter RNG instead of
// numpy's MT19937): for ensembles too large to draw on the host. Temperatures are NOT filled (dw_init_temperatures).
extern "C" int dw_init_random(dw_handle *h, uint64_t seed, double light_proportion, double dark_proportion, double initial_al,
                              double initial_ad) {
    if (!h) return DW_E_INVALID;
    DW_CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    int rc = dev_alloc(h, &h->cov, (size_t)h->cfg.batch * 2 * h->NN);
    if (rc) return rc;
    const DevParams P = make_params(h);
    k_init_random<<<grid_for((size_t)P.B * h->NN), 256, 0, h->stream>>>(P, seed, h->world0, light_proportion, dark_proportion,
                                                                         initial_al, initial_ad, h->cov, h->agent_xy, h->agent_state);
    DW_LAUNCHED(h);
    h->cov_valid = true;
    h->cov_L = h->clk.L;
    h->grid_valid = false;
    h->lat_valid = false;
    h->pre = PRE_NONE;
    state_changed(h);
    return DW_OK;
}

// initialize_grid's temperature fill (daisy_world_rl.py:304-324): ch0 = p-l-d, ch3..5 = unrounded T, Tl, Td at clk.L
extern "C" int dw_init_temperatures(dw_handle *h) {
    if (!h) return DW_E_INVALID;
    DW_CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    if (h->cov_valid && !h->grid_valid) {
        // lean reset state: remember the luminosity; the fields are filled when (if) the 7-channel grid is materialised,
        // the diagnostics come straight from the cover planes
        h->cov_L = h->clk.L;
        h->pre = PRE_COV;
        h->L_last = h->clk.L;
        state_changed(h);
        return DW_OK;
    }
    if (!h->grid_valid) return dw_fail(h, DW_E_STATE, "dw_init_temperatures", "upload a grid first");
    const DevParams P = make_params(h);
    k_init_fields<<<grid_for((size_t)P.B * h->NN), 256, 0, h->stream>>>(P, h->cfg.S * h->clk.L, h->grid[h->cur]);
    DW_LAUNCHED(h);
    h->pre = PRE_GRID;
    h->pre_grid = h->grid[h->cur];
    h->L_last = h->clk.L;
    state_changed(h);
    return DW_OK;
}

// A step's action bytes go through pinned staging memory: a pageable cudaMemcpyAsync blocks the host for every copy, a
// pinned one is enqueued and the step ends with ONE synchronisation.
#define DW_PIN_ACTION_MAX (64 * 1024)
static int ensure_pinned(dw_handle *h) {
    if (h->pin) return DW_OK;
    DW_CUDA_TRY(h, cudaMallocHost((void **)&h->pin, DW_PIN_ACTION_MAX));
    return DW_OK;
}

// The reference accepts ANY integer action (daisy_world_rl.py:190-212): `a == 8` stays, otherwise `a % 4` (Python modulo:
// non-negative for negative a) picks the move, and `a > 4` grazes. The kernels decode an int8 code c with the same three
// tests (c == 8, c & 3, c > 4), so a maps to: 0..8 itself; a > 8 -> 12 + a % 4 (move a % 4 and graze); a < 0 -> a mod 4
// (move, no graze).
static inline int8_t canonical_action(int64_t a) {
    if (a >= 0 && a <= 8) return (int8_t)a;
    if (a > 8) return (int8_t)(12 + (a & 3));
    return (int8_t)(((a % 4) + 4) % 4);
}

static int stage_action(dw_handle *h, const int64_t *action, size_t count) {
    if (h->action_cap < count) {
        if (h->action_dev) cudaFree(h->action_dev);
        h->action_dev = nullptr;
        DW_CUDA_TRY(h, cudaMalloc((void **)&h->action_dev, count));
        h->action_cap = count;
    }
    if (count <= DW_PIN_ACTION_MAX) {
        // every earlier use of the staging area was followed by a synchronisation of this stream or is ordered before this
        // copy on it; the action bytes are read by the copy engine before the kernels that follow can touch anything else
        int rc = ensure_pinned(h);
        if (rc) return rc;
        DW_CUDA_TRY(h, cudaStreamSynchronize(h->stream));   // cheap when idle: the previous upload from this area has been consumed
        int8_t *a8 = reinterpret_cast<int8_t *>(h->pin);
        for (size_t i = 0; i < count; ++i) a8[i] = canonical_action(action[i]);
        DW_CUDA_TRY(h, cudaMemcpyAsync(h->action_dev, a8, count, cudaMemcpyHostToDevice, h->stream));
        return DW_OK;
    }
    std::vector<int8_t> a8(count);
    for (size_t i = 0; i < count; ++i) a8[i] = canonical_action(action[i]);
    DW_CUDA_TRY(h, cudaMemcpyAsync(h->action_dev, a8.data(), count, cudaMemcpyHostToDevice, h->stream));
    DW_CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    return DW_OK;
}

static int launch_agents(dw_handle *h, const int8_t *act_dev, int ab, int am, int policy, uint64_t seed, bool on_cov = false,
                         bool clip = true) {
    if (h->cfg.n_agents == 0) return DW_OK;
    const DevParams P = make_params(h);
    const size_t NN = h->NN;
    policy = dw_resolve_policy(policy, h->epsilon, seed, (uint32_t)h->clk.step_count);
    if (on_cov)
        k_agents_grid<<<(P.B + 127) / 128, 128, 0, h->stream>>>(P, h->cov, 2 * NN, 0, NN, h->agent_xy, h->agent_state, act_dev, ab, am,
                                                                 policy, seed, (uint32_t)h->clk.step_count, h->world0);
    else
        k_agents_grid<<<(P.B + 127) / 128, 128, 0, h->stream>>>(P, h->grid[h->cur], 7 * NN, NN, 2 * NN, h->agent_xy, h->agent_state,
                                                                 act_dev, ab, am, policy, seed, (uint32_t)h->clk.step_count, h->world0,
                                                                 clip ? 1 : 0);
    DW_LAUNCHED(h);
    return DW_OK;
}

// forward + stamp + reward/done (+ optional lifespan counters) + clock: the tail of step() after update_agents
static int launch_forward_tail(dw_handle *h, bool counters, unsigned int *alive_slot) {
    const DevParams P = make_params(h);
    const size_t total = (size_t)P.B * h->NN;
    double *in = h->grid[h->cur], *out = h->grid[1 - h->cur];
    DW_CUDA_TRY(h, cudaMemsetAsync(h->world_max, 0, (size_t)P.B * 2 * sizeof(unsigned long long), h->stream));
    SrcGrid src{in, 7 * h->NN, h->NN};
    launch_forward(h, P, h->cfg.S * h->clk.L, src, out, in, h->world_max, h->ch6_dirty[1 - h->cur] ? 1 : 0);
    DW_LAUNCHED(h);
    h->ch6_dirty[1 - h->cur] = false;
    h->pre = PRE_GRID;
    h->pre_grid = in;
    h->L_last = h->clk.L;
    h->cur = 1 - h->cur;
    int rc = launch_stamp(h, out, counters, alive_slot, true);
    if (rc) return rc;
    h->grid_valid = true;
    h->cov_valid = false;
    h->lat_valid = false;
    state_changed(h);
    update_L(h->clk);
    return DW_OK;
}

static int mlp_actions(dw_handle *h);
static int run_steps_fused(dw_handle *h, int K, int policy, const int8_t *act_dev, uint64_t seed, unsigned int *alive);
static bool dw_fused_supported(const dw_handle *h);

// Between dw_agents_begin and dw_agents_collide the agent states are unclipped: every other stepping call is refused.
static int refuse_open(dw_handle *h, const char *what) {
    return h->agents_open ? dw_fail(h, DW_E_STATE, what, "dw_agents_begin not closed by dw_agents_collide") : DW_OK;
}

// What the agent kernels of one step run. A step's actions come from one of four sources: explicit host actions [ab<=B,
// am<=n] (policy < 0, staged to the device), NULL (policy < 0: step(None)), the device MLP (DW_POLICY_MLP: its actions are
// computed here from the current state, then replayed) or a device policy decided inside the kernels.
struct StepActions {
    const int8_t *act;   // device int8 [ab,am] of DW_POLICY_REPLAY, else NULL
    int ab, am;
    int policy;          // DW_POLICY_REPLAY, DW_POLICY_NONE or the device policy
    uint64_t seed;       // the caller's for device policies, 0 for explicit actions (REPLAY and NONE do not read it)
};
static int resolve_actions(dw_handle *h, const char *what, const int64_t *action, int32_t ab, int32_t am, int32_t policy,
                           uint64_t seed, StepActions *sa) {
    int rc = refuse_open(h, what);
    if (rc) return rc;
    if (policy == DW_POLICY_REPLAY || policy > DW_POLICY_MLP)
        return dw_fail(h, DW_E_INVALID, what, "policy must be < 0 (explicit action / NULL) or a device policy");
    const int B = h->cfg.batch, n = h->cfg.n_agents;
    if (policy < 0) {
        *sa = StepActions{nullptr, 0, 0, DW_POLICY_NONE, 0};
        if (!action || n == 0) return DW_OK;
        if (ab < 0 || am < 0 || ab > B || am > n) return dw_fail(h, DW_E_INVALID, what, "action must be [ab<=B, am<=n]");
        rc = stage_action(h, action, (size_t)ab * am);
        if (rc) return rc;
        *sa = StepActions{h->action_dev, ab, am, DW_POLICY_REPLAY, 0};
        return DW_OK;
    }
    *sa = StepActions{nullptr, 0, 0, policy, seed};
    if (policy != DW_POLICY_MLP) return DW_OK;
    if (n == 0) {
        sa->policy = DW_POLICY_NONE;
        return DW_OK;
    }
    // the network's actions from the observation of the current state: before anything of this step is launched
    rc = mlp_actions(h);
    if (rc) return rc;
    *sa = StepActions{h->action_dev, B, n, DW_POLICY_REPLAY, seed};
    return DW_OK;
}

extern "C" int dw_update_agents(dw_handle *h, const int64_t *action, int32_t ab, int32_t am) {
    if (!h) return DW_E_INVALID;
    DW_CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    if (h->cfg.n_agents == 0) return DW_OK;
    if (!action) return dw_fail(h, DW_E_INVALID, "dw_update_agents", "action must be [ab<=B, am<=n]");
    StepActions sa;
    int rc = resolve_actions(h, "dw_update_agents", action, ab, am, -1, 0, &sa);
    if (!rc) rc = ensure_grid(h);
    if (rc) return rc;
    rc = launch_agents(h, sa.act, sa.ab, sa.am, sa.policy, sa.seed);
    h->lat_valid = false;
    h->cov_valid = false;
    state_changed(h);
    return rc;
}

// step() keeps the state where the fused kernels keep it (packed lattice / lean reset planes) whenever the physics is one
// the fast path covers: one K = 1 launch of the fused kernel instead of materialising the fp64 [B,7,N,N] grid (64 B per
// cell). env.grid, diagnostics and observations are rebuilt on demand from the pre-state the step started from.
// Partial actions (ab < B or am < n) and exotic kernels take the materialising path.
static bool lean_step_ok(const dw_handle *h, const int64_t *action, int32_t ab, int32_t am) {
    if (!dw_fused_supported(h)) return false;
    if (h->cfg.n_agents > 0 && action && (ab != h->cfg.batch || am != h->cfg.n_agents)) return false;
    return h->lat_valid || h->cov_valid || h->grid_valid;
}
struct CountLifeGuard {
    dw_handle *h; bool old;
    CountLifeGuard(dw_handle *h_, bool v) : h(h_), old(h_->count_life) { h->count_life = v; }
    ~CountLifeGuard() { h->count_life = old; }
};

// One step() with its actions from any source (resolve_actions), lean or materialising (lean_step_ok); the outputs stay in
// the device's output block
static int step_once(dw_handle *h, const int64_t *action, int32_t ab, int32_t am, int32_t policy, uint64_t seed) {
    StepActions sa;
    int rc = resolve_actions(h, "dw_step_packed", action, ab, am, policy, seed, &sa);
    if (rc) return rc;
    if (lean_step_ok(h, policy < 0 ? action : nullptr, ab, am)) {
        CountLifeGuard guard(h, false);
        return run_steps_fused(h, 1, sa.policy, sa.act, sa.seed, h->alive);
    }
    rc = ensure_grid(h);
    if (!rc) rc = launch_agents(h, sa.act, sa.ab, sa.am, sa.policy, sa.seed);
    if (rc) return rc;
    return launch_forward_tail(h, false, nullptr);
}

// ---- collision_mode == 1 (daisy_world_rl.py:220-242): update_agents in two calls around the caller's RNG draws ----
extern "C" int dw_agents_begin(dw_handle *h, const int64_t *action, int32_t ab, int32_t am, int32_t policy, uint64_t seed,
                               int64_t *agent_indices) {
    if (!h) return DW_E_INVALID;
    DW_CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    if (h->cfg.n_agents == 0) return DW_OK;
    StepActions sa;
    int rc = resolve_actions(h, "dw_agents_begin", action, ab, am, policy, seed, &sa);
    if (!rc) rc = ensure_grid(h);
    if (!rc) rc = launch_agents(h, sa.act, sa.ab, sa.am, sa.policy, sa.seed, false, false);
    if (rc) return rc;
    h->agents_open = true;
    h->lat_valid = false;
    h->cov_valid = false;
    state_changed(h);
    return dw_get_agents(h, agent_indices, nullptr);
}

extern "C" int dw_agents_collide(dw_handle *h, const double *noise, const int32_t *cell_offsets, double food_chain_penalty) {
    if (!h) return DW_E_INVALID;
    DW_CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    const size_t B = h->cfg.batch, n = h->cfg.n_agents;
    if (n == 0) return DW_OK;
    if (!h->agents_open) return dw_fail(h, DW_E_STATE, "dw_agents_collide", "no dw_agents_begin pending");
    if (!cell_offsets) return dw_fail(h, DW_E_INVALID, "dw_agents_collide", "cell_offsets [B+1] required");
    const size_t cells = (size_t)cell_offsets[B];
    if (cell_offsets[0] != 0 || (cells && !noise)) return dw_fail(h, DW_E_INVALID, "dw_agents_collide", "cell_offsets must start at 0; noise [cells, n]");
    for (size_t b = 0; b < B; ++b)
        if (cell_offsets[b + 1] < cell_offsets[b]) return dw_fail(h, DW_E_INVALID, "dw_agents_collide", "cell_offsets must not decrease");
    // scratch: [losers B*n | noise cells*n | offsets (B+1 int32)]
    int rc = ensure_scratch(h, B * n + cells * n + (B + 2) / 2 + 1);
    if (!rc) rc = dev_alloc(h, &h->slow_count, (size_t)2);
    if (rc) return rc;
    double *los = h->scratch, *noise_dev = h->scratch + B * n;
    int32_t *off_dev = reinterpret_cast<int32_t *>(noise_dev + cells * n);
    if (cells) DW_CUDA_TRY(h, cudaMemcpyAsync(noise_dev, noise, cells * n * sizeof(double), cudaMemcpyHostToDevice, h->stream));
    DW_CUDA_TRY(h, cudaMemcpyAsync(off_dev, cell_offsets, (B + 1) * sizeof(int32_t), cudaMemcpyHostToDevice, h->stream));
    DW_CUDA_TRY(h, cudaMemsetAsync(h->slow_count + 1, 0, sizeof(unsigned int), h->stream));
    const DevParams P = make_params(h);
    k_collide<<<(P.B + 127) / 128, 128, 0, h->stream>>>(P, h->agent_xy, h->agent_state, noise_dev, off_dev, food_chain_penalty, los,
                                                        h->slow_count + 1);
    DW_LAUNCHED(h);
    unsigned int bad = 0;
    DW_CUDA_TRY(h, cudaMemcpyAsync(&bad, h->slow_count + 1, sizeof(bad), cudaMemcpyDeviceToHost, h->stream));
    DW_CUDA_TRY(h, cudaStreamSynchronize(h->stream));       // also keeps the pageable noise / offsets alive until they are read
    h->agents_open = false;
    if (bad) return dw_fail(h, DW_E_INVALID, "dw_agents_collide", "shared-cell counts differ from the positions on the device");
    return DW_OK;
}

// The rest of step() after dw_agents_collide with the notebook's lifespan counters (done_at, agents_done_at) advanced like
// dw_run does; *worlds_alive = worlds with max(grid[:,1:3]) > 0.005 after this step. Synchronises.
extern "C" int dw_step_tail_counted(dw_handle *h, int64_t *worlds_alive) {
    if (!h) return DW_E_INVALID;
    DW_CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    int rc = refuse_open(h, "dw_step_tail_counted");
    if (!rc) rc = ensure_grid(h);
    if (rc) return rc;
    DW_CUDA_TRY(h, cudaMemsetAsync(h->alive, 0, sizeof(unsigned int), h->stream));
    rc = launch_forward_tail(h, true, h->alive);
    if (rc) return rc;
    unsigned int alive = 0;
    DW_CUDA_TRY(h, cudaMemcpyAsync(&alive, h->alive, sizeof(alive), cudaMemcpyDeviceToHost, h->stream));
    DW_CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    if (worlds_alive) *worlds_alive = alive;
    return DW_OK;
}

static int mlp_upload(dw_handle *h, const double *params, int sets) {
    const size_t count = (size_t)sets * DW_MLP_PARAMS;
    if (h->mlp_cap < count) {
        if (h->mlp_dev) cudaFree(h->mlp_dev);
        h->mlp_dev = nullptr;
        DW_CUDA_TRY(h, cudaMalloc((void **)&h->mlp_dev, count * sizeof(double)));
        h->mlp_cap = count;
    }
    DW_CUDA_TRY(h, cudaMemcpyAsync(h->mlp_dev, params, count * sizeof(double), cudaMemcpyHostToDevice, h->stream));
    DW_CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    h->mlp_set = true;
    return DW_OK;
}

extern "C" int dw_set_mlp(dw_handle *h, const double *parameters, int32_t n_parameters) {
    if (!h || !parameters) return DW_E_INVALID;
    if (n_parameters != DW_MLP_PARAMS) return dw_fail(h, DW_E_INVALID, "dw_set_mlp", "expected 63*16 + 16*32 + 32*9 = 1808 parameters");
    DW_CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    int rc = mlp_upload(h, parameters, 1);
    if (rc) return rc;
    h->pop_members = 0;
    return DW_OK;
}

extern "C" int dw_set_mlp_population(dw_handle *h, const double *members, int32_t n_members, int32_t adversary_index) {
    if (!h || !members) return DW_E_INVALID;
    if (n_members < 1 || adversary_index < 0 || adversary_index >= n_members || h->cfg.batch % n_members)
        return dw_fail(h, DW_E_INVALID, "dw_set_mlp_population", "batch must split evenly over the members; 0 <= adversary < n_members");
    DW_CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    int rc = mlp_upload(h, members, n_members);
    if (rc) return rc;
    h->pop_members = n_members;
    h->pop_adversary = adversary_index;
    return DW_OK;
}

static int compute_obs(dw_handle *h);

// DW_POLICY_MLP: actions of every agent for the next step from the current observations -> h->action_dev (int8 [B,n])
static int mlp_actions(dw_handle *h) {
    const size_t count = (size_t)h->cfg.batch * h->cfg.n_agents;
    if (!count) return DW_OK;
    if (!h->mlp_set) return dw_fail(h, DW_E_STATE, "DW_POLICY_MLP", "call dw_set_mlp first");
    if (h->action_cap < count) {
        if (h->action_dev) cudaFree(h->action_dev);
        h->action_dev = nullptr;
        DW_CUDA_TRY(h, cudaMalloc((void **)&h->action_dev, count));
        h->action_cap = count;
    }
    const int n = h->cfg.n_agents, wpm = h->pop_members ? h->cfg.batch / h->pop_members : 0;
    if (count <= 65536 && !h->grid_valid && !h->obs_valid && h->lat_valid && (h->pre == PRE_LAT || h->pre == PRE_COV)) {
        // between fused steps: windows and network in one kernel (one warp per agent: latency-optimal for the launch-bound
        // ensemble sizes; larger ones are throughput-bound and take the two thread-per-element kernels below)
        const DevParams P = make_params(h);
        const double SL = h->cfg.S * h->L_last;
        const unsigned blocks = (unsigned)((count + 3) / 4);
        if (h->pre == PRE_LAT)
            k_obs_mlp<SrcLattice><<<blocks, 128, 0, h->stream>>>(P, SL, SrcLattice{h->lat_pre, h->NN}, h->agent_xy, h->agent_state, h->mlp_dev,
                                                                  count, h->action_dev, wpm, n / 2, h->pop_adversary);
        else
            k_obs_mlp<SrcCov><<<blocks, 128, 0, h->stream>>>(P, SL, SrcCov{h->cov, h->NN}, h->agent_xy, h->agent_state, h->mlp_dev, count,
                                                              h->action_dev, wpm, n / 2, h->pop_adversary);
        DW_LAUNCHED(h);
        return DW_OK;
    }
    int rc = compute_obs(h);
    if (rc) return rc;
    k_mlp_act<<<(unsigned)((count + 127) / 128), 128, 0, h->stream>>>(h->mlp_dev, h->obs, count, h->action_dev, wpm, n, n / 2,
                                                                        h->pop_adversary);
    DW_LAUNCHED(h);
    return DW_OK;
}

extern "C" int dw_forward(dw_handle *h, double *grid_in, double *grid_out) {
    if (!h || !grid_in || !grid_out) return DW_E_INVALID;
    DW_CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    const size_t G = (size_t)h->cfg.batch * 7 * h->NN;
    int rc = dev_alloc(h, &h->fwd_in, G);
    if (!rc) rc = dev_alloc(h, &h->fwd_out, G);
    if (rc) return rc;
    const DevParams P = make_params(h);
    DW_CUDA_TRY(h, cudaMemcpyAsync(h->fwd_in, grid_in, G * sizeof(double), cudaMemcpyHostToDevice, h->stream));
    SrcGrid src{h->fwd_in, 7 * h->NN, h->NN};
    launch_forward(h, P, h->cfg.S * h->clk.L, src, h->fwd_out, h->fwd_in, nullptr, 1);
    DW_LAUNCHED(h);
    rc = launch_stamp(h, h->fwd_out, false, nullptr, false);
    if (rc) return rc;
    // the reference's forward() refreshes env.temp/beta/growth as a side effect: the diagnostics are served from this call's
    // input until the live state advances; the live state's own pre-state is left alone
    h->fwd_diag = true;
    h->fwd_L = h->clk.L;
    DW_CUDA_TRY(h, cudaMemcpyAsync(grid_out, h->fwd_out, G * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
    // ch0 of the argument is mutated in place by the reference (:381)
    for (int b = 0; b < h->cfg.batch; ++b)
        DW_CUDA_TRY(h, cudaMemcpyAsync(grid_in + (size_t)b * 7 * h->NN, h->fwd_in + (size_t)b * 7 * h->NN, h->NN * sizeof(double),
                                       cudaMemcpyDeviceToHost, h->stream));
    DW_CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    return DW_OK;
}

// observation windows at `pos` [nb,m,2] (device) without a materialised grid, when the state allows it (lean_obs_ok)
static bool lean_obs_ok(const dw_handle *h) {
    if (h->grid_valid) return false;
    return h->cov_valid || (h->lat_valid && (h->pre == PRE_LAT || h->pre == PRE_COV));
}
static int launch_lean_obs(dw_handle *h, const int32_t *pos, int nb, int m, double *out) {
    const DevParams P = make_params(h);
    const int g = grid_for((size_t)nb * m * 9);
    if (h->cov_valid) {
        // the state right after reset(): initialize_grid's unrounded fields at the reset luminosity, no agent stamp
        k_obs_from_pre<SrcCov><<<g, 256, 0, h->stream>>>(P, h->cfg.S * h->cov_L, SrcCov{h->cov, h->NN}, pos, nb, m, h->agent_xy,
                                                         h->agent_state, out, 1);
    } else if (h->pre == PRE_LAT) {
        k_obs_from_pre<SrcLattice><<<g, 256, 0, h->stream>>>(P, h->cfg.S * h->L_last, SrcLattice{h->lat_pre, h->NN}, pos, nb, m,
                                                             h->agent_xy, h->agent_state, out, 0);
    } else {
        k_obs_from_pre<SrcCov><<<g, 256, 0, h->stream>>>(P, h->cfg.S * h->L_last, SrcCov{h->cov, h->NN}, pos, nb, m, h->agent_xy,
                                                         h->agent_state, out, 0);
    }
    DW_LAUNCHED(h);
    return DW_OK;
}

static int compute_obs(dw_handle *h) {
    if (h->obs_valid) return DW_OK;
    const size_t B = h->cfg.batch, n = h->cfg.n_agents;
    if (n == 0) { h->obs_valid = true; return DW_OK; }
    int rc = ensure_out_block(h, true);
    if (rc) return rc;
    if (lean_obs_ok(h)) {
        // lean state: re-evaluate only the agents' windows from the state the last step started from (or from the reset
        // planes) instead of materialising the whole 7-channel grid
        rc = launch_lean_obs(h, h->agent_xy, (int)B, (int)n, h->obs);
        if (rc) return rc;
        h->obs_valid = true;
        return DW_OK;
    }
    rc = ensure_grid(h);
    if (rc) return rc;
    const DevParams P = make_params(h);
    k_obs<<<grid_for(B * n * 63), 256, 0, h->stream>>>(P, h->grid[h->cur], h->agent_xy, (int)B, (int)n, h->obs);
    DW_LAUNCHED(h);
    h->obs_valid = true;
    return DW_OK;
}

extern "C" int dw_get_obs(dw_handle *h, double *obs) {
    if (!h) return DW_E_INVALID;
    DW_CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    const size_t count = (size_t)h->cfg.batch * h->cfg.n_agents * 63;
    int rc = compute_obs(h);
    if (rc) return rc;
    if (count && obs) DW_CUDA_TRY(h, cudaMemcpyAsync(obs, h->obs, count * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
    DW_CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    return DW_OK;
}

// ---- packed step: everything step() returns in ONE device->host copy ------------------------------------------------------
extern "C" int dw_step_out_layout(dw_handle *h, int64_t *layout) {
    if (!h || !layout) return DW_E_INVALID;
    layout[0] = 0;
    layout[1] = (int64_t)out_done_off(h);
    layout[2] = (int64_t)out_obs_off(h);
    layout[3] = (int64_t)out_total(h);
    return DW_OK;
}

// the output block of the step that just ran -> out (the reward | done part, or all of it with the observations), and the
// clock after that step
static int copy_step_outputs(dw_handle *h, int32_t want_obs, void *out, dw_clock *clk) {
    const bool obs = want_obs && h->cfg.n_agents > 0;
    if (obs) {
        int rc = compute_obs(h);
        if (rc) return rc;
    }
    DW_CUDA_TRY(h, cudaMemcpyAsync(out, h->out_block, obs ? out_total(h) : out_obs_off(h), cudaMemcpyDeviceToHost, h->stream));
    DW_CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    if (clk) *clk = h->clk;
    return DW_OK;
}

extern "C" int dw_step_packed(dw_handle *h, const int64_t *action, int32_t ab, int32_t am, int32_t policy, uint64_t seed,
                              int32_t want_obs, void *out, dw_clock *clk) {
    if (!h || !out) return DW_E_INVALID;
    DW_CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    int rc = step_once(h, action, ab, am, policy, seed);
    return rc ? rc : copy_step_outputs(h, want_obs, out, clk);
}

extern "C" int dw_step_tail_packed(dw_handle *h, int32_t want_obs, void *out, dw_clock *clk) {
    if (!h || !out) return DW_E_INVALID;
    DW_CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    int rc = refuse_open(h, "dw_step_tail_packed");
    if (!rc) rc = ensure_grid(h);
    if (!rc) rc = launch_forward_tail(h, false, nullptr);
    return rc ? rc : copy_step_outputs(h, want_obs, out, clk);
}

// Page-locked host memory for the packed outputs: a device->host copy into it is one DMA at PCIe rate with no staging
// copy (pageable destinations are staged by the driver at a fraction of that).
extern "C" int dw_host_alloc(uint64_t bytes, void **out) {
    if (!out) return DW_E_INVALID;
    *out = nullptr;
    cudaError_t e = cudaMallocHost(out, bytes ? bytes : 8);
    if (e != cudaSuccess) return dw_fail(nullptr, DW_E_CUDA, "dw_host_alloc", cudaGetErrorString(e));
    return DW_OK;
}
extern "C" int dw_host_free(void *p) {
    if (p) cudaFreeHost(p);
    return DW_OK;
}

// test hook: see k_debug_screen_error. grid: host [B,7,N,N] (only channels 1,2 are read); out[6] = measured maxima
// {covers, bare, temperatures} and the filter half-widths {eps_c, eps_b, eps_T} they must stay below.
extern "C" int dw_debug_screen_error(dw_handle *h, const double *grid, double *out) {
    if (!h || !grid || !out) return DW_E_INVALID;
    DW_CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    const size_t G = (size_t)h->cfg.batch * 7 * h->NN;
    int rc = dev_alloc(h, &h->fwd_in, G);
    if (!rc) rc = dev_alloc(h, &h->slow_count, (size_t)2);
    if (!rc) rc = ensure_scratch(h, 4);
    if (rc) return rc;
    const DevParams P = make_params(h);
    DW_CUDA_TRY(h, cudaMemcpyAsync(h->fwd_in, grid, G * sizeof(double), cudaMemcpyHostToDevice, h->stream));
    unsigned long long *acc = reinterpret_cast<unsigned long long *>(h->scratch);
    DW_CUDA_TRY(h, cudaMemsetAsync(acc, 0, 3 * sizeof(unsigned long long), h->stream));
    SrcGrid src{h->fwd_in, 7 * h->NN, h->NN};
    k_debug_screen_error<SrcGrid><<<grid_for((size_t)P.B * h->NN), 256, 0, h->stream>>>(P, h->cfg.S * h->clk.L, src, acc);
    DW_LAUNCHED(h);
    DW_CUDA_TRY(h, cudaMemcpyAsync(out, acc, 3 * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
    DW_CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    out[3] = P.eps_c; out[4] = P.eps_b; out[5] = P.eps_T;
    return DW_OK;
}

extern "C" int dw_get_obs_at(dw_handle *h, const int64_t *agent_indices, int32_t b, int32_t m, double *obs) {
    if (!h || b < 0 || m < 0 || b > h->cfg.batch) return DW_E_INVALID;
    DW_CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    const size_t count = (size_t)b * m * 63;
    if (!count) return DW_OK;
    if (!agent_indices || !obs) return DW_E_INVALID;
    const bool lean = lean_obs_ok(h);          // e.g. reset()'s get_obs: windows from the lean planes, no [B,7,N,N] grid
    int rc = lean ? DW_OK : ensure_grid(h);
    if (rc) return rc;
    rc = ensure_scratch(h, count + (size_t)b * m);   // obs + positions (int32 pairs fit in one double each)
    if (rc) return rc;
    std::vector<int32_t> xy((size_t)b * m * 2);
    for (size_t i = 0; i < xy.size(); ++i) xy[i] = (int32_t)agent_indices[i];
    int32_t *pos = (int32_t *)(h->scratch + count);
    DW_CUDA_TRY(h, cudaMemcpyAsync(pos, xy.data(), xy.size() * sizeof(int32_t), cudaMemcpyHostToDevice, h->stream));
    if (lean) {
        rc = launch_lean_obs(h, pos, b, m, h->scratch);
        if (rc) return rc;
    } else {
        const DevParams P = make_params(h);
        k_obs<<<grid_for(count), 256, 0, h->stream>>>(P, h->grid[h->cur], pos, b, m, h->scratch);
        DW_LAUNCHED(h);
    }
    DW_CUDA_TRY(h, cudaMemcpyAsync(obs, h->scratch, count * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
    DW_CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    return DW_OK;
}

extern "C" int dw_get_grid(dw_handle *h, double *grid) {
    if (!h || !grid) return DW_E_INVALID;
    DW_CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    int rc = ensure_grid(h);
    if (rc) return rc;
    DW_CUDA_TRY(h, cudaMemcpyAsync(grid, h->grid[h->cur], (size_t)h->cfg.batch * 7 * h->NN * sizeof(double), cudaMemcpyDeviceToHost,
                                   h->stream));
    DW_CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    return DW_OK;
}

static int export_f32(dw_handle *h, const double *src, size_t count, float *dst) {
    int rc = ensure_scratch(h, (count + 1) / 2);
    if (rc) return rc;
    float *tmp = reinterpret_cast<float *>(h->scratch);
    k_to_f32<<<grid_for(count), 256, 0, h->stream>>>(src, count, tmp);
    DW_LAUNCHED(h);
    DW_CUDA_TRY(h, cudaMemcpyAsync(dst, tmp, count * sizeof(float), cudaMemcpyDeviceToHost, h->stream));
    DW_CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    return DW_OK;
}

// ---- fp32 mode: the grid of a lattice-resident state materialised with fp32 arithmetic (dw_f32.cuh) ------------------------
static bool dw_fast_path_cfg_ok(const dw_config &c);
static void make_fast_coef(const dw_config &c, FastCoef &F);
static void make_step_coef(const dw_config &c, double L, StepCoef &s);

// the state must be on the lattice with the post-graze lattice of the last step at hand, and the constants must be the
// fast path's (D4-symmetric kernels, g > 0); everything else is served by the fp64 materialisation + conversion
static bool f32_arith_ok(const dw_handle *h) {
    return h->lat_valid && h->pre == PRE_LAT && h->lat_pre && dw_fast_path_cfg_ok(h->cfg) && !getenv("DW_F32_EXPORT_ONLY");
}

static void make_f32_coef(const dw_config &c, const FastCoef &F, const StepCoef &S, const DevParams &P, F32Coef &Q) {
    Q.w0 = (float)F.w0; Q.w12 = (float)F.w12; Q.w2 = (float)F.w2;
    Q.dtp = (float)F.dtp; Q.dtm = (float)F.dtm; Q.dtg = (float)F.dtg;
    Q.xk_l = (float)F.xk_l; Q.xk_d = (float)F.xk_d; Q.xdd = (float)F.xdd; Q.topt = (float)F.topt;
    Q.t0 = (float)F.t0; Q.tk_l = (float)F.tk_l; Q.tk_d = (float)F.tk_d;
    Q.x0 = (float)S.x0; Q.xs_l = (float)S.xs_l; Q.xs_d = (float)S.xs_d;
    Q.inv_sqrt_g = (float)(1.0 / sqrt(c.g));
    Q.p1000 = (float)(1000.0 * c.p);
    // error bound of the fp32 evaluation (derivation in dw_f32.cuh), safety factor 2 included
    const double u = 5.9604644775390625e-8, sg = sqrt(c.g), dt = fabs(c.dt);
    const double eD = sg * (400.0 * 4.5e-7 + 2.0 * u * fabs(c.temp_optimal));
    const double rbmax = dt * fmax(fabs(c.p), fabs(c.p - 2.0));
    Q.k1 = (float)(2.0 * (2.0 * eD * rbmax));
    Q.k2 = (float)(2.0 * (u * (17.0 * rbmax + 8.0 * dt)));
    Q.c0 = (float)(2.0 * (u * (2000.0 + 6000.0 * dt * fabs(c.gamma))));
    Q.c0b = (float)(4.0 * u * 1000.0 * fmax(1.0, fabs(c.p)));
    const double g2 = c.g * c.g;
    Q.xlo = (float)(g2 * P.xlo * 1.0001);
    Q.xhi = (float)(g2 * P.xhi * 0.9999);
}

// grid32 <- the current state (channels 0..6, agent stamp included)
static int materialise_f32(dw_handle *h) {
    const size_t B = h->cfg.batch, NN = h->NN;
    int rc = dev_alloc(h, &h->grid32, B * 7 * NN);
    if (!rc) rc = dev_alloc(h, &h->f32_stats, (size_t)2);
    if (rc) return rc;
    const DevParams P = make_params(h);
    F32Args A{};
    A.P = P;
    make_fast_coef(h->cfg, A.F);
    make_step_coef(h->cfg, h->L_last, A.C);
    make_f32_coef(h->cfg, A.F, A.C, P, A.Q);
    if ((P.N & 1) == 0)
        k_forward_f32<2><<<grid_for(B * NN / 2), 256, 0, h->stream>>>(A, h->lat_pre, h->lat[h->lcur], h->grid32, h->f32_stats);
    else
        k_forward_f32<1><<<grid_for(B * NN), 256, 0, h->stream>>>(A, h->lat_pre, h->lat[h->lcur], h->grid32, h->f32_stats);
    DW_LAUNCHED(h);
    if (P.n_agents > 0) {
        k_stamp_f32<<<(P.B + 127) / 128, 128, 0, h->stream>>>(P, h->grid32, h->agent_xy, h->agent_state);
        DW_LAUNCHED(h);
    }
    h->f32_cells += B * NN;
    return DW_OK;
}

extern "C" int dw_get_grid_f32(dw_handle *h, float *grid) {
    if (!h || !grid) return DW_E_INVALID;
    DW_CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    if (f32_arith_ok(h)) {
        int rc = materialise_f32(h);
        if (rc) return rc;
        DW_CUDA_TRY(h, cudaMemcpyAsync(grid, h->grid32, (size_t)h->cfg.batch * 7 * h->NN * sizeof(float), cudaMemcpyDeviceToHost, h->stream));
        DW_CUDA_TRY(h, cudaStreamSynchronize(h->stream));
        return DW_OK;
    }
    int rc = ensure_grid(h);
    if (rc) return rc;
    return export_f32(h, h->grid[h->cur], (size_t)h->cfg.batch * 7 * h->NN, grid);
}

extern "C" int dw_get_obs_f32(dw_handle *h, float *obs) {
    if (!h) return DW_E_INVALID;
    DW_CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    const size_t count = (size_t)h->cfg.batch * h->cfg.n_agents * 63;
    if (count && f32_arith_ok(h)) {
        if (!obs) return DW_E_INVALID;
        int rc = materialise_f32(h);
        if (!rc) rc = ensure_scratch(h, (count + 1) / 2);
        if (rc) return rc;
        float *tmp = reinterpret_cast<float *>(h->scratch);
        const DevParams P = make_params(h);
        k_obs_f32<<<grid_for(count), 256, 0, h->stream>>>(P, h->grid32, h->agent_xy, P.B, P.n_agents, tmp);
        DW_LAUNCHED(h);
        DW_CUDA_TRY(h, cudaMemcpyAsync(obs, tmp, count * sizeof(float), cudaMemcpyDeviceToHost, h->stream));
        DW_CUDA_TRY(h, cudaStreamSynchronize(h->stream));
        return DW_OK;
    }
    int rc = compute_obs(h);
    if (rc || !count) return rc;
    if (!obs) return DW_E_INVALID;
    return export_f32(h, h->obs, count, obs);
}

extern "C" int dw_f32_stats(dw_handle *h, uint64_t *out) {
    if (!h || !out) return DW_E_INVALID;
    DW_CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    unsigned long long t[2] = {0, 0};
    if (h->f32_stats) {
        DW_CUDA_TRY(h, cudaMemcpyAsync(t, h->f32_stats, sizeof(t), cudaMemcpyDeviceToHost, h->stream));
        DW_CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    }
    out[0] = h->f32_cells; out[1] = t[0]; out[2] = t[1];
    return DW_OK;
}

extern "C" int dw_debug_time_materialise(dw_handle *h, int32_t fp32, int32_t reps, double *ms_per_call) {
    if (!h || !ms_per_call || reps < 1) return DW_E_INVALID;
    DW_CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    if (!f32_arith_ok(h)) return dw_fail(h, DW_E_STATE, "dw_debug_time_materialise", "needs a lattice-resident state (run fused steps first)");
    cudaEvent_t e0, e1;
    DW_CUDA_TRY(h, cudaEventCreate(&e0));
    DW_CUDA_TRY(h, cudaEventCreate(&e1));
    int rc = DW_OK;
    for (int r = -1; r < reps && !rc; ++r) {           // r = -1: warm-up (allocations)
        if (r == 0) DW_CUDA_TRY(h, cudaEventRecord(e0, h->stream));
        if (fp32) rc = materialise_f32(h);
        else { h->grid_valid = false; rc = ensure_grid(h); }
    }
    DW_CUDA_TRY(h, cudaEventRecord(e1, h->stream));
    DW_CUDA_TRY(h, cudaEventSynchronize(e1));
    float ms = 0.f;
    DW_CUDA_TRY(h, cudaEventElapsedTime(&ms, e0, e1));
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    *ms_per_call = (double)ms / reps;
    return rc;
}

extern "C" int dw_get_agents(dw_handle *h, int64_t *agent_indices, double *agent_states) {
    if (!h) return DW_E_INVALID;
    DW_CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    const size_t B = h->cfg.batch, n = h->cfg.n_agents;
    if (!n) return DW_OK;
    std::vector<int32_t> xy(B * n * 2);
    if (agent_indices) DW_CUDA_TRY(h, cudaMemcpyAsync(xy.data(), h->agent_xy, xy.size() * sizeof(int32_t), cudaMemcpyDeviceToHost, h->stream));
    if (agent_states) DW_CUDA_TRY(h, cudaMemcpyAsync(agent_states, h->agent_state, B * n * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
    DW_CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    if (agent_indices) for (size_t i = 0; i < xy.size(); ++i) agent_indices[i] = xy[i];
    return DW_OK;
}

static int diag_to_scratch(dw_handle *h, int32_t which, size_t extra, size_t *count_out);

extern "C" int dw_get_diag(dw_handle *h, int32_t which, double *out) {
    if (!h || !out || which < 0 || which > DW_DIAG_GROWTH) return DW_E_INVALID;
    DW_CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    size_t count = 0;
    int rc = diag_to_scratch(h, which, 0, &count);
    if (rc) return rc;
    DW_CUDA_TRY(h, cudaMemcpyAsync(out, h->scratch, count * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
    DW_CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    return DW_OK;
}

// unrounded diagnostic field `which` of the last forward into h->scratch (count elements)
static int diag_to_scratch(dw_handle *h, int32_t which, size_t extra, size_t *count_out) {
    if (h->pre == PRE_NONE && !h->fwd_diag) return dw_fail(h, DW_E_STATE, "dw_get_diag", "no forward pass has run on this state yet");
    const DevParams P = make_params(h);
    const size_t total = (size_t)P.B * h->NN, count = total * (which == DW_DIAG_GROWTH ? 2 : 1);
    int rc = ensure_scratch(h, count + extra);
    if (rc) return rc;
    const double SL = h->cfg.S * (h->fwd_diag ? h->fwd_L : h->L_last);
    if (h->fwd_diag)       // the last forward was a standalone forward(grid) call: its input is the diagnostics' source
        k_diag<SrcGrid><<<grid_for(total), 256, 0, h->stream>>>(P, SL, SrcGrid{h->fwd_in, 7 * h->NN, h->NN}, which, h->scratch);
    else if (h->pre == PRE_GRID) k_diag<SrcGrid><<<grid_for(total), 256, 0, h->stream>>>(P, SL, SrcGrid{h->pre_grid, 7 * h->NN, h->NN}, which, h->scratch);
    else if (h->pre == PRE_COV) k_diag<SrcCov><<<grid_for(total), 256, 0, h->stream>>>(P, SL, SrcCov{h->cov, h->NN}, which, h->scratch);
    else k_diag<SrcLattice><<<grid_for(total), 256, 0, h->stream>>>(P, SL, SrcLattice{h->lat_pre, h->NN}, which, h->scratch);
    DW_LAUNCHED(h);
    *count_out = count;
    return DW_OK;
}

extern "C" int dw_get_diag_stats(dw_handle *h, int32_t which, double *out) {
    if (!h || !out || which < 0 || which > DW_DIAG_GROWTH) return DW_E_INVALID;
    DW_CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    const int blocks = 148 * 4;
    size_t count = 0;
    int rc = diag_to_scratch(h, which, (size_t)blocks * 4 + 4, &count);
    if (rc) return rc;
    double *partial = h->scratch + count, *res = partial + (size_t)blocks * 4;
    k_stats_partial<<<blocks, 256, 0, h->stream>>>(h->scratch, count, partial);
    k_stats_final<<<1, 256, 0, h->stream>>>(partial, blocks, (double)count, h->scratch, res);
    DW_LAUNCHED(h);
    DW_CUDA_TRY(h, cudaMemcpyAsync(out, res, 4 * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
    DW_CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    return DW_OK;
}

extern "C" int dw_get_cover_stats(dw_handle *h, double *out) {
    if (!h || !out) return DW_E_INVALID;
    DW_CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    const int blocks = 148 * 4;
    const size_t cells = (size_t)h->cfg.batch * h->NN;
    int rc = ensure_scratch(h, (size_t)blocks * 4 + 4 + 2 * cells);
    if (rc) return rc;
    double *partial = h->scratch, *res = partial + (size_t)blocks * 4;
    if (h->lat_valid && !h->grid_valid) {
        k_lattice_cover_partial<<<blocks, 256, 0, h->stream>>>(h->lat[h->lcur], cells, partial);
        k_cover_final<<<1, 256, 0, h->stream>>>(partial, blocks, (double)cells, res);
        DW_LAUNCHED(h);
    } else {
        // fp64 representations: two passes of the generic reduction over the light / dark planes
        rc = ensure_grid(h);
        if (rc) return rc;
        double *planes = res + 4, tmp[8];
        for (int c = 0; c < 2; ++c) {
            DW_CUDA_TRY(h, cudaMemcpy2DAsync(planes, h->NN * sizeof(double), h->grid[h->cur] + (size_t)(1 + c) * h->NN, 7 * h->NN * sizeof(double),
                                             h->NN * sizeof(double), h->cfg.batch, cudaMemcpyDeviceToDevice, h->stream));
            k_stats_partial<<<blocks, 256, 0, h->stream>>>(planes, cells, partial);
            k_stats_final<<<1, 256, 0, h->stream>>>(partial, blocks, (double)cells, planes, res);
            DW_LAUNCHED(h);
            DW_CUDA_TRY(h, cudaMemcpyAsync(tmp + 4 * c, res, 4 * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
            DW_CUDA_TRY(h, cudaStreamSynchronize(h->stream));
        }
        out[0] = tmp[0]; out[1] = tmp[4]; out[2] = tmp[3]; out[3] = tmp[7];
        return DW_OK;
    }
    DW_CUDA_TRY(h, cudaMemcpyAsync(out, res, 4 * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
    DW_CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    return DW_OK;
}

// ---- lifespan runs ---------------------------------------------------------------------------------------
extern "C" int dw_reset_lifespans(dw_handle *h) {
    if (!h) return DW_E_INVALID;
    DW_CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    const size_t B = h->cfg.batch, n = h->cfg.n_agents;
    DW_CUDA_TRY(h, cudaMemsetAsync(h->done_at, 0, B * sizeof(int64_t), h->stream));
    if (n) DW_CUDA_TRY(h, cudaMemsetAsync(h->agents_done_at, 0, B * n * sizeof(int64_t), h->stream));
    return DW_OK;
}

extern "C" int dw_get_lifespans(dw_handle *h, int64_t *done_at, int64_t *agents_done_at) {
    if (!h) return DW_E_INVALID;
    DW_CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    const size_t B = h->cfg.batch, n = h->cfg.n_agents;
    if (done_at) DW_CUDA_TRY(h, cudaMemcpyAsync(done_at, h->done_at, B * sizeof(int64_t), cudaMemcpyDeviceToHost, h->stream));
    if (agents_done_at && n)
        DW_CUDA_TRY(h, cudaMemcpyAsync(agents_done_at, h->agents_done_at, B * n * sizeof(int64_t), cudaMemcpyDeviceToHost, h->stream));
    DW_CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    return DW_OK;
}

__global__ void k_lifespan_stats(int B, int n, const int64_t *done_at, const int64_t *agents_done_at, const unsigned int *alive_last,
                                 double *out) {
    // single block; exact in fp64 for any realistic ensemble (integers < 2^53)
    __shared__ double sh[6][32];
    double s[5] = {0, 0, 0, 0, 0};
    for (int b = threadIdx.x; b < B; b += blockDim.x) {
        const double v = (double)done_at[b];
        s[0] += v; s[1] += v * v;
        for (int i = 0; i < n; ++i) {
            const double a = (double)agents_done_at[(size_t)b * n + i];
            s[2] += a; s[3] += a * a;
        }
    }
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    for (int k = 0; k < 4; ++k) {
        double v = s[k];
        for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
        if (lane == 0) sh[k][w] = v;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        double t[4] = {0, 0, 0, 0};
        for (int k = 0; k < 4; ++k) for (int i = 0; i < (int)(blockDim.x >> 5); ++i) t[k] += sh[k][i];
        out[0] = (double)B; out[1] = t[0]; out[2] = t[1]; out[3] = (double)B * n; out[4] = t[2]; out[5] = t[3];
        out[6] = alive_last ? (double)*alive_last : 0.0; out[7] = 0.0;
    }
}

extern "C" int dw_lifespan_stats_device(dw_handle *h, double *out_dev) {
    if (!h || !out_dev) return DW_E_INVALID;
    DW_CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    k_lifespan_stats<<<1, 1024, 0, h->stream>>>(h->cfg.batch, h->cfg.n_agents, h->done_at, h->agents_done_at, nullptr, out_dev);
    DW_LAUNCHED(h);
    return DW_OK;
}

// ---- checkpoint ---------------------------------------------------------------------------------------------
static int ckpt_save(dw_handle *h, int slot) {
    const size_t B = h->cfg.batch, n = h->cfg.n_agents, NN = h->NN;
    auto &c = h->ck[slot];
    int rc = DW_OK;
    if (h->grid_valid) {
        rc = dev_alloc(h, &c.grid, B * 7 * NN);
        if (rc) return rc;
        DW_CUDA_TRY(h, cudaMemcpyAsync(c.grid, h->grid[h->cur], B * 7 * NN * sizeof(double), cudaMemcpyDeviceToDevice, h->stream));
    }
    c.have_cov = h->cov_valid || h->pre == PRE_COV;
    if (c.have_cov) {
        rc = dev_alloc(h, &c.cov, B * 2 * NN);
        if (rc) return rc;
        DW_CUDA_TRY(h, cudaMemcpyAsync(c.cov, h->cov, B * 2 * NN * sizeof(double), cudaMemcpyDeviceToDevice, h->stream));
    }
    c.cov_valid = h->cov_valid;
    c.cov_L = h->cov_L;
    if (h->lat_valid) {
        rc = dev_alloc(h, &c.lat, B * NN);
        if (!rc) rc = dev_alloc(h, &c.lat_pre, B * NN);
        if (rc) return rc;
        DW_CUDA_TRY(h, cudaMemcpyAsync(c.lat, h->lat[h->lcur], B * NN * sizeof(uint32_t), cudaMemcpyDeviceToDevice, h->stream));
        if (h->pre == PRE_LAT)
            DW_CUDA_TRY(h, cudaMemcpyAsync(c.lat_pre, h->lat_pre, B * NN * sizeof(uint32_t), cudaMemcpyDeviceToDevice, h->stream));
    }
    rc = dev_alloc(h, &c.agent_xy, B * n * 2);
    if (!rc) rc = dev_alloc(h, &c.agent_state, B * n);
    if (!rc) rc = dev_alloc(h, &c.done_at, B);
    if (!rc) rc = dev_alloc(h, &c.agents_done_at, B * n);
    if (rc) return rc;
    if (n) {
        DW_CUDA_TRY(h, cudaMemcpyAsync(c.agent_xy, h->agent_xy, B * n * 2 * sizeof(int32_t), cudaMemcpyDeviceToDevice, h->stream));
        DW_CUDA_TRY(h, cudaMemcpyAsync(c.agent_state, h->agent_state, B * n * sizeof(double), cudaMemcpyDeviceToDevice, h->stream));
        DW_CUDA_TRY(h, cudaMemcpyAsync(c.agents_done_at, h->agents_done_at, B * n * sizeof(int64_t), cudaMemcpyDeviceToDevice, h->stream));
    }
    DW_CUDA_TRY(h, cudaMemcpyAsync(c.done_at, h->done_at, B * sizeof(int64_t), cudaMemcpyDeviceToDevice, h->stream));
    c.have = true; c.grid_valid = h->grid_valid; c.lat_valid = h->lat_valid; c.clk = h->clk;
    // a PRE_GRID pre-state lives in the other ping-pong buffer and is not checkpointed: diagnostics of the
    // step before the checkpoint are not restorable, the state itself is.
    c.pre = (h->pre == PRE_LAT || h->pre == PRE_COV) ? h->pre : PRE_NONE;
    c.L_last = h->L_last;
    c.ch6_dirty_saved = h->ch6_dirty[h->cur];
    return DW_OK;
}

static int ckpt_restore(dw_handle *h, int slot) {
    auto &c = h->ck[slot];
    if (!c.have) return dw_fail(h, DW_E_STATE, "dw_checkpoint_restore", "no checkpoint saved");
    const size_t B = h->cfg.batch, n = h->cfg.n_agents, NN = h->NN;
    if (c.grid_valid) {
        int rc = ensure_grid_buffers(h);
        if (rc) return rc;
        DW_CUDA_TRY(h, cudaMemcpyAsync(h->grid[h->cur], c.grid, B * 7 * NN * sizeof(double), cudaMemcpyDeviceToDevice, h->stream));
    }
    if (c.have_cov) {
        int rc = dev_alloc(h, &h->cov, B * 2 * NN);
        if (rc) return rc;
        DW_CUDA_TRY(h, cudaMemcpyAsync(h->cov, c.cov, B * 2 * NN * sizeof(double), cudaMemcpyDeviceToDevice, h->stream));
    }
    h->cov_valid = c.cov_valid;
    h->cov_L = c.cov_L;
    if (c.lat_valid) {
        DW_CUDA_TRY(h, cudaMemcpyAsync(h->lat[h->lcur], c.lat, B * NN * sizeof(uint32_t), cudaMemcpyDeviceToDevice, h->stream));
        if (c.pre == PRE_LAT)
            DW_CUDA_TRY(h, cudaMemcpyAsync(h->lat_pre, c.lat_pre, B * NN * sizeof(uint32_t), cudaMemcpyDeviceToDevice, h->stream));
    }
    if (n) {
        DW_CUDA_TRY(h, cudaMemcpyAsync(h->agent_xy, c.agent_xy, B * n * 2 * sizeof(int32_t), cudaMemcpyDeviceToDevice, h->stream));
        DW_CUDA_TRY(h, cudaMemcpyAsync(h->agent_state, c.agent_state, B * n * sizeof(double), cudaMemcpyDeviceToDevice, h->stream));
        DW_CUDA_TRY(h, cudaMemcpyAsync(h->agents_done_at, c.agents_done_at, B * n * sizeof(int64_t), cudaMemcpyDeviceToDevice, h->stream));
    }
    DW_CUDA_TRY(h, cudaMemcpyAsync(h->done_at, c.done_at, B * sizeof(int64_t), cudaMemcpyDeviceToDevice, h->stream));
    h->grid_valid = c.grid_valid; h->lat_valid = c.lat_valid; h->clk = c.clk; h->pre = c.pre; h->L_last = c.L_last;
    if (c.grid_valid) h->ch6_dirty[h->cur] = c.ch6_dirty_saved;   // the flags describe physical buffers: `cur` may have flipped since the save
    state_changed(h);
    return DW_OK;
}

extern "C" int dw_checkpoint_save(dw_handle *h) {
    if (!h) return DW_E_INVALID;
    DW_CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    return ckpt_save(h, 0);
}
extern "C" int dw_checkpoint_restore(dw_handle *h) {
    if (!h) return DW_E_INVALID;
    DW_CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    return ckpt_restore(h, 0);
}

extern "C" int dw_set_profiling(dw_handle *h, int32_t on) {
    if (!h) return DW_E_INVALID;
    DW_CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    if (on && !h->ev[0]) {
        DW_CUDA_TRY(h, cudaEventCreate(&h->ev[0]));
        DW_CUDA_TRY(h, cudaEventCreate(&h->ev[1]));
    }
    h->profiling = on != 0;
    h->prof = dw_profile{};
    h->ev_pending = false;
    return DW_OK;
}
extern "C" int dw_get_profile(dw_handle *h, dw_profile *out) {
    if (!h || !out) return DW_E_INVALID;
    *out = h->prof;
    return DW_OK;
}

// FP64 FMA peak of the device, measured: the roofline denominator of the fused kernel (MEASURED_PEAKS.json has
// only HBM and bf16 numbers). 8 independent DFMA chains per thread, 2048 resident threads per SM.
__global__ void __launch_bounds__(256) k_fp64_peak(double *out, int iters, double a, double b) {
    double v[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) v[i] = (double)(threadIdx.x + i);
    for (int it = 0; it < iters; ++it) {
#pragma unroll
        for (int i = 0; i < 8; ++i) v[i] = __fma_rn(v[i], a, b);
    }
    double s = 0;
#pragma unroll
    for (int i = 0; i < 8; ++i) s += v[i];
    if (s == 12345.678) out[0] = s;   // keep the chains alive
}

extern "C" int dw_debug_fp64_peak(dw_handle *h, int32_t iters, int32_t reps, double *tflops_best, double *ms_best) {
    if (!h || iters < 1 || reps < 1 || !tflops_best) return DW_E_INVALID;
    DW_CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    int rc = ensure_scratch(h, 16);
    if (rc) return rc;
    cudaEvent_t e0, e1;
    DW_CUDA_TRY(h, cudaEventCreate(&e0));
    DW_CUDA_TRY(h, cudaEventCreate(&e1));
    int sms = 148;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, h->cfg.device);
    const int blocks = sms * 8, threads = 256;
    double best = 1e30;
    for (int r = 0; r < reps + 1; ++r) {
        DW_CUDA_TRY(h, cudaEventRecord(e0, h->stream));
        k_fp64_peak<<<blocks, threads, 0, h->stream>>>(h->scratch, iters, 0.999999, 1e-9);
        DW_CUDA_TRY(h, cudaGetLastError());
        DW_CUDA_TRY(h, cudaEventRecord(e1, h->stream));
        DW_CUDA_TRY(h, cudaEventSynchronize(e1));
        float ms = 0;
        DW_CUDA_TRY(h, cudaEventElapsedTime(&ms, e0, e1));
        if (r > 0 && ms < best) best = ms;
    }
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    const double flops = 2.0 * 8.0 * (double)iters * (double)blocks * threads;
    *tflops_best = flops / (best * 1e-3) / 1e12;
    if (ms_best) *ms_best = best;
    return DW_OK;
}

// ---- diagnostics hooks -------------------------------------------------------------------------------------
extern "C" int dw_set_world_offset(dw_handle *h, uint32_t world0) {
    if (!h) return DW_E_INVALID;
    h->world0 = world0;
    return DW_OK;
}

extern "C" int dw_debug_state(dw_handle *h, int32_t *flags) {
    if (!h || !flags) return DW_E_INVALID;
    flags[0] = h->grid_valid; flags[1] = h->lat_valid; flags[2] = h->cov_valid; flags[3] = (int32_t)h->pre;
    return DW_OK;
}

extern "C" int dw_debug_slow_count(dw_handle *h, uint64_t *count, int32_t reset) {
    if (!h || !count) return DW_E_INVALID;
    DW_CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    *count = 0;
    if (!h->slow_count) return DW_OK;
    unsigned int c = 0;
    DW_CUDA_TRY(h, cudaMemcpyAsync(&c, h->slow_count, sizeof(c), cudaMemcpyDeviceToHost, h->stream));
    DW_CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    *count = c;
    if (reset) DW_CUDA_TRY(h, cudaMemsetAsync(h->slow_count, 0, sizeof(unsigned int), h->stream));
    return DW_OK;
}

extern "C" int dw_debug_markstein(dw_handle *h, uint32_t kmax, uint32_t *bad) {
    if (!h || !bad) return DW_E_INVALID;
    DW_CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    int rc = dev_alloc(h, &h->slow_count, (size_t)2);
    if (rc) return rc;
    DW_CUDA_TRY(h, cudaMemsetAsync(h->slow_count + 1, 0, sizeof(unsigned int), h->stream));
    k_debug_markstein<<<148 * 4, 256, 0, h->stream>>>(kmax, h->slow_count + 1);
    DW_CUDA_TRY(h, cudaGetLastError());
    DW_CUDA_TRY(h, cudaMemcpyAsync(bad, h->slow_count + 1, sizeof(unsigned int), cudaMemcpyDeviceToHost, h->stream));
    DW_CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    return DW_OK;
}

extern "C" int dw_debug_markstein_f32(dw_handle *h, uint32_t kmax, uint32_t *bad) {
    if (!h || !bad) return DW_E_INVALID;
    DW_CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    int rc = dev_alloc(h, &h->slow_count, (size_t)2);
    if (rc) return rc;
    DW_CUDA_TRY(h, cudaMemsetAsync(h->slow_count + 1, 0, sizeof(unsigned int), h->stream));
    k_debug_markstein_f32<<<148 * 4, 256, 0, h->stream>>>(kmax, h->slow_count + 1);
    DW_CUDA_TRY(h, cudaGetLastError());
    DW_CUDA_TRY(h, cudaMemcpyAsync(bad, h->slow_count + 1, sizeof(unsigned int), cudaMemcpyDeviceToHost, h->stream));
    DW_CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    return DW_OK;
}

extern "C" int dw_debug_root4(dw_handle *h, const double *x, double *y, int32_t n) {
    if (!h || !x || !y || n < 1) return DW_E_INVALID;
    DW_CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    int rc = ensure_scratch(h, 2 * (size_t)n);
    if (rc) return rc;
    DW_CUDA_TRY(h, cudaMemcpyAsync(h->scratch, x, n * sizeof(double), cudaMemcpyHostToDevice, h->stream));
    k_debug_root4<<<(n + 255) / 256, 256, 0, h->stream>>>(h->scratch, h->scratch + n, n);
    DW_LAUNCHED(h);
    DW_CUDA_TRY(h, cudaMemcpyAsync(y, h->scratch + n, n * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
    DW_CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    return DW_OK;
}

// ---- dw_run / dw_run_chunk ----------------------------------------------------------------------------------
#include "dw_run.inl"

// ---- single giant grid (include/daisyworld_b200_tiled.h) -----------------------------------------------------
#include "dw_tiled_api.inl"
