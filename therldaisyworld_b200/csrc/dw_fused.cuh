// Fused multi-step lattice kernels: one CTA owns one world in shared memory and runs K env steps per launch.
//
// After the first forward pass every cover value is k/1000 with integer k in [0,1000] (np.round(.,3),
// daisy_world_rl.py:452), so a world is stored as one packed u32 per cell (light k | dark k << 16): 16 KB for
// 64x64.  The 3x3 stencils become exact integer sums on the packed words (ALU pipe), and the per-cell physics is
// a short fp64 sequence ("fast path") that is algebraically equal to the reference formulas but not in the
// reference's rounding order.  Exactness is restored by a filter: the fast path's result x (in milli-cover
// units) has a proven error bound far below the filter width; whenever x lies within the filter (F.tie_*) of a rounding
// tie the cell is recomputed by dw_literal_cell() in the oracle's operation order.  Everything else the step
// needs (agent moves, grazing, greedy argmax, lifespan counters) follows the literal order as well, so a fused
// run is value-identical to stepping the oracle -- tests/test_gpu_run_parity.py.
//
// Roofline: the kernel is bound by the FP64 pipe (64 DFMA/clk/SM); HBM traffic is 8 B per cell per LAUNCH.
#pragma once
#include <type_traits>
#include "dw_common.cuh"

constexpr int kTileRowUnroll = 4;       // unroll factor of the 4-row tile loop (1 keeps the body inside the i-cache)
constexpr int kN64MinBlocks = 4;        // resident CTAs per SM the 64x64 and sub-64 kernels are compiled for (64 registers)
#define DW_FUSED_MAX_STEPS 4096        // longest launch (coefficient table / alive counters)
#define DW_FUSED_MAX_AGENTS 1024
#define DW_FIX_BITS 20                 // fixed-point fraction bits of the rounding trick (ulp of 1.5*2^32)
#define DW_TIE_EPS_MIN 4               // smallest filter half-width in units of 2^-DW_FIX_BITS (3.8e-6 milli-cover); the host widens
#define DW_TIE_EPS_MAX 256             // it per handle from the physics constants (make_fast_coef, error budget in DESIGN.md section 2)

// The fast path works with X' = g^2 * X (X = T_l^4 resp. T_d^4): its fourth root is T' = sqrt(g)*T, so that
// beta = 1 - g*(Topt-T)^2 = 1 - (sqrt(g)*Topt - T')^2 is ONE fma.  All X coefficients below carry the factor g^2.
struct FastCoef {        // launch-constant coefficients of the fast path (host-computed, fp64)
    double w0, w12, w2;  // rho (milli) = w0*k + (w1-w2)*E + w2*S8
    double dtp, dtm, dtg;  // dt*p, dt/1000, dt*gamma
    double xk_l, xk_d;   // g^2 * X_l coefficients of the centre covers: (q2-q)*(al-ab)/1000, (q2-q)*(ad-ab)/1000
    double xdd;          // g^2 * (X_d - X_l) = g^2 * q2*(al-ad)
    double topt;         // sqrt(g) * Topt
    // series mode: X_T = T^4 (scaled by g^2) = X_l + t0 + tk_l*kl + tk_d*kd, with t0 = -g^2 q2 (Al0 - al), tk = -g^2 q2 (a - ab)/1000
    double t0, tk_l, tk_d;
    // rounding + tie filter (see DW rounding note below): magic = 1.5*2^32 + 0.5 + eps*2^-FIX, tie_thresh = (2 eps) << (32-FIX)
    double magic;
    unsigned int tie_thresh, pad_;
    // Unused. Keeps sizeof(FastCoef) and the offsets of the members after it in FusedArgs / LookArgs: the kernels that take
    // them sit at 64 registers and their register allocation (and local-memory use) reacts to parameter offsets.
    double pad_layout_[3];
};
struct StepCoef {        // per-step (luminosity dependent) coefficients
    double x0;           // g^2 * (cL + (q-cL)*A0 + (q2-q)*Al0 - q2*al)
    double pad_layout_;  // unused; keeps the 48-byte layout (without it k_tiled_step spills inside the DFMA chain)
    double xs_l, xs_d;   // g^2 * (q-cL)*a*(al-ab)/1000, g^2 * (q-cL)*a*(ad-ab)/1000   (a = adjacent tap)
    double SL;           // S*L for the literal path
    int policy, pad_;    // the policy of this step (DW_POLICY_EPS_GREEDY resolved to GREEDY / RANDOM on the host)
};

struct FusedArgs {
    DevParams P;
    FastCoef F;
    const StepCoef *sc;         // [K] per-step coefficients (global memory)
    const uint32_t *lat_in;     // [B,N,N]
    uint32_t *lat;              // [B,N,N] in-place state (persistent kernel)
    uint32_t *lat_out;          // [B,N,N]
    uint32_t *lat_pre;          // [B,N,N] post-graze state the LAST step of the launch started from
    int32_t *agent_xy;          // [B,n,2]
    double *agent_state;        // [B,n]
    const int8_t *actions;      // [K,B,n] (REPLAY)
    int64_t *done_at;           // [B]
    int64_t *agents_done_at;    // [B,n]
    unsigned int *alive;        // [K] per-step count of worlds that are not grid_done
    double *reward;             // [B,n] or [B,2]
    uint8_t *done;
    unsigned long long seed;
    unsigned int step0;         // env.step_count at launch (RANDOM policy counter)
    unsigned int world0;        // global index of this handle's first world (RANDOM policy counter)
    int K, policy;
    int count_life, pad2_;      // 1: add this launch's steps to the lifespan counters done_at / agents_done_at (dw_run); 0: step()
    unsigned int *slow_count;   // diagnostics: number of literal recomputations (may be NULL)
    // series mode (k_fused_n64_persist<true>): per-step ensemble sums, [K] each: sqrt(g)*T of the step's forward (unrounded),
    // light and dark milli-cover after the step
    double *series_T;
    unsigned long long *series_l, *series_d;
    // persistent kernel only
    int Kc;                     // steps per work item
    int n_pairs, n_chunks;      // work items = n_pairs (worlds) * n_chunks, chunk-major
    unsigned int *queue;        // [1] next work item (zeroed before the launch)
    unsigned int *pair_done;    // [n_pairs] chunks completed per world (zeroed before the launch)
    // DW_POLICY_MLP inside the persistent 64x64 kernel (k_fused_n64_persist<.., true>)
    const double *mlp_w;        // [sets][DW_MLP_PARAMS] network weights (device)
    int mlp_wpm, mlp_half, mlp_adv, pad3_;   // population mode (wpm > 0): worlds per member, agents on the member's net, adversary set
    double SL_prev;             // S*L of the step before the launch's first one (observation windows of step 0)
    double *rew_series;         // [K][B*n] agent states after each step's update_agents (population post-pass, k_pop_post), or NULL
    // [B*n] bit j = "agent was not done after step j of this launch" (K <= 64), or NULL: lets a statistics-only caller that ran
    // past the notebook's stopping step take the surplus out of agents_done_at instead of rewinding (dw_trim_lifespans)
    unsigned long long *alive_mask;
};

__device__ __forceinline__ double dw_u2d(uint32_t k) {        // exact u32 -> f64 through the 2^52 trick
    return __hiloint2double(0x43300000, (int)k) - 4503599627370496.0;
}
// Packed half -> f64 by I2F.F64.U16: one issue slot on the XU pipe. The 2^52 trick of dw_u2d costs three issue slots and
// two cycles of the FP64 pipe, which bounds dw_fast_cells (DESIGN.md section 4).
template <bool HI>
__device__ __forceinline__ double dw_half2d(uint32_t p) {
    return HI ? (double)(unsigned short)(p >> 16) : (double)(unsigned short)(p & 0xffffu);
}
// Rounding of x (milli units) to the lattice with the tie filter folded into ONE add: v = x + (1.5*2^32 + 0.5 + EPS*2^-FIX)
// has the ulp 2^-FIX, and its mantissa holds round((x + 0.5) * 2^FIX) + EPS as a signed fixed-point number F offset by 2^51
// (|x| < 2^31). f = low word of v, h = high word:
//   tie flag: frac(x + .5) * 2^FIX + EPS (mod 2^FIX) < 2 EPS   <=>   (unsigned)(f << (32-FIX)) < F.tie_thresh;
//   floor(x + .5) = F >> FIX   unless frac(x + .5) is within EPS*2^-FIX below 1 -- but then the cell is flagged anyway.
// The low word alone holds only 12 integer bits of F >> FIX and wraps modulo 4096 outside x + .5 in [-2048, 2048): a cell that
// dies by 2100 milli-cover in one step would come back at 1000. So the value is taken with ONE funnel shift of both words,
// (h:f) >> FIX, whose low 16 bits are F >> FIX exactly for x + .5 in [-32768, 32768) (DW_WIDE_WINDOW) -- the same instruction
// count as a shift of f alone. The s16x2 clamp to [0, 1000] then saturates like the reference's clip (which comes before its
// rounding). dw_fast_cell saturates any x; the tile loops' dw_fast_cells stay exact inside the 16-bit window, which holds
// every cell update whose bound |x - k| <= rho_max (rho_b,max |beta|_max + dt gamma) is below 31768 (DESIGN.md section 2).
// EPS is chosen per handle on the host (F.magic, F.tie_thresh).
#define DW_WIDE_WINDOW 32768
#define DW_MAGIC_HI 0x41F80000      // high word of v for x + .5 in [0, 4096): (h - DW_MAGIC_HI) = F >> 32

// floor(x + .5) clamped to [0, 1000] from the words of v, for any x. Inf and NaN sums (X' <= 0: NaN temperatures, where the
// reference's grid is NaN too) keep what the low word always gave them, (f >> FIX) clamped.
__device__ __forceinline__ unsigned dw_round_any(int h, int f) {
    if ((h & 0x7ff00000) == 0x7ff00000) return (unsigned)min(max(f >> DW_FIX_BITS, 0), 1000);
    if (h < 0x41F00000 || h > 0x41FFFFFF) return h > DW_MAGIC_HI ? 1000u : 0u;    // |x| >= 2^31 (signed: v < 0 is below)
    const long long F = ((long long)(h - DW_MAGIC_HI) << 32) + (long long)(unsigned)f;
    return (unsigned)min(max(F >> DW_FIX_BITS, 0ll), 1000ll);
}

// One cell of the fast path. pc: packed centre, E: packed sum of the 4 edge neighbours, S: packed sum of all 8.
// Returns the packed new cell; *tiemin is lowered below F.tie_thresh when either species sits within the filter of
// a rounding tie (the caller then recomputes the cell in literal order).
// Straight-line (no branches) so that several cells can be interleaved by the scheduler.
__device__ __forceinline__ uint32_t dw_fast_cell(const FastCoef &F, const StepCoef &C, uint32_t pc, uint32_t E, uint32_t S,
                                                 unsigned *tiemin) {
    const double kl = dw_u2d(pc & 0xffffu), kd = dw_u2d(pc >> 16);
    const double El = dw_u2d(E & 0xffffu), Ed = dw_u2d(E >> 16);
    const double Sl = dw_u2d(S & 0xffffu), Sd = dw_u2d(S >> 16);
    const double Rl = __fma_rn(F.w2, Sl, __fma_rn(F.w12, El, F.w0 * kl));
    const double Rd = __fma_rn(F.w2, Sd, __fma_rn(F.w12, Ed, F.w0 * kd));
    const double rb = __fma_rn(-F.dtm, Rl + Rd, F.dtp);                       // dt * bare neighbourhood density
    const double Xl = __fma_rn(C.xs_l, Sl, __fma_rn(C.xs_d, Sd, __fma_rn(F.xk_l, kl, __fma_rn(F.xk_d, kd, C.x0))));
    const double Xd = Xl + F.xdd;
    const double dTl = F.topt - dw_root4_fast(Xl);                            // sqrt(g) * (Topt - T_l)
    const double dTd = F.topt - dw_root4_fast(Xd);
    const double bl = __fma_rn(-dTl, dTl, 1.0);
    const double bd = __fma_rn(-dTd, dTd, 1.0);
    const double xl = __fma_rn(Rl, __fma_rn(rb, bl, -F.dtg), kl);             // l + dt*dl in milli units
    const double xd = __fma_rn(Rd, __fma_rn(rb, bd, -F.dtg), kd);
    const double vl = xl + F.magic, vd = xd + F.magic;
    const int fl = __double2loint(vl), fd = __double2loint(vd), hl = __double2hiint(vl), hd = __double2hiint(vd);
    *tiemin = __vimin3_u32(*tiemin, (unsigned)fl << (32 - DW_FIX_BITS), (unsigned)fd << (32 - DW_FIX_BITS));
    // outside the 16-bit window of the tile loops' rounding (rare): saturate
    if ((unsigned)(hl - (DW_MAGIC_HI - 8)) >= 16u || (unsigned)(hd - (DW_MAGIC_HI - 8)) >= 16u)
        return dw_round_any(hl, fl) | (dw_round_any(hd, fd) << 16);
    // floor(x + .5) of both species packed as s16x2, clamped to [0,1000] by one VIMNMX.S16x2.RELU
    const unsigned packed = __byte_perm(__funnelshift_r(fl, hl, DW_FIX_BITS), __funnelshift_r(fd, hd, DW_FIX_BITS), 0x5410);
    return __vimin_s16x2_relu(packed, 1000u | (1000u << 16));
}

// Two cells in explicit lockstep: the fp64 chain of one cell is serial (8-cycle dependent latency, measured), so the
// source interleaves two independent cells statement by statement to give the scheduler ILP without more warps.
// DIAG: tcells = how many of the W cells (a prefix) add their temperature to *tsum (cells outside a partial tile do not).
template <int W, bool DIAG = false>
__device__ __forceinline__ void dw_fast_cells(const FastCoef &F, const StepCoef &C, const uint32_t (&pc)[W], const uint32_t (&E)[W],
                                              const uint32_t (&S)[W], unsigned *tiemin, uint32_t (&out)[W], double *tsum = nullptr,
                                              int tcells = W) {
    double kl[W], kd[W], El[W], Ed[W], Sl[W], Sd[W], Rl[W], Rd[W], rb[W], Xl[W], Xd[W];
#pragma unroll
    for (int i = 0; i < W; ++i) { kl[i] = dw_half2d<false>(pc[i]); kd[i] = dw_half2d<true>(pc[i]); }
#pragma unroll
    for (int i = 0; i < W; ++i) { Sl[i] = dw_half2d<false>(S[i]); Sd[i] = dw_half2d<true>(S[i]); }
#pragma unroll
    for (int i = 0; i < W; ++i) Xl[i] = __fma_rn(F.xk_l, kl[i], __fma_rn(F.xk_d, kd[i], C.x0));
#pragma unroll
    for (int i = 0; i < W; ++i) Xl[i] = __fma_rn(C.xs_l, Sl[i], __fma_rn(C.xs_d, Sd[i], Xl[i]));
#pragma unroll
    for (int i = 0; i < W; ++i) Xd[i] = Xl[i] + F.xdd;
    if (DIAG) {              // series mode: the (unrounded) temperature of the cell itself, sqrt(g)*T, summed per thread
#pragma unroll
        for (int i = 0; i < W; ++i)
            if (i < tcells) *tsum += dw_root4_fast(__fma_rn(F.tk_l, kl[i], __fma_rn(F.tk_d, kd[i], Xl[i] + F.t0)));
    }
    // seeds first: the MUFU latency (27 cycles) overlaps the rho arithmetic below
    double s1l[W], s1d[W], y0l[W], y0d[W];
#pragma unroll
    for (int i = 0; i < W; ++i) { s1l[i] = dw_rsqrt_approx(Xl[i]); s1d[i] = dw_rsqrt_approx(Xd[i]); }
#pragma unroll
    for (int i = 0; i < W; ++i) { El[i] = dw_half2d<false>(E[i]); Ed[i] = dw_half2d<true>(E[i]); }
#pragma unroll
    for (int i = 0; i < W; ++i) { Rl[i] = F.w0 * kl[i]; Rd[i] = F.w0 * kd[i]; }
#pragma unroll
    for (int i = 0; i < W; ++i) { y0l[i] = dw_rsqrt_approx(s1l[i]); y0d[i] = dw_rsqrt_approx(s1d[i]); }
#pragma unroll
    for (int i = 0; i < W; ++i) { Rl[i] = __fma_rn(F.w12, El[i], Rl[i]); Rd[i] = __fma_rn(F.w12, Ed[i], Rd[i]); }
#pragma unroll
    for (int i = 0; i < W; ++i) { Rl[i] = __fma_rn(F.w2, Sl[i], Rl[i]); Rd[i] = __fma_rn(F.w2, Sd[i], Rd[i]); }
#pragma unroll
    for (int i = 0; i < W; ++i) rb[i] = __fma_rn(-F.dtm, Rl[i] + Rd[i], F.dtp);
    // Newton step on y^4 = X for both species of all cells, stage by stage
    double zl[W], zd[W], al[W], ad[W];
    // The step of dw_root4_fast with one fp64 operation less per root: T = y0 + (X - y0^4) * (s1/2)^2 * y0 with s1/2 made by an
    // integer subtract on the exponent (ALU pipe; the MUFU seed's low word is zero), and Topt - T folded into the last FMA:
    // dT = (Topt - y0) - ((X - y0^4) * (s1/2)^2) * y0.
#pragma unroll
    for (int i = 0; i < W; ++i) {
        const double hl = __hiloint2double(__double2hiint(s1l[i]) - 0x00100000, 0), hd = __hiloint2double(__double2hiint(s1d[i]) - 0x00100000, 0);
        zl[i] = y0l[i] * y0l[i]; zd[i] = y0d[i] * y0d[i]; al[i] = hl * hl; ad[i] = hd * hd;
    }
#pragma unroll
    for (int i = 0; i < W; ++i) { zl[i] = __fma_rn(-zl[i], zl[i], Xl[i]); zd[i] = __fma_rn(-zd[i], zd[i], Xd[i]); }
#pragma unroll
    for (int i = 0; i < W; ++i) { zl[i] = zl[i] * al[i]; zd[i] = zd[i] * ad[i]; al[i] = F.topt - y0l[i]; ad[i] = F.topt - y0d[i]; }
#pragma unroll
    for (int i = 0; i < W; ++i) { zl[i] = __fma_rn(-zl[i], y0l[i], al[i]); zd[i] = __fma_rn(-zd[i], y0d[i], ad[i]); }   // sqrt(g)*(Topt-T)
#pragma unroll
    for (int i = 0; i < W; ++i) { zl[i] = __fma_rn(-zl[i], zl[i], 1.0); zd[i] = __fma_rn(-zd[i], zd[i], 1.0); }       // beta_l, beta_d
#pragma unroll
    for (int i = 0; i < W; ++i) { zl[i] = __fma_rn(rb[i], zl[i], -F.dtg); zd[i] = __fma_rn(rb[i], zd[i], -F.dtg); }
#pragma unroll
    for (int i = 0; i < W; ++i) { zl[i] = __fma_rn(Rl[i], zl[i], kl[i]); zd[i] = __fma_rn(Rd[i], zd[i], kd[i]); }     // l + dt*dl (milli)
#pragma unroll
    for (int i = 0; i < W; ++i) {
        const double vl = zl[i] + F.magic, vd = zd[i] + F.magic;
        const int fl = __double2loint(vl), fd = __double2loint(vd);
        *tiemin = __vimin3_u32(*tiemin, (unsigned)fl << (32 - DW_FIX_BITS), (unsigned)fd << (32 - DW_FIX_BITS));
        // funnel shift of both words: exact inside DW_WIDE_WINDOW (see the rounding note)
        const unsigned packed = __byte_perm(__funnelshift_r(fl, __double2hiint(vl), DW_FIX_BITS),
                                            __funnelshift_r(fd, __double2hiint(vd), DW_FIX_BITS), 0x5410);
        out[i] = __vimin_s16x2_relu(packed, 1000u | (1000u << 16));
    }
}

// Literal recomputation of one cell from the packed neighbourhood (oracle order). Rare: ~1e-5 of cell-updates.
__device__ __noinline__ uint32_t dw_slow_cell(const FusedArgs *A, double SL, const uint32_t *cb, int N, int x, int y, int ld = 0) {
    if (ld == 0) ld = N;
    const int xm = x == 0 ? N - 1 : x - 1, xp = x == N - 1 ? 0 : x + 1;
    const int ym = y == 0 ? N - 1 : y - 1, yp = y == N - 1 ? 0 : y + 1;
    const int xs[3] = {xm, x, xp}, ys[3] = {ym, y, yp};
    double l9[9], d9[9];
#pragma unroll
    for (int a = 0; a < 3; ++a)
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            const uint32_t k = cb[xs[a] * ld + ys[c]];
            l9[a * 3 + c] = dw_milli(k & 0xffffu);
            d9[a * 3 + c] = dw_milli(k >> 16);
        }
    const LitCell o = dw_literal_cell(A->P, SL, l9, d9);
    // np.round(x,3) = rint(x*1000)/1000  ->  lattice index rint(x*1000)
    const int ql = (int)rint(o.nl * 1000.0), qd = (int)rint(o.nd * 1000.0);
    if (A->slow_count) atomicAdd(A->slow_count, 1u);
    return dw_pack(ql, qd);
}

// ---- agents on the lattice (warp 0) ------------------------------------------------------------------------
struct AgentSmem {
    double *st;     // [n]
    int *xy;        // [n] x | y << 16
    int *act;       // [n]
    int *ada;       // [n] agents_done_at increments of this launch
};

__device__ __forceinline__ double dw_food(uint32_t pk) { return dw_milli(pk & 0xffffu) + dw_milli(pk >> 16); }

__device__ __forceinline__ void dw_agents_phase(const FusedArgs &A, int j, int b, uint32_t *cb, const AgentSmem &S, int lane, int ld = 0) {
    const int N = A.P.N, n = A.P.n_agents;
    if (ld == 0) ld = N;                 // row pitch of cb in words (k_fused_tile4 pads rows to a multiple of 4)
    // pass 1: decisions from the state the previous step left (= the observation the policy would have seen)
    const int pol = A.sc[j].policy;
    for (int i = lane; i < n; i += 32) {
        int a;
        if (pol == DW_POLICY_REPLAY) a = A.actions[((size_t)j * A.P.B + b) * n + i];
        else if (pol == DW_POLICY_NONE) a = 0;
        else if (pol == DW_POLICY_RANDOM) a = (int)(dw_hash_rng(A.seed, A.world0 + b, i, A.step0 + j) % 9u);
        else {
            const int x = S.xy[i] & 0xffff, y = S.xy[i] >> 16;
            const int xm = x == 0 ? N - 1 : x - 1, xp = x == N - 1 ? 0 : x + 1;
            const int ym = y == 0 ? N - 1 : y - 1, yp = y == N - 1 ? 0 : y + 1;
            const double food[4] = {dw_food(cb[x * ld + ym]), dw_food(cb[xm * ld + y]), dw_food(cb[xp * ld + y]),
                                    dw_food(cb[x * ld + yp])};
            a = dw_greedy_pick(food, pol == DW_POLICY_GREEDY);
        }
        S.act[i] = a;
    }
    __syncwarp();
    // pass 2: move + graze, agents in index order (32 at a time; inside a batch lower lanes eat first)
    for (int base = 0; base < n; base += 32) {
        const int i = base + lane;
        const bool active = i < n;
        double st = 0.0;
        int x = 0, y = 0, cell = -1;
        bool wants = false;
        if (active) {
            st = S.st[i] - A.P.agent_gamma;
            x = S.xy[i] & 0xffff;
            y = S.xy[i] >> 16;
            const int a = S.act[i];
            if (st > 0.0) {
                if (a != 8) {
                    switch (a & 3) {
                        case 0: y = y == 0 ? N - 1 : y - 1; break;
                        case 1: x = x == 0 ? N - 1 : x - 1; break;
                        case 2: x = x == N - 1 ? 0 : x + 1; break;
                        default: y = y == N - 1 ? 0 : y + 1; break;
                    }
                }
                if (a > 4) { wants = true; cell = x * ld + y; }
            }
        }
        const uint32_t pk = wants ? cb[cell] : 0u;
        __syncwarp();
        bool taken = false;
        for (int q = 0; q < 31; ++q) {
            const int cq = __shfl_sync(0xffffffffu, cell, q);
            if (q < lane && cq == cell && cell >= 0) taken = true;
        }
        if (wants) {
            st = st + (taken ? (0.0 + 0.0) : dw_food(pk));
            cb[cell] = 0u;
        }
        if (active) {
            S.st[i] = dw_clip01(st);
            S.xy[i] = x | (y << 16);
        }
        __syncwarp();
    }
}

// ---- generic-N fused kernel: one CTA per world, cells strided over threads ---------------------------------
// dynamic smem: 2*N*N u32 | n doubles | 3n ints | 4 ints
__global__ void __launch_bounds__(256) k_fused_generic(const __grid_constant__ FusedArgs A) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int N = A.P.N, n = A.P.n_agents, NN = N * N;
    const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    uint32_t *buf0 = reinterpret_cast<uint32_t *>(smem_raw);
    uint32_t *buf1 = buf0 + NN;
    AgentSmem S;
    S.st = reinterpret_cast<double *>(buf1 + NN);   // 2*NN u32 = 8*NN bytes: 8-byte aligned
    S.xy = reinterpret_cast<int *>(S.st + n);
    S.act = S.xy + n;
    S.ada = S.act + n;
    int *s_max = S.ada + n;            // [2 parities][2 species]

    const uint32_t *gin = A.lat_in + (size_t)b * NN;
    for (int c = tid; c < NN; c += blockDim.x) buf0[c] = gin[c];
    for (int i = tid; i < n; i += blockDim.x) {
        S.st[i] = A.agent_state[(size_t)b * n + i];
        S.xy[i] = A.agent_xy[((size_t)b * n + i) * 2] | (A.agent_xy[((size_t)b * n + i) * 2 + 1] << 16);
        S.ada[i] = 0;
    }
    if (tid < 4) s_max[tid] = 0;
    __syncthreads();

    uint32_t *cb = buf0, *nb = buf1;
    int life = 0;
    // per-thread cell walk: c = tid + m*blockDim  ->  (x,y) advanced incrementally
    const int dx = blockDim.x / N, dy = blockDim.x % N;
    for (int j = 0; j < A.K; ++j) {
        if (warp == 0 && n > 0) dw_agents_phase(A, j, b, cb, S, lane);
        __syncthreads();
        if (j == A.K - 1) {
            uint32_t *gp = A.lat_pre + (size_t)b * NN;
            for (int c = tid; c < NN; c += blockDim.x) gp[c] = cb[c];
        }
        const StepCoef C = A.sc[j];
        uint32_t mx = 0;
        int x = tid / N, y = tid % N;
        for (int c = tid; c < NN; c += blockDim.x) {
            const int xm = x == 0 ? N - 1 : x - 1, xp = x == N - 1 ? 0 : x + 1;
            const int ym = y == 0 ? N - 1 : y - 1, yp = y == N - 1 ? 0 : y + 1;
            const uint32_t *r0 = cb + xm * N, *r1 = cb + x * N, *r2 = cb + xp * N;
            const uint32_t E = r1[ym] + r1[yp] + r0[y] + r2[y];
            const uint32_t S8 = E + r0[ym] + r0[yp] + r2[ym] + r2[yp];
            const uint32_t pc = r1[y];
            uint32_t q = pc;
            if ((pc | S8) != 0u) {          // empty neighbourhood: rho = 0 and the cell stays exactly 0
                unsigned tiemin = 0xffffffffu;
                q = dw_fast_cell(A.F, C, pc, E, S8, &tiemin);
                if (tiemin < A.F.tie_thresh) q = dw_slow_cell(&A, C.SL, cb, N, x, y);
            }
            nb[c] = q;
            mx = __vmaxu2(mx, q);
            x += dx; y += dy;
            if (y >= N) { y -= N; x += 1; }
        }
        const unsigned ml = __reduce_max_sync(0xffffffffu, mx & 0xffffu), md = __reduce_max_sync(0xffffffffu, mx >> 16);
        int *sm = s_max + 2 * (j & 1);
        if (lane == 0) { atomicMax(sm, (int)ml); atomicMax(sm + 1, (int)md); }
        __syncthreads();
        if (warp == 0) {
            // lifespan bookkeeping of step j (notebook cell 2): grid_done = max(grid[:,1:3]) <= 0.005
            const bool grid_done = max(sm[0], sm[1]) <= 5;
            if (lane == 0) {
                if (!grid_done) { life += 1; atomicAdd(A.alive + j, 1u); }
                s_max[2 * ((j + 1) & 1)] = 0;
                s_max[2 * ((j + 1) & 1) + 1] = 0;
            }
            for (int i = lane; i < n; i += 32) S.ada[i] += (S.st[i] < 0.1) ? 0 : 1;   // reward = state (clipped >= 0)
        }
        uint32_t *t = cb; cb = nb; nb = t;
    }
    // write back (warp 0's bookkeeping above is ordered before these reads by the barrier below)
    __syncthreads();
    uint32_t *gout = A.lat_out + (size_t)b * NN;
    for (int c = tid; c < NN; c += blockDim.x) gout[c] = cb[c];
    for (int i = tid; i < n; i += blockDim.x) {
        A.agent_state[(size_t)b * n + i] = S.st[i];
        A.agent_xy[((size_t)b * n + i) * 2] = S.xy[i] & 0xffff;
        A.agent_xy[((size_t)b * n + i) * 2 + 1] = S.xy[i] >> 16;
        if (A.count_life) A.agents_done_at[(size_t)b * n + i] += S.ada[i];
        const double r = S.st[i];
        A.reward[(size_t)b * n + i] = r;
        A.done[(size_t)b * n + i] = r < 0.1;
    }
    if (tid == 0) {
        if (A.count_life) A.done_at[b] += life;
        if (n == 0) {
            const int *sm = s_max + 2 * ((A.K - 1) & 1);
            for (int c = 0; c < 2; ++c) { A.reward[2 * b + c] = sm[c] > 0 ? 1.0 : 0.0; A.done[2 * b + c] = sm[c] > 0 ? 0 : 1; }
        }
    }
}

// ---- 64x64 specialisation: 256 threads, one 4x4 tile per thread -------------------------------------------------
// Thread (tx = tid&15, ty = tid>>4) owns rows 4ty..4ty+3, columns 4tx..4tx+3.  A step loads the 6 rows ty*4-1..ty*4+4
// of its 4 columns with LDS.128 (conflict-free: a half-warp reads one contiguous 256 B row), takes the two halo
// columns from the neighbouring lanes with SHFL (tile columns wrap inside the half-warp), forms the packed 3x3
// sums with ~4.5 integer adds per cell, runs dw_fast_cell on 16 cells and writes 4 STS.128.  Cells that hit the
// tie filter are patched afterwards by the literal path, outside the unrolled code.
// Re-evaluate one 4x4 tile of a 64x64 world cell by cell (generic indexing): cells whose fast result is within the tie
// filter are recomputed in the oracle's order and patched into nb.  Returns the packed per-species max of the tile.
// Rare path, warp-cooperative: for every lane whose 4x4 tile hit the tie filter, lanes 0..15 re-evaluate one cell of that
// tile each (generic indexing); cells within the filter are recomputed in the oracle's order and patched into nb.
// Returns the lane's packed per-species max with the flagged tiles' stale fast values replaced by the corrected ones
// (only the warp-wide max of the return values is meaningful).
__device__ __noinline__ uint32_t dw_fix_warp64(const FusedArgs *A, const StepCoef *C, const uint32_t *cb, uint32_t *nb, unsigned flagged,
                                               uint32_t mx, int r0, int c0, int lane) {
    uint32_t extra = 0;
    bool mine = false;
    __syncwarp();
    while (flagged) {
        const int L = __ffs(flagged) - 1;
        flagged &= flagged - 1;
        const int tr0 = __shfl_sync(0xffffffffu, r0, L), tc0 = __shfl_sync(0xffffffffu, c0, L);
        if (lane == L) mine = true;
        if (lane < 16) {
            const int x = tr0 + (lane >> 2), y = tc0 + (lane & 3);
            const int xm = (x + 63) & 63, xp = (x + 1) & 63, ym = (y + 63) & 63, yp = (y + 1) & 63;
            const uint32_t *q0 = cb + xm * 64, *q1 = cb + x * 64, *q2 = cb + xp * 64;
            const uint32_t E = q1[ym] + q1[yp] + q0[y] + q2[y];
            const uint32_t S8 = E + q0[ym] + q0[yp] + q2[ym] + q2[yp];
            unsigned tiemin = 0xffffffffu;
            uint32_t v = dw_fast_cell(A->F, *C, q1[y], E, S8, &tiemin);
            if (tiemin < A->F.tie_thresh) {
                v = dw_slow_cell(A, C->SL, cb, 64, x, y);
                nb[x * 64 + y] = v;
            }
            extra = __vmaxu2(extra, v);
        }
    }
    __syncwarp();                                        // patches made by helper lanes are visible to the tile's owner
    return __vmaxu2(mine ? 0u : mx, extra);
}

struct Row6 { uint32_t p[4]; uint32_t hp[4]; };     // 4 packed cells of one row + their horizontal neighbour sums

__device__ __forceinline__ Row6 dw_make_row(const uint4 v, uint32_t left, uint32_t right) {
    Row6 r;
    r.p[0] = v.x; r.p[1] = v.y; r.p[2] = v.z; r.p[3] = v.w;
    r.hp[0] = left + v.y;
    r.hp[1] = v.x + v.z;
    r.hp[2] = v.y + v.w;
    r.hp[3] = v.z + right;
    return r;
}

// Row source of a whole 64x64 world in shared memory: rows wrap mod 64, halo columns come from the neighbouring lanes
// of the half-warp (tile columns wrap inside the half-warp).
struct RowsWorld64 {
    const uint32_t *cb;
    int r0, tx, lane;
    __device__ __forceinline__ Row6 load(int k) const {          // k = -1..4 relative to the thread's first row
        const uint4 v = *reinterpret_cast<const uint4 *>(cb + ((r0 + k) & 63) * 64 + tx * 4);
        const int base = lane & 16;
        const uint32_t left = __shfl_sync(0xffffffffu, v.w, base | ((lane - 1) & 15));
        const uint32_t right = __shfl_sync(0xffffffffu, v.x, base | ((lane + 1) & 15));
        return dw_make_row(v, left, right);
    }
};
struct StoreWorld64 {
    static constexpr bool kMasks = false;
    uint32_t *nb;
    int r0, tx;
    __device__ __forceinline__ void operator()(int i, uint32_t (&q)[4]) const {
        *reinterpret_cast<uint4 *>(nb + (r0 + i) * 64 + tx * 4) = make_uint4(q[0], q[1], q[2], q[3]);
    }
};

// One step of one 4x4 tile (fast path): rows come from `rows`, results go to `store`. Returns the packed per-species
// max of the 16 new cells; *tiemin drops below F.tie_thresh if some cell needs the literal recomputation.
template <class Rows, class Store, bool DIAG = false>
__device__ __forceinline__ uint32_t dw_tile_core(const FastCoef &F, const StepCoef &C, const Rows &rows, const Store &store,
                                                 unsigned *tiemin, double *tsum = nullptr) {
    uint32_t mx = 0;
    Row6 top = rows.load(-1);
    Row6 mid = rows.load(0);
#pragma unroll kTileRowUnroll
    for (int i = 0; i < 4; ++i) {
        const Row6 bot = rows.load(i + 1);
        uint32_t E[4], S8[4];
#pragma unroll
        for (int c = 0; c < 4; ++c) {
            E[c] = mid.hp[c] + top.p[c] + bot.p[c];
            S8[c] = E[c] + top.hp[c] + bot.hp[c];
        }
        uint32_t q[4];
        {                                  // two cells in lockstep, twice (one or four at a time measured slower, DESIGN.md section 4)
            const uint32_t pa[2] = {mid.p[0], mid.p[1]}, ea[2] = {E[0], E[1]}, sa[2] = {S8[0], S8[1]};
            const uint32_t pb[2] = {mid.p[2], mid.p[3]}, eb[2] = {E[2], E[3]}, sb[2] = {S8[2], S8[3]};
            uint32_t qa[2], qb[2];
            if constexpr (DIAG && Store::kMasks) {       // series mode of a partial tile: only the store's cells count in tsum
                const int v = store.cells(i);
                dw_fast_cells<2, DIAG>(F, C, pa, ea, sa, tiemin, qa, tsum, v);
                dw_fast_cells<2, DIAG>(F, C, pb, eb, sb, tiemin, qb, tsum, v - 2);
            } else {
                dw_fast_cells<2, DIAG>(F, C, pa, ea, sa, tiemin, qa, tsum);
                dw_fast_cells<2, DIAG>(F, C, pb, eb, sb, tiemin, qb, tsum);
            }
            q[0] = qa[0]; q[1] = qa[1]; q[2] = qb[0]; q[3] = qb[1];
        }
        if (Store::kMasks) {               // k_fused_tile4, padded sides: the store zeroes entries that lie outside the world
            store(i, q);
#pragma unroll
            for (int c = 0; c < 4; ++c) mx = __vmaxu2(mx, q[c]);
        } else {
#pragma unroll
            for (int c = 0; c < 4; ++c) mx = __vmaxu2(mx, q[c]);
            store(i, q);
        }
        top = mid;
        mid = bot;
    }
    return mx;
}

// One step of one 4x4 tile of a 64x64 world: cb -> nb. Returns the packed per-species max of the tile's new cells.
template <bool DIAG = false>
__device__ __forceinline__ uint32_t dw_tile_step64(const FusedArgs &A, int j, const uint32_t *cb, uint32_t *nb, int r0, int tx, int lane,
                                                   double *tsum = nullptr) {
    const StepCoef C = A.sc[j];
    unsigned tiemin = 0xffffffffu;
    uint32_t mx = dw_tile_core<RowsWorld64, StoreWorld64, DIAG>(A.F, C, RowsWorld64{cb, r0, tx, lane}, StoreWorld64{nb, r0, tx}, &tiemin, tsum);
    // rare (~2e-4 of tile-steps): some cell of this tile sits on a rounding tie -> the warp redoes that tile's ties literally
    const unsigned flagged = __ballot_sync(0xffffffffu, tiemin < A.F.tie_thresh);
    if (flagged) mx = dw_fix_warp64(&A, &A.sc[j], cb, nb, flagged, mx, r0, tx * 4, lane);
    return mx;
}

__global__ void __launch_bounds__(256, kN64MinBlocks) k_fused_n64(const __grid_constant__ FusedArgs A) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    constexpr int N = 64, NN = N * N;
    const int n = A.P.n_agents;
    const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int tx = tid & 15, ty = tid >> 4;
    uint32_t *buf0 = reinterpret_cast<uint32_t *>(smem_raw);
    uint32_t *buf1 = buf0 + NN;
    AgentSmem S;
    S.st = reinterpret_cast<double *>(buf1 + NN);
    S.xy = reinterpret_cast<int *>(S.st + n);
    S.act = S.xy + n;
    S.ada = S.act + n;
    int *s_max = S.ada + n;

    {
        const uint4 *gin = reinterpret_cast<const uint4 *>(A.lat_in + (size_t)b * NN);
        uint4 *d = reinterpret_cast<uint4 *>(buf0);
#pragma unroll
        for (int c = 0; c < NN / 4 / 256; ++c) d[tid + c * 256] = gin[tid + c * 256];
    }
    for (int i = tid; i < n; i += 256) {
        S.st[i] = A.agent_state[(size_t)b * n + i];
        S.xy[i] = A.agent_xy[((size_t)b * n + i) * 2] | (A.agent_xy[((size_t)b * n + i) * 2 + 1] << 16);
        S.ada[i] = 0;
    }
    if (tid < 4) s_max[tid] = 0;
    __syncthreads();

    uint32_t *cb = buf0, *nb = buf1;
    int life = 0;
    const int r0 = ty * 4;
    for (int j = 0; j < A.K; ++j) {
        if (warp == 0 && n > 0) dw_agents_phase(A, j, b, cb, S, lane);
        __syncthreads();
        if (j == A.K - 1) {
            uint4 *gp = reinterpret_cast<uint4 *>(A.lat_pre + (size_t)b * NN);
            const uint4 *sc4 = reinterpret_cast<const uint4 *>(cb);
#pragma unroll
            for (int c = 0; c < NN / 4 / 256; ++c) gp[tid + c * 256] = sc4[tid + c * 256];
        }
        const uint32_t mx = dw_tile_step64(A, j, cb, nb, r0, tx, lane);
        const unsigned ml = __reduce_max_sync(0xffffffffu, mx & 0xffffu), md = __reduce_max_sync(0xffffffffu, mx >> 16);
        int *sm = s_max + 2 * (j & 1);
        if (lane == 0) { atomicMax(sm, (int)ml); atomicMax(sm + 1, (int)md); }
        __syncthreads();
        if (warp == 0) {
            const bool grid_done = max(sm[0], sm[1]) <= 5;
            if (lane == 0) {
                if (!grid_done) { life += 1; atomicAdd(A.alive + j, 1u); }
                s_max[2 * ((j + 1) & 1)] = 0;
                s_max[2 * ((j + 1) & 1) + 1] = 0;
            }
            for (int i = lane; i < n; i += 32) S.ada[i] += (S.st[i] < 0.1) ? 0 : 1;
        }
        uint32_t *t = cb; cb = nb; nb = t;
    }
    __syncthreads();
    {
        uint4 *gout = reinterpret_cast<uint4 *>(A.lat_out + (size_t)b * NN);
        const uint4 *sc4 = reinterpret_cast<const uint4 *>(cb);
#pragma unroll
        for (int c = 0; c < NN / 4 / 256; ++c) gout[tid + c * 256] = sc4[tid + c * 256];
    }
    for (int i = tid; i < n; i += 256) {
        A.agent_state[(size_t)b * n + i] = S.st[i];
        A.agent_xy[((size_t)b * n + i) * 2] = S.xy[i] & 0xffff;
        A.agent_xy[((size_t)b * n + i) * 2 + 1] = S.xy[i] >> 16;
        if (A.count_life) A.agents_done_at[(size_t)b * n + i] += S.ada[i];
        const double r = S.st[i];
        A.reward[(size_t)b * n + i] = r;
        A.done[(size_t)b * n + i] = r < 0.1;
    }
    if (tid == 0) {
        if (A.count_life) A.done_at[b] += life;
        if (n == 0) {
            const int *sm = s_max + 2 * ((A.K - 1) & 1);
            for (int c = 0; c < 2; ++c) { A.reward[2 * b + c] = sm[c] > 0 ? 1.0 : 0.0; A.done[2 * b + c] = sm[c] > 0 ? 0 : 1; }
        }
    }
}

// ---- 64x64, persistent: one world per CTA-item, dynamic work queue ----------------------------------------------------
// Work item = (world, chunk of Kc steps), handed out chunk-major from a global counter: all worlds of the ensemble
// advance together and every SM keeps kN64MinBlocks CTAs busy until the end of the launch, which removes the
// wave quantisation of a one-CTA-per-world grid (1000 worlds on 148 SMs x 4 CTAs = 1.69 waves).
// Shared memory is STATIC (compile-time addresses: no pointer registers, immediate LDS/STS offsets) and the agent
// phase is the single-pass warp version below, so this kernel takes worlds with at most DW_N64_MAX_AGENTS agents;
// larger agent counts run k_fused_n64.
#define DW_N64_MAX_AGENTS 32
struct __align__(16) N64Smem {
    uint32_t buf[2][4096];
    double st[DW_N64_MAX_AGENTS];
    int xy[DW_N64_MAX_AGENTS];      // x | y << 16
    int ada[DW_N64_MAX_AGENTS];     // agents_done_at increments of this work item
    int smax[4];                    // [2 parities][2 species]
    int item;
    unsigned long long am[DW_N64_MAX_AGENTS];   // alive_mask bits of this work item
};

// Agent phase of one step for n <= 32 agents, one lane per agent, single pass (the reference's sequential loop,
// daisy_world_rl.py:186-216, resolved in parallel): every lane decides from the pre-move state, moves, and the grazers of
// one cell are ordered by MATCH.ANY -- the lowest lane eats, later ones find the cell empty and gain 0.0 (App. B.8).
// Also does the per-step agent bookkeeping (agents_done_at += !done, done = reward < 0.1) since the state is final here.
__device__ __forceinline__ void dw_agents_phase32(const FusedArgs &A, int j, int b, uint32_t *cb, N64Smem &sm, int lane, int n,
                                                  const int *mlp_act = nullptr) {
    constexpr int N = 64;
    const bool active = lane < n;
    double st = 0.0;
    int x = 0, y = 0, a = 0;
    if (active) {
        st = sm.st[lane];
        x = sm.xy[lane] & 0xffff;
        y = sm.xy[lane] >> 16;
        const int pol = A.sc[j].policy;
        if (pol == DW_POLICY_REPLAY) a = A.actions[((size_t)j * A.P.B + b) * n + lane];
        else if (pol == DW_POLICY_RANDOM) a = (int)(dw_hash_rng(A.seed, A.world0 + b, lane, A.step0 + j) % 9u);
        else if (pol == DW_POLICY_MLP) a = mlp_act[lane];        // decided by dw_mlp_decide64 before this phase
        else if (pol != DW_POLICY_NONE) {
            const int xm = (x + N - 1) & (N - 1), xp = (x + 1) & (N - 1), ym = (y + N - 1) & (N - 1), yp = (y + 1) & (N - 1);
            const uint32_t c0 = cb[x * N + ym], c1 = cb[xm * N + y], c2 = cb[xp * N + y], c3 = cb[x * N + yp];
            const double food[4] = {dw_food(c0), dw_food(c1), dw_food(c2), dw_food(c3)};
            a = dw_greedy_pick(food, pol == DW_POLICY_GREEDY);
        }
    }
    st = st - A.P.agent_gamma;
    int cell = -1 - lane;                    // non-grazers: a private key, so MATCH groups them alone
    if (active && st > 0.0) {
        if (a != 8) {
            const int d = (a & 2) ? 1 : -1;                  // a & 3 = 0: y-1, 1: x-1, 2: x+1, 3: y+1
            if (((a + 1) & 2) == 0) y = (y + d) & (N - 1);   // a & 3 in {0, 3}
            else x = (x + d) & (N - 1);
        }
        if (a > 4) cell = x * N + y;
    }
    const bool wants = cell >= 0;
    const uint32_t pk = wants ? cb[cell] : 0u;
    const unsigned peers = __match_any_sync(0xffffffffu, cell);
    __syncwarp();                            // every read of the pre-graze state is done before any cell is zeroed
    if (wants) {
        const bool taken = (peers & ((1u << lane) - 1u)) != 0u;
        st = st + (taken ? (0.0 + 0.0) : dw_food(pk));
        cb[cell] = 0u;
    }
    if (active) {
        st = dw_clip01(st);
        sm.st[lane] = st;
        sm.xy[lane] = x | (y << 16);
        sm.ada[lane] += (st < 0.1) ? 0 : 1;
        if (A.alive_mask && !(st < 0.1)) sm.am[lane] |= 1ull << (j & 63);
        if (A.rew_series) A.rew_series[((size_t)j * A.P.B + b) * n + lane] = st;
    }
}

// ---- DW_POLICY_MLP inside the fused kernel (row N1: MLP.get_action, daisy/agents/mlp.py:97-116) ------------------------------
// What the policy sees at step j is the observation the previous step returned: the 3x3x7 window of the grid that step's
// forward wrote (daisy_world_rl.py:246-263). Fused steps never write that grid, but the buffer the NEXT stencil will overwrite
// still holds the post-graze state the previous step started from, so the nine window cells are re-evaluated from it exactly
// as forward stored them (screened cell, literal next to ties; b' from the unrounded covers, rounded temperatures, agent
// stamp: last agent on a cell wins) -- the same arithmetic as k_obs_mlp, which stays the path of every other kernel family.
// One warp per agent: lanes 0..8 the window cells, then lanes = output neurons (16, 32, 9). Every output neuron is ONE
// accumulator summed in k order with separate multiply and add, so the values are those of k_mlp_act / k_obs_mlp bit for bit.
#define DW_MLP_W1 (63 * 16)
#define DW_MLP_W2 (16 * 32)
#define DW_MLP_NPARAMS (63 * 16 + 16 * 32 + 32 * 9)

// Measured against a packed routine (four agents of one world per warp, ~1700 warp-instructions per four agents against ~1200
// per agent) inside k_fused_n64_persist at 1000 worlds x 4 agents: 8.7 ms vs 10.6 ms per 383 steps --
// with 4 CTAs per SM the policy phase is bound by the latency of its dependent chain, not by its instruction count, so four
// agents on four warps beat four agents on one.
__device__ __noinline__ void dw_mlp_decide64(const FusedArgs *Ap, double SL, const uint32_t *pb, const N64Smem *smp, double *scr, int *act, int n,
                                             int agent, int b, int lane) {
    const FusedArgs &A = *Ap;
    const N64Smem &sm = *smp;
    const DevParams &P = A.P;
    double *x = scr, *h2 = scr + 64, *h1 = scr + 96, *ov = scr + 112;       // per-warp scratch: x[64] | h2[32] | h1[16] | o[16]
    if (lane < 9) {
        const double m = P.mask[lane];
        const int cx = ((sm.xy[agent] & 0xffff) + lane / 3 + 63) & 63, cy = ((sm.xy[agent] >> 16) + lane % 3 + 63) & 63;
        double l9[9], d9[9];
#pragma unroll
        for (int a = 0; a < 3; ++a)
#pragma unroll
            for (int c = 0; c < 3; ++c) {
                const uint32_t k = pb[((cx + a + 63) & 63) * 64 + ((cy + c + 63) & 63)];
                l9[a * 3 + c] = dw_milli(k & 0xffffu);
                d9[a * 3 + c] = dw_milli(k >> 16);
            }
        ScrCell c;
        if (!(P.screen && dw_screened_cell(P, SL / P.sigma, l9, d9, c))) dw_literal_rounded(P, SL, l9, d9, c);
        double ch4 = dw_k2v(c.k[4]);
        for (int k = 0; k < n; ++k)
            if ((sm.xy[k] & 0xffff) == cx && (sm.xy[k] >> 16) == cy) ch4 = sm.st[k];
        x[lane] = dw_k2v(c.k[0]) * m;
        x[9 + lane] = dw_k2v(c.k[1]) * m;
        x[18 + lane] = dw_k2v(c.k[2]) * m;
        x[27 + lane] = dw_k2v(c.k[3]) * m;
        x[36 + lane] = ch4 * m;
        x[45 + lane] = dw_k2v(c.k[5]) * m;
        x[54 + lane] = 0.0 * m;
    }
    __syncwarp();
    const double *w = A.mlp_w;
    if (A.mlp_wpm > 0) w += (size_t)(agent < A.mlp_half ? b / A.mlp_wpm : A.mlp_adv) * DW_MLP_NPARAMS;
    const double *w1 = w, *w2 = w + DW_MLP_W1, *w3 = w2 + DW_MLP_W2;
    if (lane < 16) {
        // products first (independent loads and multiplications, 21 at a time), then the sum in k order: the dependent chain is
        // 63 additions instead of 63 x (load + multiply + add)
        double h = 0.0;
#pragma unroll 1
        for (int k0 = 0; k0 < 63; k0 += 21) {
            double pr[21];
#pragma unroll
            for (int k = 0; k < 21; ++k) pr[k] = x[k0 + k] * __ldg(w1 + (k0 + k) * 16 + lane);
#pragma unroll
            for (int k = 0; k < 21; ++k) h = h + pr[k];
        }
        h1[lane] = h * (h > 0.0 ? 1.0 : 0.0);
    }
    __syncwarp();
    {
        double h = 0.0;
#pragma unroll
        for (int k = 0; k < 16; ++k) h = h + h1[k] * __ldg(w2 + k * 32 + lane);
        h2[lane] = h * (h > 0.0 ? 1.0 : 0.0);
    }
    __syncwarp();
    if (lane < 9) {
        double o = 0.0;
#pragma unroll
        for (int k = 0; k < 32; ++k) o = o + h2[k] * __ldg(w3 + k * 9 + lane);
        ov[lane] = o;
    }
    __syncwarp();
    if (lane == 0) {
        int best = 0;
        double bv = ov[0];
#pragma unroll
        for (int o = 1; o < 9; ++o) if (ov[o] > bv) { bv = ov[o]; best = o; }
        act[agent] = best;
    }
    __syncwarp();
}


struct MlpSmem {
    double scratch[8][128];
    int act[DW_N64_MAX_AGENTS];
};

template <bool DIAG, bool MLP = false>
__global__ void __launch_bounds__(256, kN64MinBlocks) k_fused_n64_persist(const __grid_constant__ FusedArgs A) {
    __shared__ N64Smem sm;
    __shared__ double s_tsum;
    __shared__ unsigned int s_cov[2];
    __shared__ typename std::conditional<MLP, MlpSmem, int>::type s_mlp;
    constexpr int NN = 4096;
    const int n = A.P.n_agents;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int tx = tid & 15, r0 = (tid >> 4) * 4;
    const int n_items = A.n_pairs * A.n_chunks;      // n_pairs = number of worlds for this kernel

    for (int it = 0;; ++it) {
        int t;
        if (A.queue) {                       // dynamic work queue (multi-chunk launches)
            if (tid == 0) sm.item = (int)atomicAdd(A.queue, 1u);
            __syncthreads();
            t = sm.item;
        } else {                             // single-chunk launch (step()): static round-robin, nothing to zero beforehand
            t = blockIdx.x + it * gridDim.x;
            __syncthreads();                 // shared memory of the previous item is free
        }
        if (t >= n_items) break;
        const int c = t / A.n_pairs, b = t - c * A.n_pairs;
        if (A.queue) {
            if (tid == 0) {
                while (atomicAdd(A.pair_done + b, 0u) < (unsigned)c) __nanosleep(200);
                __threadfence();
            }
            __syncthreads();
        }
        const int j0 = c * A.Kc, kc = min(A.Kc, A.K - j0);
        {
            const uint4 *gin = reinterpret_cast<const uint4 *>(A.lat + (size_t)b * NN);
#pragma unroll
            for (int k = 0; k < 4; ++k) reinterpret_cast<uint4 *>(sm.buf[0])[tid + k * 256] = __ldcg(gin + tid + k * 256);
        }
        if (MLP) {       // the post-graze state the step before this item started from: observation windows of the item's first step
            const uint4 *gp = reinterpret_cast<const uint4 *>(A.lat_pre + (size_t)b * NN);
#pragma unroll
            for (int k = 0; k < 4; ++k) reinterpret_cast<uint4 *>(sm.buf[1])[tid + k * 256] = __ldcg(gp + tid + k * 256);
        }
        if (tid < n) {
            const size_t g = (size_t)b * n + tid;
            sm.st[tid] = __ldcg(A.agent_state + g);
            sm.xy[tid] = __ldcg(A.agent_xy + 2 * g) | (__ldcg(A.agent_xy + 2 * g + 1) << 16);
            sm.ada[tid] = 0;
            sm.am[tid] = 0ull;
        }
        if (tid < 4) sm.smax[tid] = 0;
        if (DIAG && tid == 0) { s_tsum = 0.0; s_cov[0] = 0u; s_cov[1] = 0u; }
        __syncthreads();

        int life = 0;
#pragma unroll 1
        for (int jl = 0; jl < kc; ++jl) {
            const int j = j0 + jl;
            uint32_t *cb = sm.buf[jl & 1], *nb = sm.buf[(jl + 1) & 1];
            const int *mlp_act = nullptr;
            if constexpr (MLP) {
                if (n > 0 && A.sc[j].policy == DW_POLICY_MLP) {
                    const double SLp = j == 0 ? A.SL_prev : A.sc[j - 1].SL;
                    for (int i = warp; i < n; i += 8) dw_mlp_decide64(&A, SLp, nb, &sm, s_mlp.scratch[warp], s_mlp.act, n, i, b, lane);
                }
                mlp_act = s_mlp.act;
                __syncthreads();
            }
            if (warp == 0 && n > 0) dw_agents_phase32(A, j, b, cb, sm, lane, n, mlp_act);
            __syncthreads();
            if (!MLP && j == A.K - 1) {
                uint4 *gp = reinterpret_cast<uint4 *>(A.lat_pre + (size_t)b * NN);
#pragma unroll
                for (int k = 0; k < 4; ++k) gp[tid + k * 256] = reinterpret_cast<const uint4 *>(cb)[tid + k * 256];
            }
            double tsum = 0.0;
            const uint32_t mx = dw_tile_step64<DIAG>(A, j, cb, nb, r0, tx, lane, &tsum);
            const unsigned ml = __reduce_max_sync(0xffffffffu, mx & 0xffffu), md = __reduce_max_sync(0xffffffffu, mx >> 16);
            int *smx = sm.smax + 2 * (jl & 1);
            if (lane == 0) { atomicMax(smx, (int)ml); atomicMax(smx + 1, (int)md); }
            if (DIAG) {
                // series mode: warp-shuffle reductions of the temperature sum and of the new covers of this thread's tile
                unsigned int cl = 0, cd = 0;
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    const uint4 v = *reinterpret_cast<const uint4 *>(nb + (r0 + i) * 64 + tx * 4);   // own stores (fix-ups: see below)
                    cl += (v.x & 0xffffu) + (v.y & 0xffffu) + (v.z & 0xffffu) + (v.w & 0xffffu);
                    cd += (v.x >> 16) + (v.y >> 16) + (v.z >> 16) + (v.w >> 16);
                }
                for (int o = 16; o > 0; o >>= 1) tsum += __shfl_xor_sync(0xffffffffu, tsum, o);
                cl = __reduce_add_sync(0xffffffffu, cl);
                cd = __reduce_add_sync(0xffffffffu, cd);
                if (lane == 0) { atomicAdd(&s_tsum, tsum); atomicAdd(&s_cov[0], cl); atomicAdd(&s_cov[1], cd); }
            }
            __syncthreads();
            if (DIAG && tid == 0) {
                atomicAdd(A.series_T + j, s_tsum);
                atomicAdd(A.series_l + j, (unsigned long long)s_cov[0]);
                atomicAdd(A.series_d + j, (unsigned long long)s_cov[1]);
                s_tsum = 0.0; s_cov[0] = 0u; s_cov[1] = 0u;      // the next adds come after the next step's first barrier
            }
            if (tid == 0) {
                // lifespan bookkeeping of step j (notebook cell 2): grid_done = max(grid[:,1:3]) <= 0.005
                if (max(smx[0], smx[1]) > 5) { life += 1; atomicAdd(A.alive + j, 1u); }
                int *nx = sm.smax + 2 * ((jl + 1) & 1);
                nx[0] = 0; nx[1] = 0;
            }
        }
        __syncthreads();
        {
            uint4 *gout = reinterpret_cast<uint4 *>(A.lat + (size_t)b * NN);
#pragma unroll
            for (int k = 0; k < 4; ++k) gout[tid + k * 256] = reinterpret_cast<const uint4 *>(sm.buf[kc & 1])[tid + k * 256];
        }
        if (MLP) {      // post-graze state of the item's last step (still intact in the other buffer): next item's windows / lazy grid
            uint4 *gp = reinterpret_cast<uint4 *>(A.lat_pre + (size_t)b * NN);
#pragma unroll
            for (int k = 0; k < 4; ++k) gp[tid + k * 256] = reinterpret_cast<const uint4 *>(sm.buf[(kc + 1) & 1])[tid + k * 256];
        }
        if (tid < n) {
            const size_t g = (size_t)b * n + tid;
            const double r = sm.st[tid];
            A.agent_state[g] = r;
            A.agent_xy[2 * g] = sm.xy[tid] & 0xffff;
            A.agent_xy[2 * g + 1] = sm.xy[tid] >> 16;
            if (A.count_life) A.agents_done_at[g] = __ldcg(A.agents_done_at + g) + sm.ada[tid];
            if (A.alive_mask) A.alive_mask[g] = __ldcg(A.alive_mask + g) | sm.am[tid];
            A.reward[g] = r;
            A.done[g] = r < 0.1;
        }
        if (tid == 0) {
            if (A.count_life) A.done_at[b] = __ldcg(A.done_at + b) + life;
            if (n == 0) {
                const int *smx = sm.smax + 2 * ((kc - 1) & 1);
                for (int ch = 0; ch < 2; ++ch) { A.reward[2 * b + ch] = smx[ch] > 0 ? 1.0 : 0.0; A.done[2 * b + ch] = smx[ch] > 0 ? 0 : 1; }
            }
        }
        __syncthreads();
        if (A.queue && tid == 0) {
            __threadfence();
            atomicExch(A.pair_done + b, (unsigned)(c + 1));
        }
    }
}

// ---- worlds smaller than 64x64 (N = 8, 16, 32): (64/N)^2 worlds per CTA, tiled into one 64x64 "super-grid" -------------------
// The 256 threads keep the 4x4-cells-per-thread tiling and the fast path of the 64x64 kernel; the W = (64/N)^2 worlds of a
// CTA sit side by side in the two 64x64 shared-memory buffers (world (wy, wx) at rows wy*N.., columns wx*N..), rows wrap
// inside a world and the halo columns come from the neighbouring lanes of the world's own N/4-lane group. Work items
// are (group of W worlds, chunk of Kc steps), same persistent queue as the 64x64 kernel. Agents: all W*n of them live in
// shared memory (W*n <= DW_SUB64_MAX_AGENTS); each warp takes the agents of W/8 whole worlds (worlds are independent),
// decides for all of them, then moves and grazes them 32 at a time in flat (world, index) order, so the per-world
// sequential semantics are those of dw_agents_phase32.
#define DW_SUB64_MAX_AGENTS 256
template <int N>
struct Sub64Smem {
    uint32_t buf[2][4096];
    double st[DW_SUB64_MAX_AGENTS];
    int xy[DW_SUB64_MAX_AGENTS];        // x | y << 16, world-local
    int ada[DW_SUB64_MAX_AGENTS];
    signed char act[DW_SUB64_MAX_AGENTS];
    unsigned long long am[DW_SUB64_MAX_AGENTS];   // alive_mask bits of this work item
    int smax[2][(64 / N) * (64 / N)][2];
    int life[(64 / N) * (64 / N)];
    int item;
};

template <int N>
struct RowsSub64 {
    const uint32_t *cb;
    int row_base, lr0, tx, lane;         // first super-grid row of the world, first world-local row of the tile
    __device__ __forceinline__ Row6 load(int k) const {
        constexpr int TX = N / 4;
        const uint4 v = *reinterpret_cast<const uint4 *>(cb + (row_base + ((lr0 + k) & (N - 1))) * 64 + tx * 4);
        const int base = lane & ~(TX - 1);
        const uint32_t left = __shfl_sync(0xffffffffu, v.w, base | ((lane - 1) & (TX - 1)));
        const uint32_t right = __shfl_sync(0xffffffffu, v.x, base | ((lane + 1) & (TX - 1)));
        return dw_make_row(v, left, right);
    }
};

// literal recomputation of one cell of a sub-world (wrap inside the world)
template <int N>
__device__ __noinline__ uint32_t dw_slow_cell_sub(const FusedArgs *A, double SL, const uint32_t *cb, int X, int Y) {
    const int rb = X & ~(N - 1), cbse = Y & ~(N - 1);
    const int xs[3] = {rb | ((X - 1) & (N - 1)), X, rb | ((X + 1) & (N - 1))};
    const int ys[3] = {cbse | ((Y - 1) & (N - 1)), Y, cbse | ((Y + 1) & (N - 1))};
    double l9[9], d9[9];
#pragma unroll
    for (int a = 0; a < 3; ++a)
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            const uint32_t k = cb[xs[a] * 64 + ys[c]];
            l9[a * 3 + c] = dw_milli(k & 0xffffu);
            d9[a * 3 + c] = dw_milli(k >> 16);
        }
    const LitCell o = dw_literal_cell(A->P, SL, l9, d9);
    if (A->slow_count) atomicAdd(A->slow_count, 1u);
    return dw_pack((int)rint(o.nl * 1000.0), (int)rint(o.nd * 1000.0));
}

// warp-cooperative tie fix-up for sub-worlds; the corrected tile's maxima go straight to its world's slots. Returns true
// for lanes whose own (stale) tile maximum must not be used.
template <int N>
__device__ __noinline__ bool dw_fix_warp_sub(const FusedArgs *A, const StepCoef *C, const uint32_t *cb, uint32_t *nb, unsigned flagged,
                                             int r0, int c0, int lane, int (*smax)[2]) {
    bool mine = false;
    __syncwarp();
    while (flagged) {
        const int L = __ffs(flagged) - 1;
        flagged &= flagged - 1;
        const int tr0 = __shfl_sync(0xffffffffu, r0, L), tc0 = __shfl_sync(0xffffffffu, c0, L);
        if (lane == L) mine = true;
        if (lane < 16) {
            const int X = tr0 + (lane >> 2), Y = tc0 + (lane & 3);
            const int rb = X & ~(N - 1), cbse = Y & ~(N - 1);
            const int xm = rb | ((X - 1) & (N - 1)), xp = rb | ((X + 1) & (N - 1)), ym = cbse | ((Y - 1) & (N - 1)), yp = cbse | ((Y + 1) & (N - 1));
            const uint32_t *q0 = cb + xm * 64, *q1 = cb + X * 64, *q2 = cb + xp * 64;
            const uint32_t E = q1[ym] + q1[yp] + q0[Y] + q2[Y];
            const uint32_t S8 = E + q0[ym] + q0[yp] + q2[ym] + q2[yp];
            unsigned tiemin = 0xffffffffu;
            uint32_t v = dw_fast_cell(A->F, *C, q1[Y], E, S8, &tiemin);
            if (tiemin < A->F.tie_thresh) {
                v = dw_slow_cell_sub<N>(A, C->SL, cb, X, Y);
                nb[X * 64 + Y] = v;
            }
            int *sm = smax[(tr0 / N) * (64 / N) + tc0 / N];
            atomicMax(sm, (int)(v & 0xffffu));
            atomicMax(sm + 1, (int)(v >> 16));
        }
    }
    __syncwarp();
    return mine;
}

// Called by every warp that owns worlds: the agents [a_lo, a_hi) (flat (world, index) order) of whole worlds. Worlds are
// independent, so the warps of a CTA run their agent phases concurrently.
template <int N>
__device__ __forceinline__ void dw_agents_phase_sub(const FusedArgs &A, int j, int group, uint32_t *cb, Sub64Smem<N> &sm, int lane, int n,
                                                    int a_lo, int n_act) {
    constexpr int WX = 64 / N, W = WX * WX;
    const int pol = A.sc[j].policy;
    // pass 1: every agent decides from the pre-move state
    for (int a = a_lo + lane; a < n_act; a += 32) {
        const int wl = a / n, i = a - wl * n;
        const int x = sm.xy[a] & 0xffff, y = sm.xy[a] >> 16;
        const size_t gw = (size_t)group * W + wl;
        int act = 0;
        if (pol == DW_POLICY_REPLAY) act = A.actions[((size_t)j * A.P.B + gw) * n + i];
        else if (pol == DW_POLICY_RANDOM) act = (int)(dw_hash_rng(A.seed, A.world0 + (uint32_t)gw, i, A.step0 + j) % 9u);
        else if (pol != DW_POLICY_NONE) {
            const int r = (wl / WX) * N, c = (wl % WX) * N;
            const int xm = (x + N - 1) & (N - 1), xp = (x + 1) & (N - 1), ym = (y + N - 1) & (N - 1), yp = (y + 1) & (N - 1);
            const double food[4] = {dw_food(cb[(r + x) * 64 + c + ym]), dw_food(cb[(r + xm) * 64 + c + y]),
                                    dw_food(cb[(r + xp) * 64 + c + y]), dw_food(cb[(r + x) * 64 + c + yp])};
            act = dw_greedy_pick(food, pol == DW_POLICY_GREEDY);
        }
        sm.act[a] = (signed char)act;
    }
    __syncwarp();
    // pass 2: move + graze, 32 agents at a time in flat (world, index) order; inside a round MATCH.ANY orders the grazers
    // of a cell, across rounds the earlier round has already emptied it
    for (int base = a_lo; base < n_act; base += 32) {
        const int a = base + lane;
        const bool active = a < n_act;
        double st = 0.0;
        int x = 0, y = 0, cell = -1 - lane;
        if (active) {
            st = sm.st[a] - A.P.agent_gamma;
            x = sm.xy[a] & 0xffff;
            y = sm.xy[a] >> 16;
            const int act = sm.act[a];
            if (st > 0.0) {
                if (act != 8) {
                    const int d = (act & 2) ? 1 : -1;
                    if (((act + 1) & 2) == 0) y = (y + d) & (N - 1);
                    else x = (x + d) & (N - 1);
                }
                if (act > 4) {
                    const int wl = a / n;
                    cell = ((wl / WX) * N + x) * 64 + (wl % WX) * N + y;
                }
            }
        }
        const bool wants = cell >= 0;
        const uint32_t pk = wants ? cb[cell] : 0u;
        const unsigned peers = __match_any_sync(0xffffffffu, cell);
        __syncwarp();
        if (wants) {
            const bool taken = (peers & ((1u << lane) - 1u)) != 0u;
            st = st + (taken ? (0.0 + 0.0) : dw_food(pk));
            cb[cell] = 0u;
        }
        if (active) {
            st = dw_clip01(st);
            sm.st[a] = st;
            sm.xy[a] = x | (y << 16);
            sm.ada[a] += (st < 0.1) ? 0 : 1;
            if (A.alive_mask && !(st < 0.1)) sm.am[a] |= 1ull << (j & 63);
        }
        __syncwarp();
    }
}

template <int N, bool DIAG = false>
__global__ void __launch_bounds__(256, kN64MinBlocks) k_fused_sub64_persist(const __grid_constant__ FusedArgs A) {
    constexpr int WX = 64 / N, W = WX * WX, TX = N / 4;
    __shared__ Sub64Smem<N> sm;
    __shared__ double s_tsum;               // series mode (DIAG): per-step sums over the CTA's worlds, see k_fused_n64_persist
    __shared__ unsigned int s_cov[2];
    const int n = A.P.n_agents, B = A.P.B;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int tx = tid & 15, ty = tid >> 4;
    const int wl = (ty / TX) * WX + tx / TX;            // this thread's world inside the CTA
    const int row_base = (ty / TX) * N, lr0 = (ty % TX) * 4, r0 = ty * 4;
    const int n_items = A.n_pairs * A.n_chunks;        // n_pairs = number of world groups

    for (int it = 0;; ++it) {
        int t;
        if (A.queue) {
            if (tid == 0) sm.item = (int)atomicAdd(A.queue, 1u);
            __syncthreads();
            t = sm.item;
        } else {                             // single-chunk launch: static round-robin (see k_fused_n64_persist)
            t = blockIdx.x + it * gridDim.x;
            __syncthreads();
        }
        if (t >= n_items) break;
        const int c = t / A.n_pairs, g = t - c * A.n_pairs;
        if (A.queue) {
            if (tid == 0) {
                while (atomicAdd(A.pair_done + g, 0u) < (unsigned)c) __nanosleep(200);
                __threadfence();
            }
            __syncthreads();
        }
        const int j0 = c * A.Kc, kc = min(A.Kc, A.K - j0);
        const int n_worlds = min(W, B - g * W);
        const int n_act = n_worlds * n;
        // global [world][N][N] -> super-grid
        for (int q = tid; q < 1024; q += 256) {
            const int R = q >> 4, C4 = (q & 15) * 4;
            const int w = (R / N) * WX + C4 / N;
            uint4 v = make_uint4(0u, 0u, 0u, 0u);
            if (w < n_worlds) v = __ldcg(reinterpret_cast<const uint4 *>(A.lat + ((size_t)g * W + w) * (N * N) + (R % N) * N + (C4 % N)));
            reinterpret_cast<uint4 *>(sm.buf[0])[q] = v;
        }
        for (int a = tid; a < n_act; a += 256) {
            const size_t ga = (size_t)g * W * n + a;
            sm.st[a] = __ldcg(A.agent_state + ga);
            sm.xy[a] = __ldcg(A.agent_xy + 2 * ga) | (__ldcg(A.agent_xy + 2 * ga + 1) << 16);
            sm.ada[a] = 0;
            sm.am[a] = 0ull;
        }
        for (int q = tid; q < 2 * W * 2; q += 256) (&sm.smax[0][0][0])[q] = 0;
        if (tid < W) sm.life[tid] = 0;
        if (DIAG && tid == 0) { s_tsum = 0.0; s_cov[0] = 0u; s_cov[1] = 0u; }
        __syncthreads();

#pragma unroll 1
        for (int jl = 0; jl < kc; ++jl) {
            const int j = j0 + jl;
            uint32_t *cb = sm.buf[jl & 1], *nb = sm.buf[(jl + 1) & 1];
            {   // warp k moves the agents of worlds [k * WPW, (k + 1) * WPW) of the group
                constexpr int WPW = (W + 7) / 8;
                const int w_lo = warp * WPW, w_hi = min(w_lo + WPW, n_worlds);
                if (w_lo < w_hi && n > 0) dw_agents_phase_sub<N>(A, j, g, cb, sm, lane, n, w_lo * n, w_hi * n);
            }
            __syncthreads();
            if (j == A.K - 1) {                        // post-graze state of the launch's last step (lazy materialisation)
                for (int q = tid; q < 1024; q += 256) {
                    const int R = q >> 4, C4 = (q & 15) * 4;
                    const int w = (R / N) * WX + C4 / N;
                    if (w < n_worlds)
                        *reinterpret_cast<uint4 *>(A.lat_pre + ((size_t)g * W + w) * (N * N) + (R % N) * N + (C4 % N)) =
                            reinterpret_cast<const uint4 *>(cb)[q];
                }
            }
            const StepCoef C = A.sc[j];
            unsigned tiemin = 0xffffffffu;
            double tsum = 0.0;
            const uint32_t mx = dw_tile_core<RowsSub64<N>, StoreWorld64, DIAG>(A.F, C, RowsSub64<N>{cb, row_base, lr0, tx, lane},
                                                                                 StoreWorld64{nb, r0, tx}, &tiemin, &tsum);
            int (*smx)[2] = sm.smax[jl & 1];
            bool stale = false;
            const unsigned flagged = __ballot_sync(0xffffffffu, tiemin < A.F.tie_thresh);
            if (flagged) stale = dw_fix_warp_sub<N>(&A, &A.sc[j], cb, nb, flagged, r0, tx * 4, lane, smx);
            if (!stale && mx) { atomicMax(&smx[wl][0], (int)(mx & 0xffffu)); atomicMax(&smx[wl][1], (int)(mx >> 16)); }
            if (DIAG) {
                // series mode: this thread's tile (fix-ups included) and temperature sum, unless its world slot is empty
                unsigned int cl = 0, cd = 0;
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    const uint4 v = *reinterpret_cast<const uint4 *>(nb + (r0 + i) * 64 + tx * 4);
                    cl += (v.x & 0xffffu) + (v.y & 0xffffu) + (v.z & 0xffffu) + (v.w & 0xffffu);
                    cd += (v.x >> 16) + (v.y >> 16) + (v.z >> 16) + (v.w >> 16);
                }
                if (wl >= n_worlds) { tsum = 0.0; cl = 0; cd = 0; }
                for (int o = 16; o > 0; o >>= 1) tsum += __shfl_xor_sync(0xffffffffu, tsum, o);
                cl = __reduce_add_sync(0xffffffffu, cl);
                cd = __reduce_add_sync(0xffffffffu, cd);
                if (lane == 0) { atomicAdd(&s_tsum, tsum); atomicAdd(&s_cov[0], cl); atomicAdd(&s_cov[1], cd); }
            }
            __syncthreads();
            if (DIAG && tid == 32) {               // warp 1: warp 0 does the lifespan bookkeeping below
                atomicAdd(A.series_T + j, s_tsum);
                atomicAdd(A.series_l + j, (unsigned long long)s_cov[0]);
                atomicAdd(A.series_d + j, (unsigned long long)s_cov[1]);
                s_tsum = 0.0; s_cov[0] = 0u; s_cov[1] = 0u;      // the next adds come after the next step's first barrier
            }
            if (warp == 0) {
                // lifespan bookkeeping of step j for the CTA's worlds (notebook cell 2): grid_done = max(grid[:,1:3]) <= 0.005
                unsigned alive = 0;
                for (int w = lane; w < n_worlds; w += 32) {
                    const bool up = max(smx[w][0], smx[w][1]) > 5;
                    if (up) { sm.life[w] += 1; alive += 1; }
                }
                alive = __reduce_add_sync(0xffffffffu, alive);
                if (lane == 0 && alive) atomicAdd(A.alive + j, alive);
                int (*nx)[2] = sm.smax[(jl + 1) & 1];
                for (int w = lane; w < W; w += 32) { nx[w][0] = 0; nx[w][1] = 0; }
            }
        }
        __syncthreads();
        for (int q = tid; q < 1024; q += 256) {
            const int R = q >> 4, C4 = (q & 15) * 4;
            const int w = (R / N) * WX + C4 / N;
            if (w < n_worlds) {
                *reinterpret_cast<uint4 *>(A.lat + ((size_t)g * W + w) * (N * N) + (R % N) * N + (C4 % N)) =
                    reinterpret_cast<const uint4 *>(sm.buf[kc & 1])[q];
            }
        }
        for (int a = tid; a < n_act; a += 256) {
            const size_t ga = (size_t)g * W * n + a;
            const double r = sm.st[a];
            A.agent_state[ga] = r;
            A.agent_xy[2 * ga] = sm.xy[a] & 0xffff;
            A.agent_xy[2 * ga + 1] = sm.xy[a] >> 16;
            if (A.count_life) A.agents_done_at[ga] = __ldcg(A.agents_done_at + ga) + sm.ada[a];
            if (A.alive_mask) A.alive_mask[ga] = __ldcg(A.alive_mask + ga) | sm.am[a];
            A.reward[ga] = r;
            A.done[ga] = r < 0.1;
        }
        if (tid < n_worlds) {
            const size_t gw = (size_t)g * W + tid;
            if (A.count_life) A.done_at[gw] = __ldcg(A.done_at + gw) + sm.life[tid];
            if (n == 0) {
                const int *smx = sm.smax[(kc - 1) & 1][tid];
                for (int ch = 0; ch < 2; ++ch) { A.reward[2 * gw + ch] = smx[ch] > 0 ? 1.0 : 0.0; A.done[2 * gw + ch] = smx[ch] > 0 ? 0 : 1; }
            }
        }
        __syncthreads();
        if (A.queue && tid == 0) {
            __threadfence();
            atomicExch(A.pair_done + g, (unsigned)(c + 1));
        }
    }
}

// ---- any N that is a multiple of 4 (and fits in shared memory): one CTA per world, 4x4 tiles dealt round-robin to the threads ----
// Same fast path and tile core as the 64x64 kernel; the halo columns come from shared memory instead of SHFL (the lanes
// of a warp do not line up with a world row), the rows wrap by compare. The host picks the block size from the tile count
// and the shared-memory footprint (launch_fused). Round 2: persistent CTAs with the (world, 16-step chunk) work queue of the
// 64x64 kernel (a grid of one CTA per world ran 2.25 waves at 1000 worlds of 96x96: 25 % of the last wave idle). World sides
// that are not a multiple of 4 (round 2): shared-memory rows are
// padded to ld = 4 * ceil(N / 4) words, the last tile of a row takes its missing columns (and its right halo) from the
// wrapped columns 0, 1, .., its cells outside the world are neither stored nor counted in the maxima, and the tile rows
// below the world are computed from wrapped rows and dropped. dynamic smem: 2*N*ld u32 | n doubles | 3n ints | 4 ints.
template <bool PAD>
struct RowsTile4 {
    const uint32_t *cb;
    int N, ld, r0, c0, cl, cr, valid;   // row pitch, first row / column of the tile, wrapped halo columns, columns inside the world
    __device__ __forceinline__ Row6 load(int k) const {
        int r = r0 + k;
        r = r < 0 ? r + N : (r >= N ? r - N : r);
        const uint32_t *row = cb + r * (PAD ? ld : N);
        uint4 v = *reinterpret_cast<const uint4 *>(row + c0);
        if (PAD && valid < 4) {         // last tile of a row whose side is not a multiple of 4: the missing columns wrap to 0, 1, 2
            if (valid < 2) v.y = row[1 - valid];
            if (valid < 3) v.z = row[2 - valid];
            v.w = row[3 - valid];
        }
        return dw_make_row(v, row[cl], row[cr]);
    }
};
template <bool PAD>
struct StoreTile4 {
    static constexpr bool kMasks = PAD;
    uint32_t *nb;
    int N, ld, r0, c0, valid;
    __device__ __forceinline__ void operator()(int i, uint32_t (&q)[4]) const {
        if (!PAD) {
            *reinterpret_cast<uint4 *>(nb + (r0 + i) * N + c0) = make_uint4(q[0], q[1], q[2], q[3]);
            return;
        }
        if (r0 + i >= N) { q[0] = 0u; q[1] = 0u; q[2] = 0u; q[3] = 0u; return; }       // tile row below the world: nothing to keep
        uint32_t *d = nb + (r0 + i) * ld + c0;
        if (valid == 4) { *reinterpret_cast<uint4 *>(d) = make_uint4(q[0], q[1], q[2], q[3]); return; }
#pragma unroll
        for (int t = 0; t < 4; ++t) {
            if (t < valid) d[t] = q[t];
            else q[t] = 0u;
        }
    }
};

// warp-cooperative tie fix-up, generic N (see dw_fix_warp64)
__device__ __noinline__ uint32_t dw_fix_warp_tile4(const FusedArgs *A, const StepCoef *C, const uint32_t *cb, uint32_t *nb, unsigned flagged,
                                                   uint32_t mx, int r0, int c0, int lane, int N, int ld) {
    uint32_t extra = 0;
    bool mine = false;
    __syncwarp();
    while (flagged) {
        const int L = __ffs(flagged) - 1;
        flagged &= flagged - 1;
        const int tr0 = __shfl_sync(0xffffffffu, r0, L), tc0 = __shfl_sync(0xffffffffu, c0, L);
        if (lane == L) mine = true;
        const int x = tr0 + (lane >> 2), y = tc0 + (lane & 3);
        if (lane < 16 && x < N && y < N) {               // cells of an edge tile outside the world are skipped
            const int xm = x == 0 ? N - 1 : x - 1, xp = x == N - 1 ? 0 : x + 1, ym = y == 0 ? N - 1 : y - 1, yp = y == N - 1 ? 0 : y + 1;
            const uint32_t *q0 = cb + xm * ld, *q1 = cb + x * ld, *q2 = cb + xp * ld;
            const uint32_t E = q1[ym] + q1[yp] + q0[y] + q2[y];
            const uint32_t S8 = E + q0[ym] + q0[yp] + q2[ym] + q2[yp];
            unsigned tiemin = 0xffffffffu;
            uint32_t v = dw_fast_cell(A->F, *C, q1[y], E, S8, &tiemin);
            if (tiemin < A->F.tie_thresh) {
                v = dw_slow_cell(A, C->SL, cb, N, x, y, ld);
                nb[x * ld + y] = v;
            }
            extra = __vmaxu2(extra, v);
        }
    }
    __syncwarp();
    return __vmaxu2(mine ? 0u : mx, extra);
}

template <bool PAD, bool DIAG = false>
__global__ void __launch_bounds__(1024, 1) k_fused_tile4(const __grid_constant__ FusedArgs A) {
    static_assert(!(PAD && DIAG), "series mode: sides that are multiples of 4 (the temperature sum would include padded cells)");
    extern __shared__ __align__(16) unsigned char smem_raw[];
    __shared__ int s_item;
    __shared__ double s_tsum;               // series mode (DIAG), see k_fused_n64_persist
    __shared__ unsigned int s_cov[2];
    const int N = A.P.N, n = A.P.n_agents, NN = N * N, T = (N + 3) >> 2, TT = T * T;
    const int ld = PAD ? T * 4 : N, SN = N * ld;   // PAD: shared-memory rows padded to a multiple of 4 words (16-byte tile loads)
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nthr = blockDim.x;
    uint32_t *buf0 = reinterpret_cast<uint32_t *>(smem_raw);
    uint32_t *buf1 = buf0 + SN;
    AgentSmem S;
    S.st = reinterpret_cast<double *>(buf1 + SN);
    S.xy = reinterpret_cast<int *>(S.st + n);
    S.act = S.xy + n;
    S.ada = S.act + n;
    int *s_max = S.ada + n;
    const int rounds = (TT + nthr - 1) / nthr;
    const int n_items = A.n_pairs * A.n_chunks;      // persistent CTAs, work item = (world, chunk of Kc steps), see k_fused_n64_persist

    for (int it = 0;; ++it) {
        int t;
        if (A.queue) {
            if (tid == 0) s_item = (int)atomicAdd(A.queue, 1u);
            __syncthreads();
            t = s_item;
        } else {
            t = blockIdx.x + it * gridDim.x;
            __syncthreads();
        }
        if (t >= n_items) break;
        const int c = t / A.n_pairs, b = t - c * A.n_pairs;
        if (A.queue) {
            if (tid == 0) {
                while (atomicAdd(A.pair_done + b, 0u) < (unsigned)c) __nanosleep(200);
                __threadfence();
            }
            __syncthreads();
        }
        const int j0 = c * A.Kc, kc = min(A.Kc, A.K - j0);
        if (!PAD) {
            const uint4 *gin = reinterpret_cast<const uint4 *>(A.lat + (size_t)b * NN);
            for (int q = tid; q < NN / 4; q += nthr) reinterpret_cast<uint4 *>(buf0)[q] = __ldcg(gin + q);
        } else {
            const uint32_t *gin = A.lat + (size_t)b * NN;
            for (int q = tid; q < NN; q += nthr) buf0[(q / N) * ld + q % N] = __ldcg(gin + q);
        }
        for (int i = tid; i < n; i += nthr) {
            const size_t g = (size_t)b * n + i;
            S.st[i] = __ldcg(A.agent_state + g);
            S.xy[i] = __ldcg(A.agent_xy + 2 * g) | (__ldcg(A.agent_xy + 2 * g + 1) << 16);
            S.ada[i] = 0;
        }
        if (tid < 4) s_max[tid] = 0;
        if (DIAG && tid == 0) { s_tsum = 0.0; s_cov[0] = 0u; s_cov[1] = 0u; }
        __syncthreads();

        uint32_t *cb = buf0, *nb = buf1;
        int life = 0;
        for (int jl = 0; jl < kc; ++jl) {
            const int j = j0 + jl;
            if (warp == 0 && n > 0) dw_agents_phase(A, j, b, cb, S, lane, ld);
            __syncthreads();
            if (j == A.K - 1) {
                if (!PAD) {
                    uint4 *gp = reinterpret_cast<uint4 *>(A.lat_pre + (size_t)b * NN);
                    for (int q = tid; q < NN / 4; q += nthr) gp[q] = reinterpret_cast<const uint4 *>(cb)[q];
                } else {
                    uint32_t *gp = A.lat_pre + (size_t)b * NN;
                    for (int q = tid; q < NN; q += nthr) gp[q] = cb[(q / N) * ld + q % N];
                }
            }
            const StepCoef C = A.sc[j];
            uint32_t mx = 0;
            double tsum = 0.0;
            unsigned int cl = 0, cd = 0;
            for (int r = 0; r < rounds; ++r) {                      // uniform trip count: the fix-up below is warp-collective
                const int tile = tid + r * nthr;
                const bool active = tile < TT;
                const int ty = tile / T, tx = tile - ty * T;
                const int r0 = ty * 4, c0 = tx * 4;
                unsigned tiemin = 0xffffffffu;
                uint32_t m = 0;
                const int valid = PAD ? min(4, N - c0) : 4;
                if (active)
                    m = dw_tile_core<RowsTile4<PAD>, StoreTile4<PAD>, DIAG>(
                        A.F, C, RowsTile4<PAD>{cb, N, ld, r0, c0, c0 == 0 ? N - 1 : c0 - 1, c0 + 4 >= N ? c0 + 4 - N : c0 + 4, valid},
                        StoreTile4<PAD>{nb, N, ld, r0, c0, valid}, &tiemin, &tsum);
                const unsigned flagged = __ballot_sync(0xffffffffu, active && tiemin < A.F.tie_thresh);
                if (flagged) m = dw_fix_warp_tile4(&A, &A.sc[j], cb, nb, flagged, m, r0, c0, lane, N, ld);
                mx = __vmaxu2(mx, m);
                if (DIAG && active) {           // this tile's new covers (fix-ups included)
#pragma unroll
                    for (int i = 0; i < 4; ++i) {
                        const uint4 v = *reinterpret_cast<const uint4 *>(nb + (r0 + i) * N + c0);
                        cl += (v.x & 0xffffu) + (v.y & 0xffffu) + (v.z & 0xffffu) + (v.w & 0xffffu);
                        cd += (v.x >> 16) + (v.y >> 16) + (v.z >> 16) + (v.w >> 16);
                    }
                }
            }
            const unsigned ml = __reduce_max_sync(0xffffffffu, mx & 0xffffu), md = __reduce_max_sync(0xffffffffu, mx >> 16);
            int *sm = s_max + 2 * (jl & 1);
            if (lane == 0) { atomicMax(sm, (int)ml); atomicMax(sm + 1, (int)md); }
            if (DIAG) {
                for (int o = 16; o > 0; o >>= 1) tsum += __shfl_xor_sync(0xffffffffu, tsum, o);
                cl = __reduce_add_sync(0xffffffffu, cl);
                cd = __reduce_add_sync(0xffffffffu, cd);
                if (lane == 0) { atomicAdd(&s_tsum, tsum); atomicAdd(&s_cov[0], cl); atomicAdd(&s_cov[1], cd); }
            }
            __syncthreads();
            if (DIAG && tid == nthr - 1) {         // the last thread (any block size); warp 0's lane 0 does the bookkeeping below
                atomicAdd(A.series_T + j, s_tsum);
                atomicAdd(A.series_l + j, (unsigned long long)s_cov[0]);
                atomicAdd(A.series_d + j, (unsigned long long)s_cov[1]);
                s_tsum = 0.0; s_cov[0] = 0u; s_cov[1] = 0u;
            }
            if (warp == 0) {
                const bool grid_done = max(sm[0], sm[1]) <= 5;
                if (lane == 0) {
                    if (!grid_done) { life += 1; atomicAdd(A.alive + j, 1u); }
                    s_max[2 * ((jl + 1) & 1)] = 0;
                    s_max[2 * ((jl + 1) & 1) + 1] = 0;
                }
                for (int i = lane; i < n; i += 32) S.ada[i] += (S.st[i] < 0.1) ? 0 : 1;
            }
            uint32_t *tmp = cb; cb = nb; nb = tmp;
        }
        __syncthreads();
        if (!PAD) {
            uint4 *gout = reinterpret_cast<uint4 *>(A.lat + (size_t)b * NN);
            for (int q = tid; q < NN / 4; q += nthr) gout[q] = reinterpret_cast<const uint4 *>(cb)[q];
        } else {
            uint32_t *gout = A.lat + (size_t)b * NN;
            for (int q = tid; q < NN; q += nthr) gout[q] = cb[(q / N) * ld + q % N];
        }
        for (int i = tid; i < n; i += nthr) {
            const size_t g = (size_t)b * n + i;
            A.agent_state[g] = S.st[i];
            A.agent_xy[2 * g] = S.xy[i] & 0xffff;
            A.agent_xy[2 * g + 1] = S.xy[i] >> 16;
            if (A.count_life) A.agents_done_at[g] = __ldcg(A.agents_done_at + g) + S.ada[i];
            const double r = S.st[i];
            A.reward[g] = r;
            A.done[g] = r < 0.1;
        }
        if (tid == 0) {
            if (A.count_life) A.done_at[b] = __ldcg(A.done_at + b) + life;
            if (n == 0) {
                const int *sm = s_max + 2 * ((kc - 1) & 1);
                for (int ch = 0; ch < 2; ++ch) { A.reward[2 * b + ch] = sm[ch] > 0 ? 1.0 : 0.0; A.done[2 * b + ch] = sm[ch] > 0 ? 0 : 1; }
            }
        }
        __syncthreads();
        if (A.queue && tid == 0) {
            __threadfence();
            atomicExch(A.pair_done + b, (unsigned)(c + 1));
        }
    }
}

// fp64 grid channels 1,2 -> packed lattice; flags worlds whose covers are not exactly k/1000
__global__ void __launch_bounds__(256) k_grid_to_lattice(int B, size_t NN, const double *__restrict__ grid, uint32_t *__restrict__ lat,
                                                         unsigned int *off_lattice) {
    const size_t total = (size_t)B * NN;
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        const size_t b = i / NN, c = i - b * NN;
        const double l = grid[b * 7 * NN + NN + c], d = grid[b * 7 * NN + 2 * NN + c];
        const double kl = rint(l * 1000.0), kd = rint(d * 1000.0);
        const bool ok = kl >= 0.0 && kl <= 1000.0 && kd >= 0.0 && kd <= 1000.0 && kl / 1000.0 == l && kd / 1000.0 == d;
        if (!ok) atomicAdd(off_lattice, 1u);
        lat[i] = ok ? dw_pack((int)kl, (int)kd) : 0u;
    }
}

// debug hook: count k in [0,kmax] with dw_div1000(k) != k/1000.0 (must be 0: the division-free rounding is exact)
__global__ void k_debug_markstein(unsigned int kmax, unsigned int *bad) {
    for (unsigned int k = blockIdx.x * blockDim.x + threadIdx.x; k <= kmax; k += gridDim.x * blockDim.x) {
        const double kd = (double)k;
        if (dw_div1000(kd) != kd / 1000.0 || dw_div1000(-kd) != -kd / 1000.0) atomicAdd(bad, 1u);
    }
}

// debug/measurement hook: y[i] = dw_root4_fast(x[i])
__global__ void k_debug_root4(const double *x, double *y, int n) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) y[i] = dw_root4_fast(x[i]);
}
