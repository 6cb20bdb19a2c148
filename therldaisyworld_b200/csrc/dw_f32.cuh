// fp32 mode (north_star: "1e-5 in fp32 mode"): the 7-channel grid of the current state materialised with fp32 ARITHMETIC
// from the packed lattice, 32 B of HBM traffic per cell instead of the fp64 materialisation's 64+ B (SURVEY section 8(d)).
//
// What is fp32 and what is not: the STATE stays on the exact integer lattice (a cover flipped by 0.001 feeds back, SURVEY
// H2/B.7), so channels 1, 2 are the fp32 roundings of the exact covers. The temperatures (channels 3, 4, 5; daisy_world_rl.py
// :396-421) are evaluated in binary32 -- FFMA accumulation of T^4, two MUFU.RSQ for the fourth root -- from the post-graze
// lattice the last step started from, then rounded to 3 decimals in fp32: ~5e-7 relative plus a possible 0.001 K rounding
// flip (3e-6), inside the 1e-5 tolerance. Channel 0 (b' = round(p - l'_unrounded - d'_unrounded, 3), :449-452) needs the
// UNROUNDED new covers: they are re-evaluated in fp32 too, and b' is accepted only when 1000 b' is further from a rounding
// tie than the fp32 error bound W (below); otherwise (a few % of cells) the cell goes through the fp64 fast path with its own
// tie filter and, at last, the literal cell -- so channel 0 is exactly the fp32 rounding of the reference's value.
//
// Error bound of the fp32 evaluation of x = k + rho (rho_b beta - dt gamma) (milli-cover; u = 2^-24):
//   X' (g^2 T^4) is accumulated small terms first, the constant last: |dX'|/X' <= 6u. MUFU.RSQ: 2^-22 relative (PTX ISA:
//   2^-22.9 over the positive finite range), twice: the fourth root is good to 1.5 * 2^-22 + 1.5u = 4.5e-7, T' = sqrt(g) T
//   <= sqrt(g) * 400 (range-checked), plus the rounding of sqrt(g) Topt: |d(dT')| <= eD = sqrt(g) (400 * 4.5e-7 + 2u Topt).
//   beta = 1 - dT'^2: |d beta| <= 2 |dT'| eD + 3u (1 + dT'^2). rho (all taps non-negative): 4u relative. rho_b: 8u dt.
//   |dx| <= rho [ |rho_b| (2 eD |dT'| + 3u (1 + dT'^2)) + 8u dt (1 + dT'^2) + 6u (|rho_b| (1 + dT'^2) + dt gamma) ] + 2u |x|
//        <= rho [ k1 |dT'| + k2 (1 + dT'^2) ] + c0,   k1 = 2 eD rbmax, k2 = u (17 rbmax + 8 dt), c0 = u (2000 + 6 * 1000 dt gamma),
//   rbmax = dt max(|p|, |p - 2|). The kernel uses W = 2 (W_l + W_d) + 4u * 1000 (factor 2: safety; last term: the two subtractions).
#pragma once
#include "dw_fused.cuh"

struct F32Coef {
    float w0, w12, w2, dtp, dtm, dtg;
    float xk_l, xk_d, xdd, topt, t0, tk_l, tk_d;
    float x0, xs_l, xs_d;              // per call (luminosity of the step being materialised)
    float inv_sqrt_g, p1000;
    float k1, k2, c0, c0b;             // error-bound coefficients (already including the safety factor)
    float xlo, xhi;                    // accepted range of X' (T in 150..400 K)
};

__device__ __forceinline__ float dw_rsqrt32(float x) {
    float r;
    asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r;
}
// k / 1000 in binary32 without a division (Markstein's sequence; equal to the correctly rounded quotient for every integer
// |k| <= 2^19, checked exhaustively on the device by dw_debug_markstein_f32 / tests/test_gpu_fused_internals.py)
__device__ __forceinline__ float dw_div1000f(float k) {
    const float q = k * 0.001f;
    const float r = __fmaf_rn(-1000.0f, q, k);
    return __fmaf_rn(r, 0.001f, q);
}
// rint for |x| < 2^22 by the magic-number add (FMA pipe instead of FRND on the XU pipe)
__device__ __forceinline__ float dw_rintf_small(float x) { return (x + 12582912.0f) - 12582912.0f; }
__device__ __forceinline__ float dw_round3f(float x) { return dw_div1000f(dw_rintf_small(x * 1000.0f)); }
// exact u16 -> binary32 without I2F (XU pipe): 2^23 + k by a byte permute / mask, minus 2^23
template <int HI>
__device__ __forceinline__ float dw_half2f(uint32_t p) {
    return __uint_as_float(__byte_perm(p, 0x4B000000u, HI ? 0x7632 : 0x7610)) - 8388608.0f;
}

// fp64 fast path of one cell, unrounded: new covers in milli units (dw_fast_cell without the rounding)
__device__ __forceinline__ void dw_fast_x(const FastCoef &F, const StepCoef &C, uint32_t pc, uint32_t E, uint32_t S, double &xl, double &xd) {
    const double kl = dw_u2d(pc & 0xffffu), kd = dw_u2d(pc >> 16);
    const double El = dw_u2d(E & 0xffffu), Ed = dw_u2d(E >> 16);
    const double Sl = dw_u2d(S & 0xffffu), Sd = dw_u2d(S >> 16);
    const double Rl = __fma_rn(F.w2, Sl, __fma_rn(F.w12, El, F.w0 * kl));
    const double Rd = __fma_rn(F.w2, Sd, __fma_rn(F.w12, Ed, F.w0 * kd));
    const double rb = __fma_rn(-F.dtm, Rl + Rd, F.dtp);
    const double Xl = __fma_rn(C.xs_l, Sl, __fma_rn(C.xs_d, Sd, __fma_rn(F.xk_l, kl, __fma_rn(F.xk_d, kd, C.x0))));
    const double Xd = Xl + F.xdd;
    const double dTl = F.topt - dw_root4_fast(Xl), dTd = F.topt - dw_root4_fast(Xd);
    xl = __fma_rn(Rl, __fma_rn(rb, __fma_rn(-dTl, dTl, 1.0), -F.dtg), kl);
    xd = __fma_rn(Rd, __fma_rn(rb, __fma_rn(-dTd, dTd, 1.0), -F.dtg), kd);
}

// fp64 tier of the bare fraction of one cell, shared by the fp32-mode kernels of the ensemble and of the giant world
// (csrc/dw_tiled.cuh) so that the tiers cannot diverge between the two lattice layouts. In: the cell's packed word pc, its
// neighbourhood sums E, S, and win(a, c) = the packed word of the window cell in row a, column c (0..2; (1, 1) is the cell)
// for the literal cell. Returns 1000 b' as the reference rounds it. A window over scalars: capturing index arrays makes
// the compiler drop the non-coherent loads of k_forward_f32's main loop.
template <class Win>
__device__ __forceinline__ float dw_f32_bare_tiers(const DevParams &P, const FastCoef &F, const StepCoef &C, uint32_t pc, uint32_t E,
                                                   uint32_t S, Win win, unsigned *nlit) {
    // lattice fast path, unrounded covers -> b' with the tie filter of the screened forward (P.eps_b, units of 0.001);
    // then the literal cell. (Range failures come here too: the fp64 fast path is exact-or-flagged on its own.)
    double dxl, dxd;
    dw_fast_x(F, C, pc, E, S, dxl, dxd);
    dxl = fmin(fmax(dxl, 0.0), 1000.0);
    dxd = fmin(fmax(dxd, 0.0), 1000.0);
    const double dxb = (1000.0 * P.p - dxl) - dxd;
    double kb64 = rint(dxb);
    const bool in_range = dxl == dxl && dxd == dxd && P.screen;     // NaN (X' <= 0): literal
    if (!in_range || !(0.5 - fabs(dxb - kb64) > P.eps_b)) {
        *nlit += 1;
        double l9[9], d9[9];
#pragma unroll
        for (int a = 0; a < 3; ++a)
#pragma unroll
            for (int c = 0; c < 3; ++c) {
                const uint32_t k = win(a, c);
                l9[a * 3 + c] = dw_milli(k & 0xffffu);
                d9[a * 3 + c] = dw_milli(k >> 16);
            }
        const LitCell o = dw_literal_cell(P, C.SL, l9, d9);
        kb64 = rint(o.nb * 1000.0);
    }
    return (float)kb64;
}

// fp64 tier of cell (x, y) of a wrapped N x N lattice (rare: ~2 % of cells; out of line, called after the thread's stores so
// that nothing of the fp32 evaluation is live across the call).
// Measured alternatives (4000 worlds of 64x64, this in-place call: 0.185 ms): deferring the ~3e5 flagged cells to a dense second
// kernel through a work list costs more than the divergence it removes -- one shared counter 0.257 ms (the warp-aggregated
// atomics serialise), per-warp list segments without atomics 0.230 ms.
__device__ __noinline__ float dw_f32_bare_slow(const DevParams *Pp, const FastCoef *Fp, const StepCoef *Cp, const uint32_t *g, unsigned N,
                                               unsigned x, unsigned y, unsigned *nlit) {
    const unsigned xm = x == 0 ? N - 1 : x - 1, xp = x == N - 1 ? 0 : x + 1;
    const unsigned ym = y == 0 ? N - 1 : y - 1, yp = y == N - 1 ? 0 : y + 1;
    const uint32_t *r0 = g + xm * N, *r1 = g + x * N, *r2 = g + xp * N;
    const uint32_t pc = r1[y];
    const uint32_t E = r1[ym] + r1[yp] + r0[y] + r2[y];
    const uint32_t S = E + r0[ym] + r0[yp] + r2[ym] + r2[yp];
    return dw_f32_bare_tiers(*Pp, *Fp, *Cp, pc, E, S, [=](int a, int c) {
        return g[(a == 0 ? xm : a == 1 ? x : xp) * N + (c == 0 ? ym : c == 1 ? y : yp)];
    }, nlit);
}

struct F32Out { float b, T, Tl, Td; bool ok; };
// fp32 evaluation of one cell from its packed neighbourhood sums: the three temperatures (sqrt(g) T) and the bare fraction
// (milli units, rounded) with the verdict of its screen
__device__ __forceinline__ F32Out dw_f32_cell(const F32Coef &Q, uint32_t pc, uint32_t E, uint32_t S) {
    const float kl = dw_half2f<0>(pc), kd = dw_half2f<1>(pc);
    const float El = dw_half2f<0>(E), Ed = dw_half2f<1>(E);
    const float Sl = dw_half2f<0>(S), Sd = dw_half2f<1>(S);
    const float Rl = __fmaf_rn(Q.w2, Sl, __fmaf_rn(Q.w12, El, Q.w0 * kl));
    const float Rd = __fmaf_rn(Q.w2, Sd, __fmaf_rn(Q.w12, Ed, Q.w0 * kd));
    const float rb = __fmaf_rn(-Q.dtm, Rl + Rd, Q.dtp);
    // small terms first, the constant last (error bound in the header)
    const float Xl = __fmaf_rn(Q.xs_l, Sl, __fmaf_rn(Q.xs_d, Sd, __fmaf_rn(Q.xk_l, kl, Q.xk_d * kd))) + Q.x0;
    const float Xd = Xl + Q.xdd;
    const float XT = __fmaf_rn(Q.tk_l, kl, __fmaf_rn(Q.tk_d, kd, Q.t0)) + Xl;
    F32Out o;
    o.Tl = dw_rsqrt32(dw_rsqrt32(Xl));
    o.Td = dw_rsqrt32(dw_rsqrt32(Xd));
    o.T = dw_rsqrt32(dw_rsqrt32(XT));
    const float dTl = Q.topt - o.Tl, dTd = Q.topt - o.Td;
    const float bl = __fmaf_rn(-dTl, dTl, 1.0f), bd = __fmaf_rn(-dTd, dTd, 1.0f);
    float xl = __fmaf_rn(Rl, __fmaf_rn(rb, bl, -Q.dtg), kl);
    float xd = __fmaf_rn(Rd, __fmaf_rn(rb, bd, -Q.dtg), kd);
    xl = fminf(fmaxf(xl, 0.0f), 1000.0f);
    xd = fminf(fmaxf(xd, 0.0f), 1000.0f);
    const float xb = (Q.p1000 - xl) - xd;
    o.b = dw_rintf_small(xb);
    const float Wl = __fmaf_rn(Rl, __fmaf_rn(Q.k1, fabsf(dTl), Q.k2 * (2.0f - bl)), Q.c0);
    const float Wd = __fmaf_rn(Rd, __fmaf_rn(Q.k1, fabsf(dTd), Q.k2 * (2.0f - bd)), Q.c0);
    const float lo = fminf(fminf(Xl, Xd), XT), hi = fmaxf(fmaxf(Xl, Xd), XT);
    o.ok = lo > Q.xlo && hi < Q.xhi && (0.5f - fabsf(xb - o.b) > Wl + Wd + Q.c0b);
    return o;
}

// W cells per thread (W = 2: horizontally adjacent, N even, 8-byte loads and stores; W = 1: any N). pre: post-graze lattice
// the last step started from; cur: the lattice after that step (exact new covers). out: float [B,7,N,N], channels 0..6
// written (4 before the agent stamp). stats[0] += cells sent to the fp64 tier, stats[1] += cells that needed the literal cell.
struct F32Args { DevParams P; FastCoef F; StepCoef C; F32Coef Q; };
template <int W>
__global__ void __launch_bounds__(256, 4) k_forward_f32(const __grid_constant__ F32Args A, const uint32_t *__restrict__ pre,
                                                        const uint32_t *__restrict__ cur, float *__restrict__ out,
                                                        unsigned long long *stats) {
    const DevParams &P = A.P;
    const F32Coef &Q = A.Q;
    const unsigned N = (unsigned)P.N, NN = N * N, GN = NN / W, gN = N / W;
    const size_t total = (size_t)P.B * GN, stride = (size_t)gridDim.x * blockDim.x;
    size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
    CellWalk w(i, stride, GN);
    unsigned n64 = 0, nlit = 0;
    for (; i < total; i += stride, w.next()) {
        const unsigned x = w.c / gN, y = W * (w.c - x * gN);
        const unsigned xm = x == 0 ? N - 1 : x - 1, xp = x == N - 1 ? 0 : x + 1;
        const unsigned ym = y == 0 ? N - 1 : y - 1, yq = y + W >= N ? 0 : y + W;
        const uint32_t *g = pre + (size_t)w.b * NN;
        uint32_t row[3][W + 2];                  // rows x-1, x, x+1; columns y-1 .. y+W
        const unsigned rs[3] = {xm * N, x * N, xp * N};
#pragma unroll
        for (int a = 0; a < 3; ++a) {
            row[a][0] = g[rs[a] + ym];
            if (W == 2) {
                const uint2 v = *reinterpret_cast<const uint2 *>(g + rs[a] + y);
                row[a][1] = v.x; row[a][2] = v.y;
            } else row[a][1] = g[rs[a] + y];
            row[a][W + 1] = g[rs[a] + yq];
        }
        uint32_t pn[W];
        if (W == 2) {
            const uint2 v = *reinterpret_cast<const uint2 *>(cur + (size_t)w.b * NN + x * N + y);
            pn[0] = v.x; pn[W - 1] = v.y;
        } else pn[0] = cur[(size_t)w.b * NN + x * N + y];
        float ch[7][W];
        bool ok[W];
#pragma unroll
        for (int c = 0; c < W; ++c) {
            const uint32_t pc = row[1][c + 1];
            const uint32_t E = row[1][c] + row[1][c + 2] + row[0][c + 1] + row[2][c + 1];
            const uint32_t S = E + row[0][c] + row[0][c + 2] + row[2][c] + row[2][c + 2];
            const F32Out o = dw_f32_cell(Q, pc, E, S);
            ok[c] = o.ok;
            ch[0][c] = dw_div1000f(o.b);
            ch[1][c] = dw_div1000f(dw_half2f<0>(pn[c]));
            ch[2][c] = dw_div1000f(dw_half2f<1>(pn[c]));
            ch[3][c] = dw_round3f(o.T * Q.inv_sqrt_g);
            ch[4][c] = dw_round3f(o.Tl * Q.inv_sqrt_g);
            ch[5][c] = dw_round3f(o.Td * Q.inv_sqrt_g);
            ch[6][c] = 0.0f;
        }
        float *ob = out + (size_t)w.b * 7 * NN + x * N + y;
#pragma unroll
        for (int q = 0; q < 7; ++q) {
            if (W == 2) *reinterpret_cast<float2 *>(ob + (size_t)q * NN) = make_float2(ch[q][0], ch[q][W - 1]);
            else ob[(size_t)q * NN] = ch[q][0];
        }
        // cells whose fp32 bare fraction sits within its error bound of a rounding tie (or outside the accepted range):
        // fp64 tier, the stored channel 0 is overwritten
#pragma unroll
        for (int c = 0; c < W; ++c) {
            if (!ok[c]) {
                n64 += 1;
                ob[c] = dw_div1000f(dw_f32_bare_slow(&A.P, &A.F, &A.C, g, N, x, y + c, &nlit));
            }
        }
    }
    if (stats) {
        n64 = __reduce_add_sync(__activemask(), n64);
        nlit = __reduce_add_sync(__activemask(), nlit);
        if ((threadIdx.x & 31) == 0 && n64) { atomicAdd(stats, (unsigned long long)n64); atomicAdd(stats + 1, (unsigned long long)nlit); }
    }
}

// debug hook: integers |k| <= kmax whose dw_div1000f differs from the correctly rounded binary32 quotient (must be 0)
__global__ void k_debug_markstein_f32(unsigned int kmax, unsigned int *bad) {
    for (unsigned int k = blockIdx.x * blockDim.x + threadIdx.x; k <= kmax; k += gridDim.x * blockDim.x) {
        const float kf = (float)k;
        if (dw_div1000f(kf) != __fdiv_rn(kf, 1000.0f) || dw_div1000f(-kf) != __fdiv_rn(-kf, 1000.0f)) atomicAdd(bad, 1u);
    }
}

// agent stamp on channel 4 (daisy_world_rl.py:454-459): agent order, dead agents included, later agents win
__global__ void __launch_bounds__(128) k_stamp_f32(DevParams P, float *grid, const int32_t *agent_xy, const double *agent_state) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= P.B) return;
    const int N = P.N, n = P.n_agents;
    const size_t NN = (size_t)N * N;
    float *g4 = grid + (size_t)b * 7 * NN + 4 * NN;
    for (int i = 0; i < n; ++i) {
        const int x = agent_xy[((size_t)b * n + i) * 2], y = agent_xy[((size_t)b * n + i) * 2 + 1];
        g4[(size_t)x * N + y] = (float)agent_state[(size_t)b * n + i];
    }
}

// get_obs on the fp32 grid (daisy_world_rl.py:246-263)
__global__ void __launch_bounds__(256) k_obs_f32(DevParams P, const float *__restrict__ grid, const int32_t *__restrict__ pos, int nb, int m,
                                                 float *__restrict__ obs) {
    const size_t total = (size_t)nb * m * 63;
    const int N = P.N;
    const size_t NN = (size_t)N * N;
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        const size_t ag = i / 63;
        const int e = (int)(i - ag * 63);
        const int ch = e / 9, a = (e % 9) / 3, c = e % 3;
        const int b = (int)(ag / m);
        int x = pos[ag * 2] + a - 1, y = pos[ag * 2 + 1] + c - 1;
        x = ((x % N) + N) % N;
        y = ((y % N) + N) % N;
        obs[i] = grid[((size_t)b * 7 + ch) * NN + (size_t)x * N + y] * (float)P.mask[a * 3 + c];
    }
}
