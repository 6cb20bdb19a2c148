// Shared device-side definitions for the B200-native RLDaisyWorld step.
//
// "Literal" arithmetic = the canonical IEEE-binary64 operation order of the reference's step
// (daisy/daisy_world_rl.py:340-461 with daisy/nn/functional.py:12-49 restated as a 3x3 toroidal
// stencil).  The whole library is compiled with -fmad=false, so a*b+c below is two roundings exactly
// like NumPy; fused multiply-adds appear only where __fma_rn is written out (fast lattice path).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/daisyworld_b200.h"

// Physics constants as the kernels see them (copied from dw_config on every launch, so attribute
// mutation between steps behaves like the reference).
struct DevParams {
    int B, N, n_agents, pad_;
    double p, g, S, sigma, gamma, q, q2, temp_optimal, dt, agent_gamma;
    double ab, al, ad;
    double w[9];      // daisy-spread taps by neighbour, row-major (the env's kernel turned 180 degrees, make_params_cfg)
    double adj[9];    // adjacent-albedo taps by neighbour, likewise (centre tap skipped when it is 0, see dw_literal_cell)
    double mask[9];   // observation mask
    // screened forward (dw_screened_cell): sum of the adjacent-albedo taps, tie-filter half-widths (in units of 0.001) of
    // the covers, the bare fraction and the temperatures, accepted range of T^4; screen = 0 forces the literal path
    double adj_sum, eps_c, eps_b, eps_T, xlo, xhi;
    int screen, pad2_;
};

__device__ __forceinline__ double dw_root4(double x) { return sqrt(sqrt(x)); }
__device__ __forceinline__ double dw_pow4(double x) { double x2 = x * x; return x2 * x2; }
__device__ __forceinline__ double dw_div1000(double k);
// np.round(x, 3) = rint(x*1000)/1000 (true division); the division-free form is exact for |rint(x*1000)| <= 2e6
__device__ __forceinline__ double dw_round3(double x) {
    const double k = rint(x * 1000.0);
    return fabs(k) <= 2.0e6 ? dw_div1000(k) : k / 1000.0;
}
__device__ __forceinline__ double dw_clip01(double x) {
    x = x < 0.0 ? 0.0 : x;
    return x > 1.0 ? 1.0 : x;
}

struct LitCell {
    double nb, nl, nd;             // unrounded new covers (clipped l', d'; b' = (p-l')-d')
    double T, Tl, Td, Te;          // unrounded temperatures
    double beta, beta_l, beta_d;   // growth rates
    double dl, dd;                 // growth
    double b0;                     // (p-l)-d of the centre cell (written back in place by forward, :381)
};

// One cell of RLDaisyWorld.forward in literal order. l9/d9: 3x3 neighbourhood (row-major, wrap applied
// by the caller) of the light / dark covers; SL = S*L.
__device__ __forceinline__ LitCell dw_literal_cell(const DevParams &P, double SL, const double (&l9)[9],
                                                   const double (&d9)[9]) {
    LitCell o;
    double nb_b = 0.0, nb_l = 0.0, nb_d = 0.0, rho_l = 0.0, rho_d = 0.0;
    bool first = true;
#pragma unroll
    for (int k = 0; k < 9; ++k) {
        double tl = P.w[k] * l9[k], td = P.w[k] * d9[k];
        if (k == 0) { rho_l = tl; rho_d = td; }
        else { rho_l = rho_l + tl; rho_d = rho_d + td; }
        if (k == 4 && P.adj[4] == 0.0) continue;      // zero centre tap is skipped (oracle/daisy_numpy.py)
        double bk = (P.p - l9[k]) - d9[k];
        double vb = P.adj[k] * bk, vl = P.adj[k] * l9[k], vd = P.adj[k] * d9[k];
        if (first) { nb_b = vb; nb_l = vl; nb_d = vd; first = false; }
        else { nb_b = nb_b + vb; nb_l = nb_l + vl; nb_d = nb_d + vd; }
    }
    const double l = l9[4], d = d9[4];
    o.b0 = (P.p - l) - d;
    const double Al = (P.ab * o.b0 + P.al * l) + P.ad * d;
    const double A = (P.ab * nb_b + P.al * nb_l) + P.ad * nb_d;
    o.Te = dw_root4((SL * (1 - A)) / P.sigma);
    o.T = dw_root4(P.q * (A - Al) + dw_pow4(o.Te));
    const double T4 = dw_pow4(o.T);
    o.Tl = dw_root4(P.q2 * (Al - P.al) + T4);
    o.Td = dw_root4(P.q2 * (Al - P.ad) + T4);
    const double dT = P.temp_optimal - o.T, dTl = P.temp_optimal - o.Tl, dTd = P.temp_optimal - o.Td;
    o.beta = 1 - P.g * (dT * dT);
    o.beta_l = 1 - P.g * (dTl * dTl);
    o.beta_d = 1 - P.g * (dTd * dTd);
    const double rb = (P.p - rho_l) - rho_d;
    o.dl = rho_l * (rb * o.beta_l - P.gamma);
    o.dd = rho_d * (rb * o.beta_d - P.gamma);
    o.nl = dw_clip01(l + P.dt * o.dl);
    o.nd = dw_clip01(d + P.dt * o.dd);
    o.nb = (P.p - o.nl) - o.nd;
    return o;
}

// Packed lattice cell: light milli-cover in bits 0..15, dark in bits 16..31 (both 0..1000).
__device__ __forceinline__ uint32_t dw_pack(int kl, int kd) { return (uint32_t)kl | ((uint32_t)kd << 16); }
// k/1000 correctly rounded (== the value np.round(x,3) stores) without a division: Markstein's sequence
// q = k*(1/1000), r = k - 1000q (exact in an FMA), q + r*(1/1000).  Verified exhaustively against k/1000.0 for every
// integer 0 <= k <= 2e6 (tests/test_oracle_c.py::test_markstein_division_exhaustive and the GPU twin).
__device__ __forceinline__ double dw_div1000(double k) {
    const double q = k * 0.001;
    const double r = __fma_rn(-1000.0, q, k);
    return __fma_rn(r, 0.001, q);
}
__device__ __forceinline__ double dw_milli(uint32_t k) {
    return dw_div1000(__hiloint2double(0x43300000, (int)k) - 4503599627370496.0);
}

// ---- fast fourth root ------------------------------------------------------------------------------------
__device__ __forceinline__ double dw_rsqrt_approx(double x) {
    double r;
    asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(x));
    return r;
}
__device__ __forceinline__ double dw_rcp_approx(double x) {
    double r;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(x));
    return r;
}
// X^(1/4) for X in the physical range (1e8..1e11): two MUFU.RSQ64H seeds (s1 ~ X^-1/2, y0 = rsqrt(s1) ~ X^1/4), then
// one Newton step on y^4 = X with 1/(4 y0^3) approximated by s1*s1*y0/4.  Relative error <= ~2e-12 (measured in
// tests/test_gpu_fused_internals.py), 6 fp64-pipe ops.
__device__ __forceinline__ double dw_root4_fast(double X) {
    const double s1 = dw_rsqrt_approx(X);
    const double y0 = dw_rsqrt_approx(s1);                    // X^(1/4) (1+d), |d| < 2^-21
    const double z = y0 * y0;
    const double res = __fma_rn(-z, z, X);                    // X - y0^4
    const double a = s1 * s1;
    const double b3 = a * y0;                                 // ~ 1/y0^3
    return __fma_rn(res * b3, 0.25, y0);
}


// ---- screened forward cell -----------------------------------------------------------------------------------------
// The materialising kernels need the literal result of every channel AFTER np.round(., 3). dw_literal_cell costs ~300 fp64
// instructions (eight IEEE square roots, a division, one rounding per operation); this evaluates the same cell with fused
// multiply-adds, the temperatures straight from T^4 = q (A - Al) + S L (1 - A) / sigma (no Te round trip) and the fast
// fourth root, then checks every value it is about to round: if x * 1000 is further from a rounding tie than the error
// bound of the fast evaluation (P.eps_*: fourth root 3e-12 relative, everything else a few ulp; make_params_cfg), the
// rounded result IS the literal one. Otherwise -- or if the cell leaves the range the bound assumes (T in 150..400 K,
// neighbourhood densities in [0, 1], NaNs) -- it returns false and the caller recomputes the cell literally (~1e-4 of cells).
struct ScrCell {
    double k[6];      // rint(1000 * {b', l', d', T, T_l, T_d}): the stored value is dw_k2v(k)
    double b0;        // (p - l) - d of the centre cell
};
__device__ __forceinline__ double dw_k2v(double k) { return fabs(k) <= 2.0e6 ? dw_div1000(k) : k / 1000.0; }
__device__ __forceinline__ bool dw_screen_round(double x, double eps, double &k) {
    const double s = x * 1000.0;
    k = rint(s);
    return 0.5 - fabs(s - k) > eps;
}
__device__ __forceinline__ bool dw_screened_cell(const DevParams &P, double SLs /* S L / sigma */, const double (&l9)[9],
                                                 const double (&d9)[9], ScrCell &o, double *raw = nullptr) {
    double rl = P.w[0] * l9[0], rd = P.w[0] * d9[0], sl = P.adj[0] * l9[0], sd = P.adj[0] * d9[0];
#pragma unroll
    for (int k = 1; k < 9; ++k) {
        rl = __fma_rn(P.w[k], l9[k], rl);
        rd = __fma_rn(P.w[k], d9[k], rd);
        sl = __fma_rn(P.adj[k], l9[k], sl);
        sd = __fma_rn(P.adj[k], d9[k], sd);
    }
    const double l = l9[4], d = d9[4];
    o.b0 = (P.p - l) - d;
    const double cl = P.al - P.ab, cd = P.ad - P.ab, abp = P.ab * P.p;
    const double A = __fma_rn(cl, sl, __fma_rn(cd, sd, abp * P.adj_sum));
    const double Al = __fma_rn(cl, l, __fma_rn(cd, d, abp));
    const double XT = __fma_rn(P.q, A - Al, SLs * (1.0 - A));
    const double Xl = __fma_rn(P.q2, Al - P.al, XT), Xd = __fma_rn(P.q2, Al - P.ad, XT);
    const double T = dw_root4_fast(XT), Tl = dw_root4_fast(Xl), Td = dw_root4_fast(Xd);
    const double dTl = P.temp_optimal - Tl, dTd = P.temp_optimal - Td;
    const double bl = __fma_rn(-P.g * dTl, dTl, 1.0), bd = __fma_rn(-P.g * dTd, dTd, 1.0);
    const double rb = (P.p - rl) - rd;
    const double nl = dw_clip01(__fma_rn(P.dt, rl * __fma_rn(rb, bl, -P.gamma), l));
    const double nd = dw_clip01(__fma_rn(P.dt, rd * __fma_rn(rb, bd, -P.gamma), d));
    const double nb = (P.p - nl) - nd;
    if (raw) { raw[0] = nb; raw[1] = nl; raw[2] = nd; raw[3] = T; raw[4] = Tl; raw[5] = Td; }   // dw_debug_screen_error
    bool ok = XT > P.xlo && XT < P.xhi && Xl > P.xlo && Xl < P.xhi && Xd > P.xlo && Xd < P.xhi;
    ok = ok && rl >= 0.0 && rl <= 1.000001 && rd >= 0.0 && rd <= 1.000001 && fabs(rb) <= 1.000001 && fabs(nb) <= 2000.0;
    ok = dw_screen_round(nb, P.eps_b, o.k[0]) && ok;
    ok = dw_screen_round(nl, P.eps_c, o.k[1]) && ok;
    ok = dw_screen_round(nd, P.eps_c, o.k[2]) && ok;
    ok = dw_screen_round(T, P.eps_T, o.k[3]) && ok;
    ok = dw_screen_round(Tl, P.eps_T, o.k[4]) && ok;
    ok = dw_screen_round(Td, P.eps_T, o.k[5]) && ok;
    return ok;
}
// the literal values in the same form
__device__ __forceinline__ void dw_literal_rounded(const DevParams &P, double SL, const double (&l9)[9], const double (&d9)[9], ScrCell &o) {
    const LitCell c = dw_literal_cell(P, SL, l9, d9);
    o.k[0] = rint(c.nb * 1000.0); o.k[1] = rint(c.nl * 1000.0); o.k[2] = rint(c.nd * 1000.0);
    o.k[3] = rint(c.T * 1000.0); o.k[4] = rint(c.Tl * 1000.0); o.k[5] = rint(c.Td * 1000.0);
    o.b0 = c.b0;
}

#define DW_CUDA_TRY(h, expr)                                                           \
    do {                                                                               \
        cudaError_t e__ = (expr);                                                      \
        if (e__ != cudaSuccess) return dw_fail((h), DW_E_CUDA, #expr, cudaGetErrorString(e__)); \
    } while (0)
