// Materialising ("generic") kernels: one reference step on the fp64 grid[B,7,N,N], any N >= 1,
// any (off-lattice) cover values.  Used by dw_step_packed / dw_forward / dw_get_grid / dw_get_diag.
// Roofline: writes 6 live channels + reads 2 => 64 B per cell-update (SURVEY 8(d)); in literal
// arithmetic (6 fp64 sqrt pairs, 7 fp64 divides per cell) it is fp64-pipe bound at about the same rate.
#pragma once
#include "dw_common.cuh"

// ---- input loaders --------------------------------------------------------------------------------
struct SrcGrid {           // fp64 grid[B,7,N,N]
    const double *g;
    size_t world_stride;   // 7*N*N
    size_t NN;
    __device__ __forceinline__ double l(int b, size_t c) const { return g[b * world_stride + NN + c]; }
    __device__ __forceinline__ double d(int b, size_t c) const { return g[b * world_stride + 2 * NN + c]; }
};
struct SrcCov {            // fp64 cover planes [B,2,N,N] (light, dark): the lean reset state
    const double *c;
    size_t NN;
    __device__ __forceinline__ double l(int b, size_t k) const { return c[(size_t)b * 2 * NN + k]; }
    __device__ __forceinline__ double d(int b, size_t k) const { return c[(size_t)b * 2 * NN + NN + k]; }
};
struct SrcLattice {        // packed milli-covers [B,N,N]
    const uint32_t *k;
    size_t NN;
    __device__ __forceinline__ double l(int b, size_t c) const { return dw_milli(k[b * NN + c] & 0xffffu); }
    __device__ __forceinline__ double d(int b, size_t c) const { return dw_milli(k[b * NN + c] >> 16); }
};

__device__ __forceinline__ void dw_atomic_max_pos(unsigned long long *addr, double v);
// Per-world views: the world's base pointers are formed once per cell, the nine taps are small offsets from them.
struct ViewF64 {
    const double *pl, *pd;
    __device__ __forceinline__ double l(int k) const { return pl[k]; }
    __device__ __forceinline__ double d(int k) const { return pd[k]; }
    // taps k, k+1 (k even, N even: 16-byte aligned) of both fields
    __device__ __forceinline__ void pair(int k, double &l0, double &l1, double &d0, double &d1) const {
        const double2 a = *reinterpret_cast<const double2 *>(pl + k), b = *reinterpret_cast<const double2 *>(pd + k);
        l0 = a.x; l1 = a.y; d0 = b.x; d1 = b.y;
    }
    __device__ __forceinline__ void one(int k, double &l0, double &d0) const { l0 = pl[k]; d0 = pd[k]; }
};
struct ViewLat {
    const uint32_t *pk;
    __device__ __forceinline__ double l(int k) const { return dw_milli(pk[k] & 0xffffu); }
    __device__ __forceinline__ double d(int k) const { return dw_milli(pk[k] >> 16); }
    __device__ __forceinline__ void pair(int k, double &l0, double &l1, double &d0, double &d1) const {
        const uint2 a = *reinterpret_cast<const uint2 *>(pk + k);
        l0 = dw_milli(a.x & 0xffffu); d0 = dw_milli(a.x >> 16); l1 = dw_milli(a.y & 0xffffu); d1 = dw_milli(a.y >> 16);
    }
    __device__ __forceinline__ void one(int k, double &l0, double &d0) const {
        const uint32_t a = pk[k];
        l0 = dw_milli(a & 0xffffu); d0 = dw_milli(a >> 16);
    }
};
// 3x3 neighbourhoods of the two cells (x, y), (x, y + 1), y even, N even: per row one aligned pair + the two halo taps
template <class View>
__device__ __forceinline__ void dw_load9x2(const View &v, int N, int x, int y, double (&la)[9], double (&da)[9], double (&lb)[9],
                                           double (&db)[9]) {
    const int xm = x == 0 ? N - 1 : x - 1, xp = x == N - 1 ? 0 : x + 1;
    const int ym = y == 0 ? N - 1 : y - 1, yq = y + 2 == N ? 0 : y + 2;
    const int rs[3] = {xm * N, x * N, xp * N};
#pragma unroll
    for (int a = 0; a < 3; ++a) {
        double l0, l1, d0, d1, lm, dm, lq, dq;
        v.pair(rs[a] + y, l0, l1, d0, d1);
        v.one(rs[a] + ym, lm, dm);
        v.one(rs[a] + yq, lq, dq);
        la[a * 3] = lm; la[a * 3 + 1] = l0; la[a * 3 + 2] = l1;
        da[a * 3] = dm; da[a * 3 + 1] = d0; da[a * 3 + 2] = d1;
        lb[a * 3] = l0; lb[a * 3 + 1] = l1; lb[a * 3 + 2] = lq;
        db[a * 3] = d0; db[a * 3 + 1] = d1; db[a * 3 + 2] = dq;
    }
}
__device__ __forceinline__ ViewF64 dw_view(const SrcGrid &s, unsigned b) {
    const double *w = s.g + (size_t)b * s.world_stride + s.NN;
    return ViewF64{w, w + s.NN};
}
__device__ __forceinline__ ViewF64 dw_view(const SrcCov &s, unsigned b) {
    const double *w = s.c + (size_t)b * 2 * s.NN;
    return ViewF64{w, w + s.NN};
}
__device__ __forceinline__ ViewLat dw_view(const SrcLattice &s, unsigned b) { return ViewLat{s.k + (size_t)b * s.NN}; }
template <class View>
__device__ __forceinline__ void dw_load9v(const View &v, int N, int x, int y, double (&l9)[9], double (&d9)[9]) {
    const int xm = x == 0 ? N - 1 : x - 1, xp = x == N - 1 ? 0 : x + 1;
    const int ym = y == 0 ? N - 1 : y - 1, yp = y == N - 1 ? 0 : y + 1;
    const int rs[3] = {xm * N, x * N, xp * N}, ys[3] = {ym, y, yp};
#pragma unroll
    for (int a = 0; a < 3; ++a)
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            l9[a * 3 + c] = v.l(rs[a] + ys[c]);
            d9[a * 3 + c] = v.d(rs[a] + ys[c]);
        }
}

// (world, cell) of a grid-stride loop over B*N*N cells, advanced without 64-bit divisions
struct CellWalk {
    unsigned b, c, sb, sc, NN;
    __device__ __forceinline__ CellWalk(size_t i0, size_t stride, unsigned nn) : NN(nn) {
        b = (unsigned)(i0 / nn); c = (unsigned)(i0 - (size_t)b * nn);
        sb = (unsigned)(stride / nn); sc = (unsigned)(stride - (size_t)sb * nn);
    }
    __device__ __forceinline__ void next() {
        c += sc; b += sb;
        if (c >= NN) { c -= NN; b += 1; }
    }
};

// per-world maxima of the new covers (k = 1000 * cover, integer valued) into world_max [B,2] (bit patterns of the doubles)
__device__ __forceinline__ void dw_world_max_update(unsigned long long *world_max, unsigned b, double kl, double kd) {
    const unsigned m = __activemask();
    const unsigned b0 = __shfl_sync(m, b, 0);
    int il = (int)kl, id = (int)kd;
    if (m == 0xffffffffu && __all_sync(m, b == b0)) {          // whole warp in one world: two REDUX instead of 32 atomics
        il = __reduce_max_sync(m, il);
        id = __reduce_max_sync(m, id);
        if ((threadIdx.x & 31) != 0) return;
    }
    dw_atomic_max_pos(world_max + 2 * b, dw_div1000((double)il));
    dw_atomic_max_pos(world_max + 2 * b + 1, dw_div1000((double)id));
}

template <class Src>
__device__ __forceinline__ void dw_load9(const Src &src, int b, int N, int x, int y, double (&l9)[9], double (&d9)[9]) {
    const int xm = x == 0 ? N - 1 : x - 1, xp = x == N - 1 ? 0 : x + 1;
    const int ym = y == 0 ? N - 1 : y - 1, yp = y == N - 1 ? 0 : y + 1;
    const int xs[3] = {xm, x, xp}, ys[3] = {ym, y, yp};
#pragma unroll
    for (int a = 0; a < 3; ++a)
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            const size_t k = (size_t)xs[a] * N + ys[c];
            l9[a * 3 + c] = src.l(b, k);
            d9[a * 3 + c] = src.d(b, k);
        }
}

// order-preserving map of non-negative doubles to u64 for atomicMax
__device__ __forceinline__ void dw_atomic_max_pos(unsigned long long *addr, double v) {
    if (v > 0.0) atomicMax(addr, (unsigned long long)__double_as_longlong(v));
}

// ---- forward (daisy_world_rl.py:434-452) ----------------------------------------------------------
// One thread per cell. out: grid[B,7,N,N] (channels 0..5 written, 6 written only if zero6).
// writeback_b0: also store (p-l)-d into channel 0 of the INPUT grid (reference :381 mutates its argument).
// world_max: [B,2] u64 bit patterns of max(l'), max(d') (rounded), pre-zeroed; may be NULL.
template <class Src>
__global__ void __launch_bounds__(256) k_forward(DevParams P, double SL, Src src, double *__restrict__ out,
                                                 double *writeback_b0, unsigned long long *world_max, int zero6) {
    const unsigned NN = (unsigned)P.N * (unsigned)P.N;
    const size_t total = (size_t)P.B * NN, stride = (size_t)gridDim.x * blockDim.x;
    const double SLs = SL / P.sigma;
    size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
    CellWalk w(i, stride, NN);
    for (; i < total; i += stride, w.next()) {
        const int x = (int)(w.c / (unsigned)P.N), y = (int)(w.c - (unsigned)x * (unsigned)P.N);
        double l9[9], d9[9];
        dw_load9v(dw_view(src, w.b), P.N, x, y, l9, d9);
        ScrCell o;
        double v[6];
        if (P.screen && dw_screened_cell(P, SLs, l9, d9, o)) {
#pragma unroll
            for (int q = 0; q < 6; ++q) v[q] = dw_div1000(o.k[q]);            // |k| <= 2e6 inside the screened range
        } else {
            dw_literal_rounded(P, SL, l9, d9, o);
#pragma unroll
            for (int q = 0; q < 6; ++q) v[q] = dw_k2v(o.k[q]);
        }
        double *ob = out + (size_t)w.b * 7 * NN + w.c;
#pragma unroll
        for (int q = 0; q < 6; ++q) ob[(size_t)q * NN] = v[q];
        if (zero6) ob[(size_t)6 * NN] = 0.0;
        if (writeback_b0) writeback_b0[(size_t)w.b * 7 * NN + w.c] = o.b0;
        if (world_max) dw_world_max_update(world_max, w.b, o.k[1], o.k[2]);
    }
}

// Same literal step, but only the new covers are kept, as packed lattice words (the first step of a fused run from the
// off-lattice reset state: nothing else of the 7-channel grid feeds the next step).
template <class Src>
__global__ void __launch_bounds__(256) k_forward_lattice(DevParams P, double SL, Src src, uint32_t *__restrict__ lat_out,
                                                         unsigned long long *world_max) {
    const unsigned NN = (unsigned)P.N * (unsigned)P.N;
    const size_t total = (size_t)P.B * NN, stride = (size_t)gridDim.x * blockDim.x;
    const double SLs = SL / P.sigma;
    size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
    CellWalk w(i, stride, NN);
    for (; i < total; i += stride, w.next()) {
        const int x = (int)(w.c / (unsigned)P.N), y = (int)(w.c - (unsigned)x * (unsigned)P.N);
        double l9[9], d9[9];
        dw_load9v(dw_view(src, w.b), P.N, x, y, l9, d9);
        ScrCell o;
        if (!(P.screen && dw_screened_cell(P, SLs, l9, d9, o))) dw_literal_rounded(P, SL, l9, d9, o);
        lat_out[i] = ((uint32_t)(int)o.k[1]) | ((uint32_t)(int)o.k[2] << 16);
        if (world_max) dw_world_max_update(world_max, w.b, o.k[1], o.k[2]);
    }
}

// Two horizontally adjacent cells per thread (N even): aligned 16-byte loads of the shared taps and 16-byte stores of every
// channel halve the memory instructions and the address arithmetic per cell. Same screened evaluation, same results.
template <class Src>
__global__ void __launch_bounds__(256, 3) k_forward_x2(DevParams P, double SL, Src src, double *__restrict__ out,
                                                    double *writeback_b0, unsigned long long *world_max, int zero6) {
    const unsigned NN = (unsigned)P.N * (unsigned)P.N, HN = NN >> 1, hN = (unsigned)P.N >> 1;
    const size_t total = (size_t)P.B * HN, stride = (size_t)gridDim.x * blockDim.x;
    const double SLs = SL / P.sigma;
    size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
    CellWalk w(i, stride, HN);
    for (; i < total; i += stride, w.next()) {
        const int x = (int)(w.c / hN), y = 2 * (int)(w.c - (unsigned)x * hN);
        double la[9], da[9], lb[9], db[9];
        dw_load9x2(dw_view(src, w.b), P.N, x, y, la, da, lb, db);
        ScrCell oa, ob2;
        double va[6], vb[6];
        if (P.screen && dw_screened_cell(P, SLs, la, da, oa)) {
#pragma unroll
            for (int q = 0; q < 6; ++q) va[q] = dw_div1000(oa.k[q]);
        } else {
            dw_literal_rounded(P, SL, la, da, oa);
#pragma unroll
            for (int q = 0; q < 6; ++q) va[q] = dw_k2v(oa.k[q]);
        }
        if (P.screen && dw_screened_cell(P, SLs, lb, db, ob2)) {
#pragma unroll
            for (int q = 0; q < 6; ++q) vb[q] = dw_div1000(ob2.k[q]);
        } else {
            dw_literal_rounded(P, SL, lb, db, ob2);
#pragma unroll
            for (int q = 0; q < 6; ++q) vb[q] = dw_k2v(ob2.k[q]);
        }
        const unsigned c = 2u * w.c;
        double *op = out + (size_t)w.b * 7 * NN + c;
#pragma unroll
        for (int q = 0; q < 6; ++q) *reinterpret_cast<double2 *>(op + (size_t)q * NN) = make_double2(va[q], vb[q]);
        if (zero6) *reinterpret_cast<double2 *>(op + (size_t)6 * NN) = make_double2(0.0, 0.0);
        if (writeback_b0) *reinterpret_cast<double2 *>(writeback_b0 + (size_t)w.b * 7 * NN + c) = make_double2(oa.b0, ob2.b0);
        if (world_max) dw_world_max_update(world_max, w.b, fmax(oa.k[1], ob2.k[1]), fmax(oa.k[2], ob2.k[2]));
    }
}

template <class Src>
__global__ void __launch_bounds__(256, 3) k_forward_lattice_x2(DevParams P, double SL, Src src, uint32_t *__restrict__ lat_out,
                                                            unsigned long long *world_max) {
    const unsigned NN = (unsigned)P.N * (unsigned)P.N, HN = NN >> 1, hN = (unsigned)P.N >> 1;
    const size_t total = (size_t)P.B * HN, stride = (size_t)gridDim.x * blockDim.x;
    const double SLs = SL / P.sigma;
    size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
    CellWalk w(i, stride, HN);
    for (; i < total; i += stride, w.next()) {
        const int x = (int)(w.c / hN), y = 2 * (int)(w.c - (unsigned)x * hN);
        double la[9], da[9], lb[9], db[9];
        dw_load9x2(dw_view(src, w.b), P.N, x, y, la, da, lb, db);
        ScrCell oa, ob2;
        if (!(P.screen && dw_screened_cell(P, SLs, la, da, oa))) dw_literal_rounded(P, SL, la, da, oa);
        if (!(P.screen && dw_screened_cell(P, SLs, lb, db, ob2))) dw_literal_rounded(P, SL, lb, db, ob2);
        *reinterpret_cast<uint2 *>(lat_out + 2 * i) = make_uint2(((uint32_t)(int)oa.k[1]) | ((uint32_t)(int)oa.k[2] << 16),
                                                                 ((uint32_t)(int)ob2.k[1]) | ((uint32_t)(int)ob2.k[2] << 16));
        if (world_max) dw_world_max_update(world_max, w.b, fmax(oa.k[1], ob2.k[1]), fmax(oa.k[2], ob2.k[2]));
    }
}

// Test hook: largest deviation (in units of 0.001, the rounding grid) between the screened evaluation and the literal one
// over the cells the screen ACCEPTS its range for, per channel group {covers, bare fraction, temperatures}; the tie filters
// P.eps_c / eps_b / eps_T must stay well above these. out: 3 u64 holding the bit patterns of non-negative doubles.
template <class Src>
__global__ void __launch_bounds__(256) k_debug_screen_error(DevParams P, double SL, Src src, unsigned long long *out) {
    const unsigned NN = (unsigned)P.N * (unsigned)P.N;
    const size_t total = (size_t)P.B * NN, stride = (size_t)gridDim.x * blockDim.x;
    const double SLs = SL / P.sigma;
    size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
    CellWalk w(i, stride, NN);
    for (; i < total; i += stride, w.next()) {
        const int x = (int)(w.c / (unsigned)P.N), y = (int)(w.c - (unsigned)x * (unsigned)P.N);
        double l9[9], d9[9], raw[6];
        dw_load9v(dw_view(src, w.b), P.N, x, y, l9, d9);
        ScrCell o;
        dw_screened_cell(P, SLs, l9, d9, o, raw);
        const bool in_range = raw[3] > 150.0 && raw[3] < 400.0 && raw[4] > 150.0 && raw[4] < 400.0 && raw[5] > 150.0 && raw[5] < 400.0;
        if (!in_range) continue;
        const LitCell c = dw_literal_cell(P, SL, l9, d9);
        const double ec = fmax(fabs(raw[1] - c.nl), fabs(raw[2] - c.nd)) * 1000.0, eb = fabs(raw[0] - c.nb) * 1000.0;
        const double eT = fmax(fabs(raw[3] - c.T), fmax(fabs(raw[4] - c.Tl), fabs(raw[5] - c.Td))) * 1000.0;
        dw_atomic_max_pos(out, ec);
        dw_atomic_max_pos(out + 1, eb);
        dw_atomic_max_pos(out + 2, eT);
    }
}

// ---- initial temperatures (initialize_grid, daisy_world_rl.py:304-324): ch0 and ch3..5, UNROUNDED ----
__global__ void __launch_bounds__(256) k_init_fields(DevParams P, double SL, double *grid) {
    const size_t NN = (size_t)P.N * P.N;
    const size_t total = (size_t)P.B * NN;
    SrcGrid src{grid, 7 * NN, NN};
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        const int b = (int)(i / NN);
        const size_t c = i - (size_t)b * NN;
        const int x = (int)(c / P.N), y = (int)(c - (size_t)x * P.N);
        double l9[9], d9[9];
        dw_load9(src, b, P.N, x, y, l9, d9);
        const LitCell o = dw_literal_cell(P, SL, l9, d9);
        double *ob = grid + (size_t)b * 7 * NN + c;
        ob[0] = o.b0;
        ob[3 * NN] = o.T;
        ob[4 * NN] = o.Tl;
        ob[5 * NN] = o.Td;
    }
}

// ---- diagnostics: unrounded side-effect attributes of the last forward -------------------------
template <class Src>
__global__ void __launch_bounds__(256) k_diag(DevParams P, double SL, Src src, int which, double *__restrict__ out) {
    const size_t NN = (size_t)P.N * P.N;
    const size_t total = (size_t)P.B * NN;
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        const int b = (int)(i / NN);
        const size_t c = i - (size_t)b * NN;
        const int x = (int)(c / P.N), y = (int)(c - (size_t)x * P.N);
        double l9[9], d9[9];
        dw_load9(src, b, P.N, x, y, l9, d9);
        const LitCell o = dw_literal_cell(P, SL, l9, d9);
        switch (which) {
            case DW_DIAG_TEMP: out[i] = o.T; break;
            case DW_DIAG_TEMP_LIGHT: out[i] = o.Tl; break;
            case DW_DIAG_TEMP_DARK: out[i] = o.Td; break;
            case DW_DIAG_TEMP_EFFECTIVE: out[i] = o.Te; break;
            case DW_DIAG_BETA: out[i] = o.beta; break;
            case DW_DIAG_BETA_L: out[i] = o.beta_l; break;
            case DW_DIAG_BETA_D: out[i] = o.beta_d; break;
            default:
                out[(size_t)b * 2 * NN + c] = o.dl;
                out[(size_t)b * 2 * NN + NN + c] = o.dd;
        }
    }
}

// ---- agents (update_agents, daisy_world_rl.py:181-244; Greedy, agents/greedy.py:16-30) -------------
// counter RNG for DW_POLICY_RANDOM (throughput ensembles only; parity for stochastic policies is by replay)
__host__ __device__ __forceinline__ uint32_t dw_hash_rng(uint64_t seed, uint32_t world, uint32_t agent, uint32_t step) {
    uint64_t z = seed + 0x9E3779B97F4A7C15ull * ((uint64_t)world * 0x10001ull + agent + 1) + ((uint64_t)step << 32);
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    z ^= z >> 31;
    return (uint32_t)(z >> 32);
}
// DW_POLICY_EPS_GREEDY: the policy of one step -- one coin per step for the whole ensemble, like the single
// np.random.rand() of Greedy.__call__ (agents/greedy.py:23). Resolved on the host (per launch or per step-table entry).
__host__ __device__ __forceinline__ int dw_resolve_policy(int policy, double epsilon, uint64_t seed, uint32_t step) {
    if (policy != DW_POLICY_EPS_GREEDY) return policy;
    const double u = (double)dw_hash_rng(seed ^ 0x5EEDC01D5EEDC01Dull, 0xffffffffu, 0xffffffffu, step) * (1.0 / 4294967296.0);
    return u < epsilon ? DW_POLICY_RANDOM : DW_POLICY_GREEDY;
}

// greedy / anti-greedy choice from the four Von Neumann neighbours' l+d (candidates in action order
// 4..7 = (x,y-1), (x-1,y), (x+1,y), (x,y+1)); first extremum wins like np.argmax/np.argmin.
__device__ __forceinline__ int dw_greedy_pick(const double (&food)[4], bool greedy) {
    int best = 0;
    double bv = food[0];
#pragma unroll
    for (int k = 1; k < 4; ++k) {
        const bool better = greedy ? (food[k] > bv) : (food[k] < bv);
        if (better) { bv = food[k]; best = k; }
    }
    return 4 + best;
}

// One thread per world, agents strictly in index order (grazing conflicts: lower index eats first).
// action: device int8 [ab,am] (policy REPLAY/explicit), ignored for other policies.
// covers: base pointer of the cover storage; world w's light / dark planes start at w*world_stride + l_off / d_off
// (7-channel grid: 7NN, NN, 2NN; lean cover planes: 2NN, 0, NN).
__global__ void __launch_bounds__(128) k_agents_grid(DevParams P, double *covers, size_t world_stride, size_t l_off, size_t d_off,
                                                     int32_t *agent_xy, double *agent_state, const int8_t *action, int ab, int am,
                                                     int policy, uint64_t seed, uint32_t step, uint32_t world0, int clip = 1) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= P.B) return;
    const int N = P.N, n = P.n_agents;
    double *gl = covers + (size_t)b * world_stride + l_off, *gd = covers + (size_t)b * world_stride + d_off;
    int32_t *xy = agent_xy + (size_t)b * n * 2;
    double *st = agent_state + (size_t)b * n;
    for (int i = 0; i < n; ++i) st[i] = st[i] - P.agent_gamma;
    const int lim_b = (policy == DW_POLICY_REPLAY) ? ab : P.B, lim_m = (policy == DW_POLICY_REPLAY) ? am : n;
    // Observation-driven policies decide from the grid BEFORE any agent of this step moves or grazes
    // (obs comes from the previous step). Two passes keep that order: decide all, then apply in order.
    if (b < lim_b) {
        for (int i = 0; i < lim_m; ++i) {
            int a;
            const int x = xy[2 * i], y = xy[2 * i + 1];
            if (policy == DW_POLICY_REPLAY) a = action[(size_t)b * am + i];
            else if (policy == DW_POLICY_NONE) a = 0;
            else if (policy == DW_POLICY_RANDOM) a = (int)(dw_hash_rng(seed, world0 + b, i, step) % 9u);
            else {
                const int xm = x == 0 ? N - 1 : x - 1, xp = x == N - 1 ? 0 : x + 1;
                const int ym = y == 0 ? N - 1 : y - 1, yp = y == N - 1 ? 0 : y + 1;
                const size_t c[4] = {(size_t)x * N + ym, (size_t)xm * N + y, (size_t)xp * N + y, (size_t)x * N + yp};
                double food[4];
#pragma unroll
                for (int k = 0; k < 4; ++k) food[k] = gl[c[k]] + gd[c[k]];
                a = dw_greedy_pick(food, policy == DW_POLICY_GREEDY);
            }
            // stash the decision in the (unused by now) high bits of x: keeps the kernel free of scratch memory
            xy[2 * i] = x | (a << 24);
        }
        for (int i = 0; i < lim_m; ++i) {
            const int packed = xy[2 * i];
            const int a = (packed >> 24) & 0xf;
            int x = packed & 0xffffff, y = xy[2 * i + 1];
            if (st[i] > 0.0) {
                if (a != 8) {
                    switch (a & 3) {
                        case 0: y -= 1; break;
                        case 1: x -= 1; break;
                        case 2: x += 1; break;
                        default: y += 1; break;
                    }
                }
                x = x < 0 ? x + N : (x >= N ? x - N : x);
                y = y < 0 ? y + N : (y >= N ? y - N : y);
                if (a > 4) {
                    const size_t c = (size_t)x * N + y;
                    st[i] = st[i] + (gl[c] + gd[c]);
                    gl[c] *= 0.0;
                    gd[c] *= 0.0;
                }
            }
            xy[2 * i] = x;
            xy[2 * i + 1] = y;
        }
    }
    if (clip)                          // collision_mode == 1 resolves collisions on the unclipped states first (k_collide)
        for (int i = 0; i < n; ++i) st[i] = dw_clip01(st[i]);
}

// ---- collision_mode == 1 (daisy_world_rl.py:220-242) ----
// np.sum of m contiguous doubles as NumPy adds them (0 + pairwise sum: fewer than 8 sequentially, up to 128 with 8
// interleaved accumulators, larger blocks split in halves rounded down to a multiple of 8).
__device__ double dw_numpy_pairwise(const double *a, int m) {
    if (m < 8) {
        double r = 0.0;
        for (int i = 0; i < m; ++i) r = r + a[i];
        return r;
    }
    if (m <= 128) {
        double r[8];
        for (int k = 0; k < 8; ++k) r[k] = a[k];
        int i = 8;
        for (; i < m - (m % 8); i += 8)
            for (int k = 0; k < 8; ++k) r[k] = r[k] + a[i + k];
        double res = ((r[0] + r[1]) + (r[2] + r[3])) + ((r[4] + r[5]) + (r[6] + r[7]));
        for (; i < m; ++i) res = res + a[i];
        return res;
    }
    int m2 = m / 2;
    m2 -= m2 % 8;
    return dw_numpy_pairwise(a, m2) + dw_numpy_pairwise(a + m2, m - m2);
}

// One thread per world, after k_agents_grid(clip = 0). The reference scans the cells of a world in row-major order and,
// where more than one agent sits, draws npr.rand(1, n, 1): noise[k, 0..n) is the k-th such draw of the whole batch,
// cell_off[b] the index of world b's first one (the host front counts the shared cells from the post-move positions and
// draws from the caller's global stream in that order). Per shared cell: temp = 1.0 * state + 0.01 * noise for all n
// agents, winner value = max over the residents, eat = np.sum of the states of the residents whose temp differs from
// it (unclipped, dead agents included), every agent whose temp EQUALS the winner value gains penalty * eat; the losers
// keep their state (the reference's zeroing assigns into a copy, :242). Then the clip of :244.
// mismatch counts worlds whose number of shared cells differs from the host's.
__global__ void __launch_bounds__(128) k_collide(DevParams P, const int32_t *agent_xy, double *agent_state, const double *noise,
                                                 const int32_t *cell_off, double penalty, double *losers_scratch, unsigned int *mismatch) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= P.B) return;
    const int N = P.N, n = P.n_agents;
    const int32_t *xy = agent_xy + (size_t)b * n * 2;
    double *st = agent_state + (size_t)b * n;
    double *los = losers_scratch + (size_t)b * n;
    int k = cell_off[b];
    const int kend = cell_off[b + 1];
    int last = -1;
    for (;;) {
        int key = 0x7fffffff;
        for (int i = 0; i < n; ++i) {
            const int c = xy[2 * i] * N + xy[2 * i + 1];
            if (c > last && c < key) key = c;
        }
        if (key == 0x7fffffff) break;
        last = key;
        int residents = 0;
        for (int i = 0; i < n; ++i) residents += (xy[2 * i] * N + xy[2 * i + 1] == key) ? 1 : 0;
        if (residents < 2) continue;
        if (k >= kend) { k += 1; continue; }          // more shared cells than the host counted: reported below
        const double *nz = noise + (size_t)k * n;
        k += 1;
        double winner = 0.0;
        bool first = true;
        for (int i = 0; i < n; ++i)
            if (xy[2 * i] * N + xy[2 * i + 1] == key) {
                const double t = 1.0 * st[i] + 0.01 * nz[i];
                winner = first ? t : fmax(winner, t);
                first = false;
            }
        int m = 0;
        for (int i = 0; i < n; ++i)
            if (xy[2 * i] * N + xy[2 * i + 1] == key && (1.0 * st[i] + 0.01 * nz[i]) != winner) los[m++] = st[i];
        const double eat = 0.0 + dw_numpy_pairwise(los, m);
        for (int i = 0; i < n; ++i)
            if ((1.0 * st[i] + 0.01 * nz[i]) == winner) st[i] = st[i] + penalty * eat;
    }
    if (k != kend) atomicAdd(mismatch, 1u);
    for (int i = 0; i < n; ++i) st[i] = dw_clip01(st[i]);
}

// ---- stamp + reward/done + lifespan counters (forward :454-459, step :486-492, notebook cell 2) ----
// One thread per world. world_max as produced by k_forward (NULL = skip counters / n_agents==0 reward).
__global__ void __launch_bounds__(128) k_stamp_reward(DevParams P, double *grid, const int32_t *agent_xy,
                                                      const double *agent_state, const unsigned long long *world_max,
                                                      double *reward, uint8_t *done, int64_t *done_at,
                                                      int64_t *agents_done_at, unsigned int *alive_count) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= P.B) return;
    const int N = P.N, n = P.n_agents;
    const size_t NN = (size_t)N * N;
    if (grid) {                        // lean runs keep no 7-channel grid: the stamp happens when one is materialised
        double *g4 = grid + (size_t)b * 7 * NN + 4 * NN;
        for (int i = 0; i < n; ++i) {
            const int x = agent_xy[((size_t)b * n + i) * 2], y = agent_xy[((size_t)b * n + i) * 2 + 1];
            g4[(size_t)x * N + y] = agent_state[(size_t)b * n + i];
        }
    }
    if (n > 0) {
        for (int i = 0; i < n; ++i) {
            double r = agent_state[(size_t)b * n + i];
            r = r * (r > 0.0 ? 1.0 : 0.0);
            const bool dn = r < 0.1;
            if (reward) reward[(size_t)b * n + i] = r;
            if (done) done[(size_t)b * n + i] = dn;
            if (agents_done_at) agents_done_at[(size_t)b * n + i] += dn ? 0 : 1;
        }
    } else if (world_max) {
        for (int c = 0; c < 2; ++c) {
            const bool r = __longlong_as_double((long long)world_max[2 * b + c]) > 0.0;
            if (reward) reward[2 * b + c] = r ? 1.0 : 0.0;
            if (done) done[2 * b + c] = r ? 0 : 1;
        }
    }
    if (world_max && done_at) {
        const double m = fmax(__longlong_as_double((long long)world_max[2 * b]),
                              __longlong_as_double((long long)world_max[2 * b + 1]));
        const bool grid_done = m <= 0.005;
        done_at[b] += grid_done ? 0 : 1;
        if (!grid_done && alive_count) atomicAdd(alive_count, 1u);
    }
}

// ---- observations (get_obs, daisy_world_rl.py:246-263) -----------------------------------------------
// One thread per output element of obs[b,m,7,3,3]; positions: int32 [b,m,2].
__global__ void __launch_bounds__(256) k_obs(DevParams P, const double *__restrict__ grid, const int32_t *__restrict__ pos,
                                             int nb, int m, double *__restrict__ obs) {
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
        obs[i] = grid[((size_t)b * 7 + ch) * NN + (size_t)x * N + y] * P.mask[a * 3 + c];
    }
}

// Observations straight from the state the last forward STARTED from (post-graze lattice / cover planes / grid): the
// window cells are re-evaluated literally, which reproduces exactly what forward wrote there (b' from the unrounded
// covers, rounded temperatures, agent stamp: highest index on a cell wins, dead agents included) without materialising
// the whole 7-channel grid. One thread per (agent, window cell). pos: [nb,m,2] window centres (the agents' own positions
// for step()'s observation, caller-supplied ones for get_obs(agent_indices)); world of window (b, i) is b.
// init != 0: the state right after reset() instead -- src holds the initial covers themselves and the window shows
// initialize_grid's UNROUNDED fields (ch0 = p-l-d, covers, T, T_light, T_dark; no agent stamp; daisy_world_rl.py:304-324).
template <class Src>
__global__ void __launch_bounds__(256) k_obs_from_pre(DevParams P, double SL, Src src, const int32_t *__restrict__ pos, int nb, int m,
                                                      const int32_t *__restrict__ agent_xy, const double *__restrict__ agent_state,
                                                      double *__restrict__ obs, int init) {
    const int N = P.N, n = P.n_agents;
    const size_t total = (size_t)nb * m * 9;
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        const size_t ag = i / 9;
        const int w = (int)(i - ag * 9), b = (int)(ag / m);
        double *o = obs + ag * 63 + w;
        const double mk = P.mask[w];
        int x = pos[ag * 2] + w / 3 - 1, y = pos[ag * 2 + 1] + w % 3 - 1;
        x = ((x % N) + N) % N;
        y = ((y % N) + N) % N;
        double l9[9], d9[9];
        dw_load9(src, b, N, x, y, l9, d9);
        if (init) {
            const LitCell c = dw_literal_cell(P, SL, l9, d9);
            o[0] = c.b0 * mk; o[9] = l9[4] * mk; o[18] = d9[4] * mk; o[27] = c.T * mk; o[36] = c.Tl * mk; o[45] = c.Td * mk;
            o[54] = 0.0 * mk;
            continue;
        }
        ScrCell c;                                          // what forward stored there: screened, literal next to ties
        if (!(P.screen && dw_screened_cell(P, SL / P.sigma, l9, d9, c))) dw_literal_rounded(P, SL, l9, d9, c);
        double ch4 = dw_k2v(c.k[4]);
        for (int k = 0; k < n; ++k) {                       // forward :454-459, agents in order: the last one stays
            const size_t a2 = (size_t)b * n + k;
            if (agent_xy[a2 * 2] == x && agent_xy[a2 * 2 + 1] == y) ch4 = agent_state[a2];
        }
        o[0] = dw_k2v(c.k[0]) * mk;
        o[9] = dw_k2v(c.k[1]) * mk;
        o[18] = dw_k2v(c.k[2]) * mk;
        o[27] = dw_k2v(c.k[3]) * mk;
        o[36] = ch4 * mk;
        o[45] = dw_k2v(c.k[5]) * mk;
        o[54] = 0.0 * mk;
    }
}

// MLP.get_action (daisy/agents/mlp.py:97-116): x(63) -> relu(x W1)(16) -> relu(. W2)(32) -> . W3 (9) -> argmax (first
// maximum, like np.argmax). One thread per agent; relu(v) = v * (v > 0) as in the reference (:20).
// Population mode (wpm > 0, ES fitness rollouts, daisy/evo/sges.py:161-168): the worlds come in blocks of wpm per member;
// the first `half` agents of a world use the member's weights, the rest the adversary's.
__global__ void __launch_bounds__(128) k_mlp_act(const double *__restrict__ w, const double *__restrict__ obs, size_t count,
                                                 int8_t *__restrict__ action, int wpm, int n, int half, int adversary) {
    const size_t a = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
    if (a >= count) return;
    if (wpm > 0) {
        const size_t b = a / n;
        const int i = (int)(a - b * n);
        w += (size_t)(i < half ? (int)(b / wpm) : adversary) * (63 * 16 + 16 * 32 + 32 * 9);
    }
    const double *x = obs + a * 63;
    const double *w1 = w, *w2 = w + 63 * 16, *w3 = w2 + 16 * 32;
    double h1[16], h2[32];
#pragma unroll
    for (int o = 0; o < 16; ++o) h1[o] = 0.0;
    for (int k = 0; k < 63; ++k) {
        const double xk = x[k];
#pragma unroll
        for (int o = 0; o < 16; ++o) h1[o] = h1[o] + xk * w1[k * 16 + o];
    }
#pragma unroll
    for (int o = 0; o < 16; ++o) h1[o] = h1[o] * (h1[o] > 0.0 ? 1.0 : 0.0);
#pragma unroll
    for (int o = 0; o < 32; ++o) h2[o] = 0.0;
#pragma unroll
    for (int k = 0; k < 16; ++k) {
#pragma unroll
        for (int o = 0; o < 32; ++o) h2[o] = h2[o] + h1[k] * w2[k * 32 + o];
    }
#pragma unroll
    for (int o = 0; o < 32; ++o) h2[o] = h2[o] * (h2[o] > 0.0 ? 1.0 : 0.0);
    int best = 0;
    double bv = 0.0;
#pragma unroll
    for (int o = 0; o < 9; ++o) {
        double s = 0.0;
#pragma unroll
        for (int k = 0; k < 32; ++k) s = s + h2[k] * w3[k * 9 + o];
        if (o == 0 || s > bv) { bv = s; best = o; }
    }
    action[a] = (int8_t)best;
}

// Observation window + network in one kernel, one warp per agent (the policy path between one-step launches): lanes 0..8
// re-evaluate the window cells from the pre-state (as k_obs_from_pre), the 63 inputs go through shared memory, then lanes
// are output neurons (16, 32, 9) and the argmax is taken by lane 0. Same summation order as k_mlp_act.
template <class Src>
__global__ void __launch_bounds__(128) k_obs_mlp(DevParams P, double SL, Src src, const int32_t *__restrict__ agent_xy,
                                                 const double *__restrict__ agent_state, const double *__restrict__ w, size_t count,
                                                 int8_t *__restrict__ action, int wpm, int half, int adversary) {
    __shared__ double s_x[4][64], s_h1[4][16], s_h2[4][32], s_o[4][9];
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const size_t a = blockIdx.x * (size_t)(blockDim.x >> 5) + wib;
    if (a >= count) return;                                   // whole warps leave together
    const int N = P.N, n = P.n_agents;
    const int b = (int)(a / n);
    if (wpm > 0) w += (size_t)((int)(a - (size_t)b * n) < half ? b / wpm : adversary) * (63 * 16 + 16 * 32 + 32 * 9);
    double *x = s_x[wib];
    if (lane < 9) {
        const double m = P.mask[lane];
        int cx = agent_xy[a * 2] + lane / 3 - 1, cy = agent_xy[a * 2 + 1] + lane % 3 - 1;
        cx = cx < 0 ? cx + N : (cx >= N ? cx - N : cx);
        cy = cy < 0 ? cy + N : (cy >= N ? cy - N : cy);
        double l9[9], d9[9];
        dw_load9(src, b, N, cx, cy, l9, d9);
        ScrCell c;
        if (!(P.screen && dw_screened_cell(P, SL / P.sigma, l9, d9, c))) dw_literal_rounded(P, SL, l9, d9, c);
        double ch4 = dw_k2v(c.k[4]);
        for (int k = 0; k < n; ++k) {
            const size_t a2 = (size_t)b * n + k;
            if (agent_xy[a2 * 2] == cx && agent_xy[a2 * 2 + 1] == cy) ch4 = agent_state[a2];
        }
        x[lane] = dw_k2v(c.k[0]) * m;
        x[9 + lane] = dw_k2v(c.k[1]) * m;
        x[18 + lane] = dw_k2v(c.k[2]) * m;
        x[27 + lane] = dw_k2v(c.k[3]) * m;
        x[36 + lane] = ch4 * m;
        x[45 + lane] = dw_k2v(c.k[5]) * m;
        x[54 + lane] = 0.0 * m;
    }
    __syncwarp();
    const double *w1 = w, *w2 = w + 63 * 16, *w3 = w2 + 16 * 32;
    if (lane < 16) {
        double h = 0.0;
        for (int k = 0; k < 63; ++k) h = h + x[k] * w1[k * 16 + lane];
        s_h1[wib][lane] = h * (h > 0.0 ? 1.0 : 0.0);
    }
    __syncwarp();
    {
        double h = 0.0;
#pragma unroll
        for (int k = 0; k < 16; ++k) h = h + s_h1[wib][k] * w2[k * 32 + lane];
        s_h2[wib][lane] = h * (h > 0.0 ? 1.0 : 0.0);
    }
    __syncwarp();
    if (lane < 9) {
        double o = 0.0;
#pragma unroll
        for (int k = 0; k < 32; ++k) o = o + s_h2[wib][k] * w3[k * 9 + lane];
        s_o[wib][lane] = o;
    }
    __syncwarp();
    if (lane == 0) {
        int best = 0;
        double bv = s_o[wib][0];
#pragma unroll
        for (int o = 1; o < 9; ++o) if (s_o[wib][o] > bv) { bv = s_o[wib][o]; best = o; }
        action[a] = (int8_t)best;
    }
}

// One step of the population bookkeeping of get_fitness (sges.py:170-175), one block per member: while the member's loop
// is alive, sum_reward += mean(reward[:, :half]) over its worlds, the per-agent (1 - done) counters are carried along, and
// the loop ends after the step in which all of its agents are done.
__global__ void __launch_bounds__(128) k_pop_accumulate(int wpm, int n, int half, const double *__restrict__ reward,
                                                        const uint8_t *__restrict__ done, const int64_t *__restrict__ agents_done_at,
                                                        double *sum_reward, int *member_done, int64_t *member_steps, int64_t *frozen,
                                                        long long step_count, unsigned int *n_done) {
    const int m = blockIdx.x;
    if (member_done[m]) return;
    __shared__ double s_sum[4];
    __shared__ int s_alive[4];
    const size_t base = (size_t)m * wpm * n;
    double sum = 0.0;
    int alive = 0;
    for (int k = threadIdx.x; k < wpm * n; k += blockDim.x) {
        if (k % n < half) sum += reward[base + k];
        alive += done[base + k] ? 0 : 1;
        frozen[base + k] = agents_done_at[base + k];
    }
    for (int o = 16; o > 0; o >>= 1) {
        sum += __shfl_xor_sync(0xffffffffu, sum, o);
        alive += __shfl_xor_sync(0xffffffffu, alive, o);
    }
    if ((threadIdx.x & 31) == 0) { s_sum[threadIdx.x >> 5] = sum; s_alive[threadIdx.x >> 5] = alive; }
    __syncthreads();
    if (threadIdx.x == 0) {
        const double tot = ((s_sum[0] + s_sum[1]) + s_sum[2]) + s_sum[3];
        const int al = s_alive[0] + s_alive[1] + s_alive[2] + s_alive[3];
        sum_reward[m] += tot / (double)(wpm * half);
        member_steps[m] = step_count;
        if (al == 0) { member_done[m] = 1; atomicAdd(n_done, 1u); }
    }
}

// agents_done_at -= number of steps after step j of the last chunk in which the agent was not done (alive_mask, see FusedArgs)
__global__ void __launch_bounds__(256) k_trim_lifespans(size_t count, int j, const unsigned long long *__restrict__ mask,
                                                        int64_t *__restrict__ agents_done_at) {
    const size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
    if (i >= count || j >= 63) return;
    agents_done_at[i] -= __popcll(mask[i] >> (j + 1));
}

// The same bookkeeping for S steps at once from the recorded per-step agent states (fused population segments: the policy
// and the steps ran inside one launch, FusedArgs::rew_series). rew: [S][Bn] state after each step's update_agents = the
// step's reward (done = reward < 0.1); frozen[] advances by (1 - done) per step while the member's loop is alive, exactly
// what copying agents_done_at does in k_pop_accumulate. Same summation order as k_pop_accumulate.
__global__ void __launch_bounds__(128) k_pop_post(int S, int wpm, int n, int half, const double *__restrict__ rew, size_t Bn,
                                                  double *sum_reward, int *member_done, int64_t *member_steps, int64_t *frozen,
                                                  long long step0, unsigned int *n_done) {
    const int m = blockIdx.x;
    __shared__ double s_sum[4];
    __shared__ int s_alive[4];
    __shared__ int s_stop;
    if (member_done[m]) return;
    const size_t base = (size_t)m * wpm * n;
    for (int t = 0; t < S; ++t) {
        const double *r = rew + (size_t)t * Bn + base;
        double sum = 0.0;
        int alive = 0;
        for (int k = threadIdx.x; k < wpm * n; k += blockDim.x) {
            const double v = r[k];
            const bool dn = v < 0.1;
            if (k % n < half) sum += v;
            alive += dn ? 0 : 1;
            frozen[base + k] += dn ? 0 : 1;
        }
        for (int o = 16; o > 0; o >>= 1) {
            sum += __shfl_xor_sync(0xffffffffu, sum, o);
            alive += __shfl_xor_sync(0xffffffffu, alive, o);
        }
        if ((threadIdx.x & 31) == 0) { s_sum[threadIdx.x >> 5] = sum; s_alive[threadIdx.x >> 5] = alive; }
        __syncthreads();
        if (threadIdx.x == 0) {
            const double tot = ((s_sum[0] + s_sum[1]) + s_sum[2]) + s_sum[3];
            const int al = s_alive[0] + s_alive[1] + s_alive[2] + s_alive[3];
            sum_reward[m] += tot / (double)(wpm * half);
            member_steps[m] = step0 + t + 1;
            s_stop = al == 0;
            if (al == 0) { member_done[m] = 1; atomicAdd(n_done, 1u); }
        }
        __syncthreads();
        if (s_stop) return;
    }
}

// ---- ensemble statistics of a field (deterministic two-stage reduction: per-block partials, then one block) --------------
// partial[b] = {sum, sum of squares, min, max}
__device__ __forceinline__ void dw_stats_block_reduce(double s, double q, double mn, double mx, double *out4) {
    __shared__ double sh[4][8];
    for (int o = 16; o > 0; o >>= 1) {
        s += __shfl_xor_sync(0xffffffffu, s, o);
        q += __shfl_xor_sync(0xffffffffu, q, o);
        mn = fmin(mn, __shfl_xor_sync(0xffffffffu, mn, o));
        mx = fmax(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    }
    const int w = threadIdx.x >> 5;
    if ((threadIdx.x & 31) == 0) { sh[0][w] = s; sh[1][w] = q; sh[2][w] = mn; sh[3][w] = mx; }
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int i = 1; i < (int)(blockDim.x >> 5); ++i) { s += sh[0][i]; q += sh[1][i]; mn = fmin(mn, sh[2][i]); mx = fmax(mx, sh[3][i]); }
        out4[0] = s; out4[1] = q; out4[2] = mn; out4[3] = mx;
    }
}
// sums are taken of (x - x[0]): shifted data keeps the variance free of the E[x^2] - mean^2 cancellation
__global__ void __launch_bounds__(256) k_stats_partial(const double *__restrict__ x, size_t n, double *__restrict__ partial) {
    double s = 0.0, q = 0.0, mn = 1e300, mx = -1e300;
    const double shift = x[0];
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        const double v = x[i], d = v - shift;
        s += d; q += d * d; mn = fmin(mn, v); mx = fmax(mx, v);
    }
    dw_stats_block_reduce(s, q, mn, mx, partial + 4 * blockIdx.x);
}
__global__ void __launch_bounds__(256) k_stats_final(const double *__restrict__ partial, int blocks, double count, const double *__restrict__ x,
                                                     double *__restrict__ out) {
    double s = 0.0, q = 0.0, mn = 1e300, mx = -1e300;
    for (int i = threadIdx.x; i < blocks; i += blockDim.x) {
        s += partial[4 * i]; q += partial[4 * i + 1]; mn = fmin(mn, partial[4 * i + 2]); mx = fmax(mx, partial[4 * i + 3]);
    }
    __shared__ double r[4];
    dw_stats_block_reduce(s, q, mn, mx, r);
    if (threadIdx.x == 0) {
        const double dm = r[0] / count, var = r[1] / count - dm * dm;
        out[0] = x[0] + dm; out[1] = sqrt(var > 0.0 ? var : 0.0); out[2] = r[2]; out[3] = r[3];
    }
}
// covers of the packed lattice: {sum light, sum dark, max light, max dark} in milli units per block (exact integers)
__global__ void __launch_bounds__(256) k_lattice_cover_partial(const uint32_t *__restrict__ lat, size_t n, double *__restrict__ partial) {
    unsigned long long sl = 0, sd = 0;
    unsigned int ml = 0, md = 0;
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        const uint32_t w = lat[i];
        sl += w & 0xffffu; sd += w >> 16; ml = max(ml, w & 0xffffu); md = max(md, w >> 16);
    }
    // reuse the generic block reduce: sums in the s/q slots, maxima through the max slot (two passes keep it simple)
    double o1[4], o2[4];
    dw_stats_block_reduce((double)sl, (double)sd, 0.0, (double)ml, o1);
    __syncthreads();
    dw_stats_block_reduce(0.0, 0.0, 0.0, (double)md, o2);
    if (threadIdx.x == 0) {
        partial[4 * blockIdx.x] = o1[0]; partial[4 * blockIdx.x + 1] = o1[1]; partial[4 * blockIdx.x + 2] = o1[3]; partial[4 * blockIdx.x + 3] = o2[3];
    }
}
__global__ void __launch_bounds__(256) k_cover_final(const double *__restrict__ partial, int blocks, double cells, double *__restrict__ out) {
    double sl = 0.0, sd = 0.0, ml = 0.0, md = 0.0;
    for (int i = threadIdx.x; i < blocks; i += blockDim.x) {
        sl += partial[4 * i]; sd += partial[4 * i + 1]; ml = fmax(ml, partial[4 * i + 2]); md = fmax(md, partial[4 * i + 3]);
    }
    __shared__ double r1[4], r2[4];
    dw_stats_block_reduce(sl, sd, 0.0, ml, r1);
    __syncthreads();
    dw_stats_block_reduce(0.0, 0.0, 0.0, md, r2);
    if (threadIdx.x == 0) { out[0] = r1[0] / cells / 1000.0; out[1] = r1[1] / cells / 1000.0; out[2] = r1[3] / 1000.0; out[3] = r2[3] / 1000.0; }
}

__global__ void __launch_bounds__(256) k_to_f32(const double *__restrict__ x, size_t n, float *__restrict__ y) {
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) y[i] = (float)x[i];
}

// ---- device-side synthetic initial state (throughput ensembles; NOT numpy-stream compatible) -----------------------
// Same distribution as initialize_grid/initialize_agents (daisy_world_rl.py:285-302,173-179): per cell and species
// u0,u1 ~ U[0,1): cover = (u0 < proportion) * initial * u1; agents uniform on the grid with state 1.
__device__ __forceinline__ double dw_u01(uint64_t seed, uint64_t idx, uint32_t stream) {
    uint64_t z = seed + 0x9E3779B97F4A7C15ull * (idx * 4 + stream + 1);
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    z ^= z >> 31;
    return (double)(z >> 11) * (1.0 / 9007199254740992.0);
}

__global__ void __launch_bounds__(256) k_init_random(DevParams P, uint64_t seed, uint64_t world0, double prop_l, double prop_d,
                                                     double init_l, double init_d, double *cov, int32_t *agent_xy, double *agent_state) {
    const size_t NN = (size_t)P.N * P.N, total = (size_t)P.B * NN;
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        const size_t b = i / NN, c = i - b * NN;
        const uint64_t gidx = (world0 + b) * NN + c;
        const double d = dw_u01(seed, gidx, 0) < prop_d ? init_d * dw_u01(seed, gidx, 1) : 0.0;
        const double l = dw_u01(seed, gidx, 2) < prop_l ? init_l * dw_u01(seed, gidx, 3) : 0.0;
        cov[b * 2 * NN + c] = l;
        cov[b * 2 * NN + NN + c] = d;
    }
    const size_t na = (size_t)P.B * P.n_agents;
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < na; i += (size_t)gridDim.x * blockDim.x) {
        const uint64_t gidx = world0 * P.n_agents + i;
        agent_xy[2 * i] = (int)(dw_u01(seed ^ 0xA5A5A5A5ull, gidx, 0) * P.N);
        agent_xy[2 * i + 1] = (int)(dw_u01(seed ^ 0xA5A5A5A5ull, gidx, 1) * P.N);
        agent_state[i] = 1.0;
    }
}

// env.agent_indices (int64, any integers) -> wrapped int32 positions (the reference wraps with % dim, :208)
__global__ void __launch_bounds__(256) k_agent_indices_in(const long long *__restrict__ src, size_t count, int N, int32_t *__restrict__ xy) {
    const size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
    if (i >= count) return;
    long long v = src[i] % N;
    xy[i] = (int32_t)(v < 0 ? v + N : v);
}

// lean cover planes [B,2,N,N] -> 7-channel grid with channels 1,2 set and the rest zero (initialize_grid :304-312)
__global__ void __launch_bounds__(256) k_cov_to_grid(int B, size_t NN, const double *__restrict__ cov, double *__restrict__ grid) {
    const size_t total = (size_t)B * NN;
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        const size_t b = i / NN, c = i - b * NN;
        double *g = grid + b * 7 * NN + c;
        g[0] = 0; g[NN] = cov[b * 2 * NN + c]; g[2 * NN] = cov[b * 2 * NN + NN + c];
        g[3 * NN] = 0; g[4 * NN] = 0; g[5 * NN] = 0; g[6 * NN] = 0;
    }
}

// lattice -> fp64 covers (channels 1,2 only) : used when a fused run is followed by single steps
__global__ void __launch_bounds__(256) k_lattice_to_grid(int B, size_t NN, const uint32_t *__restrict__ lat, double *grid) {
    const size_t total = (size_t)B * NN;
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        const size_t b = i / NN, c = i - b * NN;
        const uint32_t k = lat[i];
        grid[b * 7 * NN + NN + c] = dw_milli(k & 0xffffu);
        grid[b * 7 * NN + 2 * NN + c] = dw_milli(k >> 16);
    }
}
