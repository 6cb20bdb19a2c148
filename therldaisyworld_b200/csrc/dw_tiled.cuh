// Single large world ("giant grid", BASELINE config 5): one toroidal N x N world too large for shared memory, held as a
// row band of `R` rows per rank (R = N on one GPU) on the packed 0.001 lattice, padded with ghost cells:
//
//     lat[(64 * tiles_y + 2) x pitch],  pitch = 64 * tiles_x + 8 words,  tiles_x = ceil(N / 64), tiles_y = ceil(R / 64)
//       row 0        ghost: the row above the band (toroidal wrap, or the neighbouring rank's last row)
//       rows 1..R    the band
//       row R + 1    ghost: the row below the band
//       word 3 / words 4..N+3 / word N+4 of a row: ghost of column N-1 / the N columns / ghost of column 0
//       words 0..2, words N+5.. and rows R+2.. are padding: never written, never read as cells (zero from the allocation)
// (N + 8 words and R + 2 rows when N and R are multiples of 64.)
//
// With the ghosts in place every 64x64 output tile needs one in-bounds 66-row x 72-word box of the source, which one
// elected thread fetches with a single TMA (cp.async.bulk.tensor.2d) into shared memory; 256 threads then run the same
// 4x4-cells-per-thread fast path as the ensemble kernel (dw_tile_core) and write their rows straight back to HBM.
// The padding keeps every box inside the allocation, so partial tiles (N or R not a multiple of 64) need no out-of-bounds
// fill: the masked instance of the kernel computes them whole and keeps only the cells inside the band.
// HBM traffic is 8 B per cell-update (4 B in, 4 B out); at the FP64-bound rate that is ~2 TB/s of the 6.5 TB/s measured,
// so this kernel is bound by the FP64 pipe like the SMEM-resident one.
//
// Agents of a giant world are many (thousands) and are replicated on every rank; the reference's sequential loop
// (daisy_world_rl.py:186-216) is resolved in parallel: decisions from the pre-move state, moves independent, and the
// grazers of one cell are ordered by an atomicMin claim (claim[(R+2) x N], INT_MAX when idle) on the agent index (the lowest index eats, later ones find the
// cell empty -- SURVEY App. B.8).  A rank applies the grazes that land in its band; grazes landing in its ghost rows only
// zero the ghost copy.  Per-agent food gains are summed over ranks by the caller (one all-reduce; exactly one rank
// contributes a non-zero term).
#pragma once
#include <cuda.h>

#include "dw_f32.cuh"
#include "dw_fused.cuh"

struct BandGeom {
    int N;       // global grid side
    int R;       // rows of this band
    int row0;    // global index of the band's first row
    int pitch;   // words (or doubles) per stored row
    int c0;      // index of column 0 inside a stored row (4 for the lattice, 0 for the fp64 planes of the first step)
};

// local stored-row indices (0..R+1) at which global row x is held by this band: interior and/or ghost copies
template <class F>
__device__ __forceinline__ void band_row_images(const BandGeom &G, int x, F f) {
    int rel = x - G.row0;
    rel = rel < 0 ? rel + G.N : rel;
    if (rel < G.R) f(rel + 1);
    if (rel == G.N - 1) f(0);
    if (rel == (G.R == G.N ? 0 : G.R)) f(G.R + 1);
}
template <class F>
__device__ __forceinline__ void band_col_images(const BandGeom &G, int y, F f) {
    f(G.c0 + y);
    if (G.c0 > 0) {
        if (y == G.N - 1) f(G.c0 - 1);
        if (y == 0) f(G.c0 + G.N);
    }
}
// interior stored row of global row x, or -1 if this band does not own it
__device__ __forceinline__ int band_owned_row(const BandGeom &G, int x) {
    int rel = x - G.row0;
    rel = rel < 0 ? rel + G.N : rel;
    return rel < G.R ? rel + 1 : -1;
}

// ---- cell accessors: packed lattice (steady state) or fp64 cover planes (the off-lattice state right after reset) ----
// load9: the covers of the 3x3 window around band row r (stored rows r .. r+2), column y
struct LatCells {
    uint32_t *p;
    __device__ __forceinline__ double food(size_t i) const { return dw_food(p[i]); }
    __device__ __forceinline__ void zero(size_t i) const { p[i] = 0u; }
    __device__ __forceinline__ void load9(const BandGeom &G, int r, int y, double (&l9)[9], double (&d9)[9]) const {
#pragma unroll
        for (int a = 0; a < 3; ++a)
#pragma unroll
            for (int c = 0; c < 3; ++c) {
                const uint32_t w = p[(size_t)(r + a) * G.pitch + G.c0 + y + c - 1];
                l9[a * 3 + c] = dw_milli(w & 0xffffu);
                d9[a * 3 + c] = dw_milli(w >> 16);
            }
    }
};
struct PlaneCells {
    double *l, *d;
    __device__ __forceinline__ double food(size_t i) const { return l[i] + d[i]; }
    __device__ __forceinline__ void zero(size_t i) const { l[i] = 0.0; d[i] = 0.0; }
    __device__ __forceinline__ void load9(const BandGeom &G, int r, int y, double (&l9)[9], double (&d9)[9]) const {
        const int ys[3] = {y == 0 ? G.N - 1 : y - 1, y, y == G.N - 1 ? 0 : y + 1};
#pragma unroll
        for (int a = 0; a < 3; ++a)
#pragma unroll
            for (int c = 0; c < 3; ++c) {
                const size_t k = (size_t)(r + a) * G.pitch + ys[c];
                l9[a * 3 + c] = l[k];
                d9[a * 3 + c] = d[k];
            }
    }
};
// column index with toroidal wrap for planes without column ghosts
__device__ __forceinline__ int band_col(const BandGeom &G, int y) {
    if (G.c0 > 0) return G.c0 + y;                       // ghosts at c0-1 and c0+N make y = -1 and y = N valid
    return y < 0 ? y + G.N : (y >= G.N ? y - G.N : y);
}

// ---- peer-memory mode (one process per GPU, P2P stores over NVLink / NVSwitch, no NCCL on the step path) --------------
// Every rank maps every other rank's exchange vector, flag array and lattice buffers (CUDA IPC).  The owner of an agent /
// the winner of a graze stores its result straight into ALL ranks' exchange vectors (exactly one writer per entry, so
// nothing has to be reduced), a band pushes its edge rows into the neighbours' ghost rows, and ranks meet at flag
// barriers (k_peer_barrier) instead of collectives.
#define DWT_MAX_RANKS 8
struct PeerTable {
    double *exch[DWT_MAX_RANKS];           // [gain1 | gain0 | act], n doubles each
    unsigned int *flags[DWT_MAX_RANKS];    // [DWT_MAX_RANKS] barrier epochs, slot r written by rank r
    int rank, R, on;                       // on == 0: single-process / NCCL mode (local stores only)
    int pad_;
    long long timeout_clocks;              // bound of a barrier spin (default 8e9 ~ 4 s; DW_PEER_TIMEOUT_MS); <= 0: default
};

// All ranks meet here: every prior write of this rank (to its own or to peer memory) is visible to a peer that has seen
// the flag. Spins are bounded (~seconds) so that a missing peer produces an error flag instead of a hung GPU.
__device__ __forceinline__ void dw_peer_barrier_body(const PeerTable &PT, unsigned int epoch, unsigned int *timed_out, int p) {
    if (p >= PT.R) return;
    __threadfence_system();
    asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(PT.flags[p] + PT.rank), "r"(epoch) : "memory");
    const unsigned int *mine = PT.flags[PT.rank] + p;
    const long long t0 = clock64(), limit = PT.timeout_clocks > 0 ? PT.timeout_clocks : 8000000000ll;
    for (;;) {
        unsigned int v;
        asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(mine) : "memory");
        if ((int)(v - epoch) >= 0) break;
        if (clock64() - t0 > limit) { *timed_out = 1u; break; }
        __nanosleep(100);
    }
    __threadfence_system();
}
__global__ void k_peer_barrier(PeerTable PT, unsigned int epoch, unsigned int *timed_out) {
    dw_peer_barrier_body(PT, epoch, timed_out, threadIdx.x);
}
// Tail of a multi-block kernel that ends in a barrier: every block calls this after its own (peer) stores; the block
// that arrives last at the ticket counter runs the barrier, so the flag is raised only after ALL blocks' stores.
__device__ __forceinline__ void dw_last_block_barrier(const PeerTable &PT, unsigned int epoch, unsigned int *timed_out, unsigned int *ticket) {
    __shared__ int s_last;
    __threadfence_system();
    __syncthreads();
    if (threadIdx.x == 0) {
        const unsigned int t = atomicAdd(ticket, 1u);
        s_last = (t == gridDim.x - 1);
        if (s_last) *ticket = 0u;                        // re-armed for the next launch (stream order)
        __threadfence();
    }
    __syncthreads();
    if (s_last) dw_peer_barrier_body(PT, epoch, timed_out, threadIdx.x);
}

// a band's first / last stored row (ghost columns included) -> the neighbours' ghost rows
// ... and then the closing barrier of the step, raised by the block that finishes last.
__global__ void __launch_bounds__(256) k_band_push_halo(const uint32_t *__restrict__ lat, int R, int pitch, uint32_t *up_ghost_bottom,
                                                        uint32_t *down_ghost_top, PeerTable PT, unsigned int epoch, unsigned int *timed_out,
                                                        unsigned int *ticket) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c < pitch) {
        up_ghost_bottom[c] = lat[(size_t)pitch + c];
        down_ghost_top[c] = lat[(size_t)R * pitch + c];
    }
    dw_last_block_barrier(PT, epoch, timed_out, ticket);
}

// ---- agents --------------------------------------------------------------------------------------------------------
template <class Cells>
__device__ __forceinline__ void k_band_decide_one(const BandGeom &G, const Cells &C, const int32_t *__restrict__ xy, int n, int policy,
                                                  const int8_t *__restrict__ replay, uint64_t seed, uint32_t step, const PeerTable &PT,
                                                  double *__restrict__ act, int i) {
    const int x = xy[2 * i], y = xy[2 * i + 1];
    const int lr = band_owned_row(G, x);
    double out = 0.0;
    if (policy == DW_POLICY_REPLAY || policy == DW_POLICY_NONE || policy == DW_POLICY_RANDOM) {
        // world-independent: every rank computes the same action for every agent (no exchange needed)
        int a = 0;
        if (policy == DW_POLICY_REPLAY) a = replay[i];
        else if (policy == DW_POLICY_RANDOM) a = (int)(dw_hash_rng(seed, 0u, (uint32_t)i, step) % 9u);
        out = (double)(a + 1);
    } else if (lr >= 0) {
        const size_t rowm = (size_t)(lr - 1) * G.pitch, row = (size_t)lr * G.pitch, rowp = (size_t)(lr + 1) * G.pitch;
        const double food[4] = {C.food(row + band_col(G, y - 1)), C.food(rowm + band_col(G, y)), C.food(rowp + band_col(G, y)),
                                C.food(row + band_col(G, y + 1))};
        out = (double)(dw_greedy_pick(food, policy == DW_POLICY_GREEDY) + 1);
        if (PT.on) {                                     // owner publishes the decision to every rank (act = exch + 2n)
            for (int p = 0; p < PT.R; ++p) PT.exch[p][2 * (size_t)n + i] = out;
            return;
        }
    } else if (PT.on) return;                            // peer-memory mode: the owner rank writes this entry
    act[i] = out;
}

// Phase 1: the owner band of each agent decides its action from the pre-move state. act[i] = action + 1 for owned
// agents, 0 otherwise (the caller sums act over ranks). Policies that do not look at the world (replay, none, random)
// fill every entry on every rank and need no exchange.
template <class Cells>
__global__ void __launch_bounds__(256) k_band_decide(BandGeom G, Cells C, const int32_t *__restrict__ xy, int n, int policy,
                                                     const int8_t *__restrict__ replay, uint64_t seed, uint32_t step, PeerTable PT,
                                                     double *__restrict__ act, unsigned int epoch, unsigned int *timed_out,
                                                     unsigned int *ticket) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) k_band_decide_one<Cells>(G, C, xy, n, policy, replay, seed, step, PT, act, i);
    if (epoch) dw_last_block_barrier(PT, epoch, timed_out, ticket);     // peer-memory mode, world-reading policies
}

// Phase 2 of agent i with state s at (x, y) (replicated on every rank): pay agent_gamma, move if still alive, and file the
// graze claim of a cell this band owns. x, y become the new position; gz[i] = 1 (returned) if the agent grazes this step.
__device__ __forceinline__ uint8_t dwt_move_claim_agent(const BandGeom &G, double agent_gamma, int32_t *xy, double *st, double s, int &x,
                                                        int &y, const double *__restrict__ act, int *claim, uint8_t *gz, int i) {
    const int a = (int)act[i] - 1;
    s = s - agent_gamma;
    st[i] = s;
    uint8_t g = 0;
    if (s > 0.0) {
        if (a != 8) {
            const int d = (a & 2) ? 1 : -1;              // a & 3 = 0: y-1, 1: x-1, 2: x+1, 3: y+1
            if (((a + 1) & 2) == 0) { y += d; y = y < 0 ? y + G.N : (y >= G.N ? y - G.N : y); }
            else { x += d; x = x < 0 ? x + G.N : (x >= G.N ? x - G.N : x); }
            xy[2 * i] = x;
            xy[2 * i + 1] = y;
        }
        if (a > 4) {
            g = 1;
            const int lr = band_owned_row(G, x);
            if (lr >= 0) atomicMin(claim + (size_t)lr * G.N + y, i);
        }
    }
    gz[i] = g;
    return g;
}

// Phase 3 of grazing agent i at (x, y): the claim winner of an owned cell eats it and clears every stored copy; a graze that
// lands in a ghost row only clears the ghost copy (the owner rank does the eating). claim_at(k) loads claim[k] the way the
// caller needs it. The winner sets won and got = the food it eats on THIS rank; both are left alone otherwise.
template <class Cells, class ClaimAt>
__device__ __forceinline__ void dwt_graze_agent(const BandGeom &G, const Cells &C, int x, int y, ClaimAt claim_at, int i, double &got,
                                                bool &won) {
    const int lr = band_owned_row(G, x);
    bool clear = true;
    if (lr >= 0) {
        if (claim_at((size_t)lr * G.N + y) == i) { got = C.food((size_t)lr * G.pitch + G.c0 + y); won = true; }
        else clear = false;                              // a lower-index agent eats here; it also does the clearing
    }
    if (clear)
        band_row_images(G, x, [&](int r) { band_col_images(G, y, [&](int cc) { C.zero((size_t)r * G.pitch + cc); }); });
}

// Phase 4 of agent i with state s at (x, y), the cell it grazed (replicated, after the gains were summed over ranks):
// state += gain if it grazed, its claim back to "idle", clip, lifespan counter. Returns the new state.
// zero_gain: peer-memory mode, where only the winners write the gain vector, so it is re-armed here.
__device__ __forceinline__ double dwt_finish_agent(const BandGeom &G, int x, int y, double s, double *gain, bool zero_gain,
                                                   const uint8_t *gz, int *claim, int64_t *agents_done_at, int i) {
    const double g = gain[i];
    if (zero_gain) gain[i] = 0.0;
    if (gz[i]) {
        s = s + g;
        const int lr = band_owned_row(G, x);
        if (lr >= 0) claim[(size_t)lr * G.N + y] = 0x7fffffff;
    }
    s = dw_clip01(s);
    agents_done_at[i] += (s < 0.1) ? 0 : 1;
    return s;
}

// Phase 2 (replicated on every rank), in peer-memory mode preceded by phase 4 of the previous step (do_finish: its gains
// are complete since its closing barrier). The two steps use different claim arrays there (step parity), so returning
// step j-1's claims to "idle" cannot collide with step j's atomicMin on the same cell. Phase-by-phase and NCCL mode have
// one claim array and finish with k_band_finish instead (do_finish = 0): merged, the return of step j-1's claims would race
// with step j's claims in the same launch.
__global__ void __launch_bounds__(256) k_band_move_claim(BandGeom G, double agent_gamma, int32_t *xy, double *st, int n,
                                                         const double *__restrict__ act, int *claim, uint8_t *gz, int do_finish,
                                                         double *gain_prev, int *claim_prev, int64_t *agents_done_at) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    double s = st[i];
    int x = xy[2 * i], y = xy[2 * i + 1];
    if (do_finish) s = dwt_finish_agent(G, x, y, s, gain_prev, true, gz, claim_prev, agents_done_at, i);
    dwt_move_claim_agent(G, agent_gamma, xy, st, s, x, y, act, claim, gz, i);
}

// Phase 3. gain[i] = food eaten by agent i on THIS rank (0 elsewhere); in peer-memory mode the winner publishes it to every
// rank instead, at exch + gain_off.
template <class Cells>
__global__ void __launch_bounds__(256) k_band_graze(BandGeom G, Cells C, const int32_t *__restrict__ xy, int n,
                                                    const uint8_t *__restrict__ gz, const int *__restrict__ claim, double *__restrict__ gain,
                                                    PeerTable PT, int gain_off) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    double got = 0.0;
    bool won = false;
    if (gz[i]) dwt_graze_agent(G, C, xy[2 * i], xy[2 * i + 1], [&](size_t k) { return claim[k]; }, i, got, won);
    if (PT.on) {                                         // the vectors were zeroed by the finish of the step that last used them
        if (won) for (int p = 0; p < PT.R; ++p) PT.exch[p][(size_t)gain_off + i] = got;
        return;
    }
    gain[i] = got;
}

// Peer-memory mode, lattice state: k_band_move_claim and k_band_graze in ONE launch. The graze needs every claim of the step
// filed, so the two halves are separated by a grid-wide barrier (monotonic counter in global memory: the host passes the
// value it has after this launch's blocks have all arrived). Only launched when the grid is at most one block per SM
// (n <= 256 * SMs), so every block is resident and the spin cannot deadlock. Saves one kernel boundary per step on the
// critical path of a step (the two agent kernels are what is left there besides the stencil).
__global__ void __launch_bounds__(256) k_band_fmc_graze(BandGeom G, double agent_gamma, int32_t *xy, double *st, int n,
                                                        const double *__restrict__ act, int *claim_new, uint8_t *gz, int do_finish,
                                                        double *gain_prev, int *claim_prev, int64_t *agents_done_at, LatCells C,
                                                        PeerTable PT, int gain_off, unsigned int *bar, unsigned int target) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    const bool active = i < n;
    int x = 0, y = 0;
    uint8_t g = 0;
    if (active) {
        double s = st[i];
        x = xy[2 * i]; y = xy[2 * i + 1];
        if (do_finish) s = dwt_finish_agent(G, x, y, s, gain_prev, true, gz, claim_prev, agents_done_at, i);
        g = dwt_move_claim_agent(G, agent_gamma, xy, st, s, x, y, act, claim_new, gz, i);
    }
    // every claim of the step is filed once all blocks have passed here
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence();
        atomicAdd(bar, 1u);
        while ((int)(*(volatile unsigned int *)bar - target) < 0) { }
        __threadfence();
    }
    __syncthreads();
    if (!active || !g) return;
    double got = 0.0;
    bool won = false;                                    // claims of other blocks of this launch: read past L1
    dwt_graze_agent(G, C, x, y, [&](size_t k) { return __ldcg(claim_new + k); }, i, got, won);
    if (won) for (int p = 0; p < PT.R; ++p) PT.exch[p][(size_t)gain_off + i] = got;
}

// Phase 4 (replicated, after the gains were summed over ranks) of phase-by-phase and NCCL mode, and of the last step in
// peer-memory mode (dwt_flush_p2p).
__global__ void __launch_bounds__(256) k_band_finish(BandGeom G, const int32_t *__restrict__ xy, int *claim, double *st, int n,
                                                     double *gain, int zero_gain, const uint8_t *__restrict__ gz, int64_t *agents_done_at) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    st[i] = dwt_finish_agent(G, xy[2 * i], xy[2 * i + 1], st[i], gain, zero_gain, gz, claim, agents_done_at, i);
}

// ---- ghost maintenance ---------------------------------------------------------------------------------------------
// The stencil kernels write the ghost COLUMNS of the rows they produce, so a ghost ROW is a copy of a whole stored row
// (pitch words): from the band's own edge rows on a single-rank torus, from the neighbours otherwise.
__global__ void __launch_bounds__(256) k_band_ghost_rows_wrap(BandGeom G, uint32_t *lat) {   // single-rank torus: R == N
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= G.pitch) return;
    lat[c] = lat[(size_t)G.R * G.pitch + c];
    lat[(size_t)(G.R + 1) * G.pitch + c] = lat[(size_t)G.pitch + c];
}
// Ghost COLUMNS of stored rows 0 .. rows - 1 from the row's own columns (toroidal): word c0 - 1 <- column N - 1, word c0 + N
// <- column 0. dwt_restore_state uploads the R + 2 rows of a snapshot without them; the padding words stay untouched.
__global__ void __launch_bounds__(256) k_band_ghost_cols(BandGeom G, uint32_t *lat, int rows) {
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= rows) return;
    uint32_t *row = lat + (size_t)r * G.pitch;
    row[G.c0 - 1] = row[G.c0 + G.N - 1];
    row[G.c0 + G.N] = row[G.c0];
}

// ---- first step: literal forward from the off-lattice fp64 cover planes [(R+2) x N] onto the padded lattice ---------
// SERIES: also adds {sum sqrt(g)*T, sum milli-light, sum milli-dark} of the band's cells to series[0..2] (see k_tiled_step)
template <bool SERIES = false>
__global__ void __launch_bounds__(256) k_band_first_step(DevParams P, double SL, BandGeom Gp, PlaneCells pre, BandGeom Gl,
                                                         uint32_t *__restrict__ lat_out, int *stepmax, double sqrt_g = 0.0,
                                                         double *series = nullptr) {
    const size_t total = (size_t)Gp.R * Gp.N;
    uint32_t mx = 0;
    double ser[3] = {0.0, 0.0, 0.0};     // series mode; the cover sums are integers below 2^53, so exact in fp64
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        const int r = (int)(i / Gp.N), y = (int)(i - (size_t)r * Gp.N);
        double l9[9], d9[9];
        pre.load9(Gp, r, y, l9, d9);
        const LitCell o = dw_literal_cell(P, SL, l9, d9);
        const uint32_t q = dw_pack((int)rint(o.nl * 1000.0), (int)rint(o.nd * 1000.0));
        uint32_t *orow = lat_out + (size_t)(r + 1) * Gl.pitch;
        orow[Gl.c0 + y] = q;
        if (y == 0) orow[Gl.c0 + Gl.N] = q;              // ghost columns of the produced row
        if (y == Gl.N - 1) orow[Gl.c0 - 1] = q;
        mx = __vmaxu2(mx, q);
        if (SERIES) {
            ser[0] += sqrt_g * o.T;
            ser[1] += (double)(q & 0xffffu);
            ser[2] += (double)(q >> 16);
        }
    }
    const unsigned ml = __reduce_max_sync(0xffffffffu, mx & 0xffffu), md = __reduce_max_sync(0xffffffffu, mx >> 16);
    if ((threadIdx.x & 31) == 0) { atomicMax(stepmax, (int)ml); atomicMax(stepmax + 1, (int)md); }
    if (SERIES) {
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            double v = ser[c];
            for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
            if ((threadIdx.x & 31) == 0) atomicAdd(series + c, v);
        }
    }
}

// ---- steady state: one stencil step of the band, 64x64 tiles, TMA-staged halo tile ---------------------------------
#define DWT_TILE 64
#define DWT_TILE_ROWS (DWT_TILE + 2)
#define DWT_TILE_PITCH (DWT_TILE + 8)
#define DWT_TILE_BYTES (DWT_TILE_ROWS * DWT_TILE_PITCH * 4)

struct TiledArgs {
    DevParams P;
    FastCoef F;
    StepCoef C;
    uint32_t *out;          // padded lattice written by this step
    int pitch;
    int tiles_x;            // tiles per row
    int tr_first, tr_skip_lo, tr_skip_hi;   // tile rows of this launch: blockIdx -> tr, skipping [tr_skip_lo, tr_skip_hi)
    int N;
    int *stepmax;           // [2] per-species max of the new band (atomicMax)
    unsigned int *slow_count;
};

__device__ __forceinline__ uint32_t dwt_smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

struct RowsTile72 {
    const uint32_t *t;      // first cell of the thread's first row inside the staged tile
    __device__ __forceinline__ Row6 load(int k) const {
        const uint32_t *p = t + k * DWT_TILE_PITCH;
        return dw_make_row(*reinterpret_cast<const uint4 *>(p), p[-1], p[4]);
    }
};
struct StoreGlobal {
    static constexpr bool kMasks = false;
    uint32_t *o;            // first cell of the thread's first output row
    int pitch;
    __device__ __forceinline__ void operator()(int i, uint32_t (&q)[4]) const {
        *reinterpret_cast<uint4 *>(o + (size_t)i * pitch) = make_uint4(q[0], q[1], q[2], q[3]);
    }
};
// series mode: StoreGlobal that also sums the packed cells it stores. Each half of a packed cell is at most 1000, so the
// 16 cells of a thread's 4x4 tile sum to at most 16000 per half and the halves cannot carry into each other.
struct StoreGlobalSum {
    static constexpr bool kMasks = false;
    uint32_t *o;
    int pitch;
    uint32_t *sum;
    __device__ __forceinline__ void operator()(int i, uint32_t (&q)[4]) const {
        *reinterpret_cast<uint4 *>(o + (size_t)i * pitch) = make_uint4(q[0], q[1], q[2], q[3]);
        *sum += (q[0] + q[1]) + (q[2] + q[3]);
    }
};
// Partial tiles: only the thread's cells inside the band (the first `rows` rows and `cols` columns of its 4x4, either may be
// <= 0 or > 4) are stored; the others are zeroed in q, so that they count neither in the maxima nor in the cover sum.
template <bool SUM>
struct StoreGlobalMasked {
    static constexpr bool kMasks = true;
    uint32_t *o;
    int pitch, rows, cols;
    uint32_t *sum;          // SUM: packed sum of the stored cells (see StoreGlobalSum)
    __device__ __forceinline__ int cells(int i) const { return i < rows ? min(max(cols, 0), 4) : 0; }
    __device__ __forceinline__ void operator()(int i, uint32_t (&q)[4]) const {
        if (i >= rows) { q[0] = 0u; q[1] = 0u; q[2] = 0u; q[3] = 0u; return; }     // below the band: ghost row or padding
        uint32_t *d = o + (size_t)i * pitch;
        if (cols >= 4) {
            *reinterpret_cast<uint4 *>(d) = make_uint4(q[0], q[1], q[2], q[3]);
        } else {                                         // right of column N-1: the ghost of column 0, then padding
#pragma unroll
            for (int t = 0; t < 4; ++t) {
                if (t < cols) d[t] = q[t];
                else q[t] = 0u;
            }
        }
        if (SUM) *sum += (q[0] + q[1]) + (q[2] + q[3]);
    }
};

// rare path, warp-cooperative: for every lane whose 4x4 tile hit the tie filter, lanes 0..15 re-evaluate one cell of that
// tile each from the staged tile; cells on a rounding tie are recomputed in literal order and patched in the output.
// tile_off / out_off: each lane's offsets of its first cell inside the staged tile / the output lattice.
// MASK (partial tiles): rows / cols as in StoreGlobalMasked; cells outside the band are neither fixed up nor counted.
template <bool MASK>
__device__ __forceinline__ uint32_t dwt_fix_tiles(const TiledArgs *A, const uint32_t *tile, unsigned flagged, uint32_t mx, int tile_off,
                                                  long long out_off, int lane, int rows, int cols) {
    uint32_t extra = 0;
    bool mine = false;
    __syncwarp();
    while (flagged) {
        const int L = __ffs(flagged) - 1;
        flagged &= flagged - 1;
        const int toff = __shfl_sync(0xffffffffu, tile_off, L);
        const long long ooff = __shfl_sync(0xffffffffu, out_off, L);
        bool cell = lane < 16;
        if (MASK) {
            const int lr = __shfl_sync(0xffffffffu, rows, L), lc = __shfl_sync(0xffffffffu, cols, L);
            cell = cell && (lane >> 2) < lr && (lane & 3) < lc;
        }
        if (lane == L) mine = true;
        if (cell) {
            const uint32_t *p = tile + toff + (lane >> 2) * DWT_TILE_PITCH + (lane & 3);
            const uint32_t *q0 = p - DWT_TILE_PITCH, *q2 = p + DWT_TILE_PITCH;
            const uint32_t E = p[-1] + p[1] + q0[0] + q2[0];
            const uint32_t S8 = E + q0[-1] + q0[1] + q2[-1] + q2[1];
            unsigned tiemin = 0xffffffffu;
            uint32_t v = dw_fast_cell(A->F, A->C, p[0], E, S8, &tiemin);
            if (tiemin < A->F.tie_thresh) {
                double l9[9], d9[9];
#pragma unroll
                for (int a = 0; a < 3; ++a)
#pragma unroll
                    for (int c = 0; c < 3; ++c) {
                        const uint32_t w = p[(a - 1) * DWT_TILE_PITCH + (c - 1)];
                        l9[a * 3 + c] = dw_milli(w & 0xffffu);
                        d9[a * 3 + c] = dw_milli(w >> 16);
                    }
                const LitCell lc = dw_literal_cell(A->P, A->C.SL, l9, d9);
                v = dw_pack((int)rint(lc.nl * 1000.0), (int)rint(lc.nd * 1000.0));
                A->out[ooff + (long long)(lane >> 2) * A->pitch + (lane & 3)] = v;
                if (A->slow_count) atomicAdd(A->slow_count, 1u);
            }
            extra = __vmaxu2(extra, v);
        }
    }
    __syncwarp();                                        // patches (made by helper lanes) before the owners re-read their cells
    return __vmaxu2(mine ? 0u : mx, extra);
}
// One copy per k_tiled_step instantiation (SERIES is otherwise unused): with a single caller the compiler propagates the
// address of that kernel's shared tile into it, which the default kernel's code and shared-memory layout depend on.
template <bool SERIES>
__device__ __noinline__ uint32_t dwt_fix_warp(const TiledArgs *A, const uint32_t *tile, unsigned flagged, uint32_t mx, int tile_off,
                                              long long out_off, int lane) {
    return dwt_fix_tiles<false>(A, tile, flagged, mx, tile_off, out_off, lane, 0, 0);
}
template <bool SERIES>
__device__ __noinline__ uint32_t dwt_fix_warp_masked(const TiledArgs *A, const uint32_t *tile, unsigned flagged, uint32_t mx, int tile_off,
                                                     long long out_off, int lane, int rows, int cols) {
    return dwt_fix_tiles<true>(A, tile, flagged, mx, tile_off, out_off, lane, rows, cols);
}

__device__ __forceinline__ void dwt_issue_tile(const CUtensorMap *tmap, const TiledArgs &A, int t, uint32_t smem_tile, uint32_t bar_a) {
    const int tc = t % A.tiles_x;
    int tr = A.tr_first + t / A.tiles_x;
    if (tr >= A.tr_skip_lo) tr += A.tr_skip_hi - A.tr_skip_lo;
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar_a), "r"((uint32_t)DWT_TILE_BYTES) : "memory");
    // box origin (word, row) of the padded lattice: tile columns 64*tc-4 .. 64*tc+67, band rows 64*tr-1 .. 64*tr+64
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
                 ::"r"(smem_tile), "l"(tmap), "r"(bar_a), "r"(tc * DWT_TILE), "r"(tr * DWT_TILE)
                 : "memory");
}

// One tile per CTA (gridDim.x = number of tiles, 19 KB of shared memory). A grid of fewer CTAs also works: a CTA then walks
// the tiles blockIdx.x, blockIdx.x + gridDim.x, ... and loads the next one once the current one is computed.
// SERIES: the step also adds the sums of its produced cells to series[0..2], one atomicAdd per column and CTA:
// {sqrt(g)*T of the forward (unrounded, from the staged pre-state), new milli-light, new milli-dark}. `series` is the last
// parameter (not a member of TiledArgs), so that every parameter offset of the default kernel stays where it was.
// MASK: the instance for a side N or a band height `rows` that is not a multiple of 64. The cells of the partial tiles that
// lie outside the band are computed from padding and dropped: not stored (the last tile row would otherwise overwrite the
// ghost row below the band), not fixed up, and counted neither in the maxima nor in the series sums. The ghost column of
// N-1 is copied by the thread that holds column N-1. `rows` follows `series` for the same reason as `series`.
template <bool SERIES = false, bool MASK = false>
__global__ void __launch_bounds__(256, 4) k_tiled_step(const __grid_constant__ CUtensorMap tmap, const __grid_constant__ TiledArgs A,
                                                       int n_tiles, double *series = nullptr, int rows = 0) {
    constexpr int kTileWords = ((DWT_TILE_BYTES + 127) / 128) * 32;       // a TMA destination must be 128-byte aligned: 19008 -> 19072 B
    __shared__ __align__(128) uint32_t tile[kTileWords];
    __shared__ __align__(8) unsigned long long bar;
    __shared__ int smax[2];
    const int tid = threadIdx.x, lane = tid & 31;
    const int tx = tid & 15, r0 = (tid >> 4) * 4;
    const uint32_t bar_a = dwt_smem_u32(&bar), tile_a = dwt_smem_u32(tile);
    int t = blockIdx.x;
    if (tid == 0) {
        smax[0] = 0; smax[1] = 0;
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(bar_a));
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        if (t < n_tiles) dwt_issue_tile(&tmap, A, t, tile_a, bar_a);
    }
    __syncthreads();                                     // barrier initialised (and armed) before anyone polls
    const int tile_off = (1 + r0) * DWT_TILE_PITCH + 4 + 4 * tx;
    uint32_t mx_all = 0;
    double tsum = 0.0;                                   // series mode: sqrt(g)*T, light and dark milli-covers of the thread's cells
    uint32_t cl = 0, cd = 0;
    for (int k = 0; t < n_tiles; ++k, t += gridDim.x) {
        {
            const uint32_t parity = (uint32_t)k & 1u;
            uint32_t ok = 0;
            while (!ok)
                asm volatile("{ .reg .pred p; mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2; selp.u32 %0, 1, 0, p; }"
                             : "=r"(ok) : "r"(bar_a), "r"(parity) : "memory");
        }
        const int tc = t % A.tiles_x;
        int tr = A.tr_first + t / A.tiles_x;
        if (tr >= A.tr_skip_lo) tr += A.tr_skip_hi - A.tr_skip_lo;
        const long long out_off = (long long)(tr * DWT_TILE + 1 + r0) * A.pitch + 4 + tc * DWT_TILE + 4 * tx;
        unsigned tiemin = 0xffffffffu;
        uint32_t mx, cov = 0;
        // MASK: rows / columns of the thread's 4x4 cells inside the band
        const int vr = MASK ? rows - (tr * DWT_TILE + r0) : 4, vc = MASK ? A.N - (tc * DWT_TILE + 4 * tx) : 4;
        if constexpr (MASK)
            mx = dw_tile_core<RowsTile72, StoreGlobalMasked<SERIES>, SERIES>(
                A.F, A.C, RowsTile72{tile + tile_off}, StoreGlobalMasked<SERIES>{A.out + out_off, A.pitch, vr, vc, &cov}, &tiemin, &tsum);
        else if constexpr (SERIES)
            mx = dw_tile_core<RowsTile72, StoreGlobalSum, true>(A.F, A.C, RowsTile72{tile + tile_off}, StoreGlobalSum{A.out + out_off, A.pitch, &cov},
                                                                &tiemin, &tsum);
        else
            mx = dw_tile_core(A.F, A.C, RowsTile72{tile + tile_off}, StoreGlobal{A.out + out_off, A.pitch}, &tiemin);
        const unsigned flagged = __ballot_sync(0xffffffffu, tiemin < A.F.tie_thresh);
        if (flagged) {
            if constexpr (MASK) mx = dwt_fix_warp_masked<SERIES>(&A, tile, flagged, mx, tile_off, out_off, lane, vr, vc);
            else mx = dwt_fix_warp<SERIES>(&A, tile, flagged, mx, tile_off, out_off, lane);
            if constexpr (SERIES) {
                if ((flagged >> lane) & 1u) {            // literal fix-ups were patched into this lane's cells: sum them again
                    const uint32_t *o = A.out + out_off;
                    cov = 0;
                    if constexpr (MASK) {
#pragma unroll
                        for (int i = 0; i < 4; ++i)
#pragma unroll
                            for (int c = 0; c < 4; ++c)
                                if (i < vr && c < vc) cov += o[(size_t)i * A.pitch + c];
                    } else {
#pragma unroll
                        for (int i = 0; i < 4; ++i) {
                            const uint4 v = *reinterpret_cast<const uint4 *>(o + (size_t)i * A.pitch);
                            cov += (v.x + v.y) + (v.z + v.w);
                        }
                    }
                }
            }
        }
        if constexpr (SERIES) { cl += cov & 0xffffu; cd += cov >> 16; }
        // ghost columns of the produced rows: the two threads of a row group that hold column 0 / N-1 copy their (final) cells
        if constexpr (MASK) {
            if (tx == 0 && tc == 0) {
                uint32_t *o = A.out + out_off;
#pragma unroll
                for (int i = 0; i < 4; ++i)
                    if (i < vr) o[(size_t)i * A.pitch + A.N] = o[(size_t)i * A.pitch];
            }
            if (tx == ((A.N - 1) & (DWT_TILE - 1)) >> 2 && tc == A.tiles_x - 1) {
                uint32_t *o = A.out + out_off + ((A.N - 1) & 3);
#pragma unroll
                for (int i = 0; i < 4; ++i)
                    if (i < vr) o[(size_t)i * A.pitch - A.N] = o[(size_t)i * A.pitch];
            }
        } else if (tx == 0 && tc == 0) {
            uint32_t *o = A.out + out_off;
#pragma unroll
            for (int i = 0; i < 4; ++i) o[(size_t)i * A.pitch + A.N] = o[(size_t)i * A.pitch];
        } else if (tx == 15 && tc == A.tiles_x - 1) {
            uint32_t *o = A.out + out_off + 3;
#pragma unroll
            for (int i = 0; i < 4; ++i) o[(size_t)i * A.pitch - A.N] = o[(size_t)i * A.pitch];
        }
        mx_all = __vmaxu2(mx_all, mx);
        __syncthreads();                                 // every read of the tile is done before the next iteration refills it
        if (tid == 0 && t + (int)gridDim.x < n_tiles) dwt_issue_tile(&tmap, A, t + gridDim.x, tile_a, bar_a);
    }
    const unsigned ml = __reduce_max_sync(0xffffffffu, mx_all & 0xffffu), md = __reduce_max_sync(0xffffffffu, mx_all >> 16);
    if (lane == 0) { atomicMax(&smax[0], (int)ml); atomicMax(&smax[1], (int)md); }
    if constexpr (SERIES) {
        // per warp, then per CTA (fixed order), then one global add per column: 3 same-address atomics per CTA and step
        __shared__ double s_ser[256 / 32][3];
        for (int o = 16; o > 0; o >>= 1) tsum += __shfl_xor_sync(0xffffffffu, tsum, o);
        cl = __reduce_add_sync(0xffffffffu, cl);
        cd = __reduce_add_sync(0xffffffffu, cd);
        if (lane == 0) { s_ser[tid >> 5][0] = tsum; s_ser[tid >> 5][1] = (double)cl; s_ser[tid >> 5][2] = (double)cd; }
        __syncthreads();
        if (tid < 3) {
            double v = 0.0;
#pragma unroll
            for (int w = 0; w < 256 / 32; ++w) v += s_ser[w][tid];
            atomicAdd(series + tid, v);
        }
    }
    __syncthreads();
    if (tid == 0) {
        if (smax[0] > 0) atomicMax(A.stepmax, smax[0]);
        if (smax[1] > 0) atomicMax(A.stepmax + 1, smax[1]);
    }
}

// ---- look-ahead decisions (peer-memory mode) ---------------------------------------------------------------------------
// The greedy decision of step j+1 reads the four neighbours of the agent in the lattice step j PRODUCES -- 4 cells per
// agent out of N x R. Waiting for the whole stencil to finish puts decide + its barrier on the critical path of every
// step; instead the owner band re-evaluates just those cells itself from the step's INPUT lattice (post-graze `lat_old`,
// same fast path + literal tie fix-up as k_tiled_step, hence the same values) while the interior tiles are still being
// computed on the main stream. Neighbours that sit in a ghost row belong to the neighbouring band: those come from the
// NEW ghost rows, which the halo push + barrier that precede this kernel on the side stream have delivered.
struct LookArgs {
    DevParams P;
    FastCoef F;
    StepCoef C;
};
__device__ __forceinline__ uint32_t dwt_new_cell(const LookArgs &A, const BandGeom &G, const uint32_t *__restrict__ lat_old,
                                                 const uint32_t *__restrict__ lat_new, int r, int yc) {
    if (r == 0 || r == G.R + 1) return lat_new[(size_t)r * G.pitch + G.c0 + yc];
    const uint32_t *p = lat_old + (size_t)r * G.pitch + G.c0 + yc;
    const uint32_t *q0 = p - G.pitch, *q2 = p + G.pitch;
    const uint32_t E = p[-1] + p[1] + q0[0] + q2[0];
    const uint32_t S8 = E + q0[-1] + q0[1] + q2[-1] + q2[1];
    unsigned tiemin = 0xffffffffu;
    uint32_t v = dw_fast_cell(A.F, A.C, p[0], E, S8, &tiemin);
    if (tiemin < A.F.tie_thresh) {
        double l9[9], d9[9];
#pragma unroll
        for (int a = 0; a < 3; ++a)
#pragma unroll
            for (int c = 0; c < 3; ++c) {
                const uint32_t w = p[(a - 1) * G.pitch + (c - 1)];
                l9[a * 3 + c] = dw_milli(w & 0xffffu);
                d9[a * 3 + c] = dw_milli(w >> 16);
            }
        const LitCell lc = dw_literal_cell(A.P, A.C.SL, l9, d9);
        v = dw_pack((int)rint(lc.nl * 1000.0), (int)rint(lc.nd * 1000.0));
    }
    return v;
}
__global__ void __launch_bounds__(256) k_band_lookahead_decide(BandGeom G, const uint32_t *__restrict__ lat_old,
                                                               const uint32_t *__restrict__ lat_new, const int32_t *__restrict__ xy, int n,
                                                               int policy, PeerTable PT, const __grid_constant__ LookArgs A,
                                                               unsigned int epoch, unsigned int *timed_out, unsigned int *ticket) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) {
        const int x = xy[2 * i], y = xy[2 * i + 1];
        const int lr = band_owned_row(G, x);
        if (lr >= 0) {
            const int ym = y == 0 ? G.N - 1 : y - 1, yp = y == G.N - 1 ? 0 : y + 1;
            // candidates in action order 4..7 = (x, y-1), (x-1, y), (x+1, y), (x, y+1), like k_band_decide_one
            const double food[4] = {dw_food(dwt_new_cell(A, G, lat_old, lat_new, lr, ym)), dw_food(dwt_new_cell(A, G, lat_old, lat_new, lr - 1, y)),
                                    dw_food(dwt_new_cell(A, G, lat_old, lat_new, lr + 1, y)), dw_food(dwt_new_cell(A, G, lat_old, lat_new, lr, yp))};
            const double out = (double)(dw_greedy_pick(food, policy == DW_POLICY_GREEDY) + 1);
            for (int p = 0; p < PT.R; ++p) PT.exch[p][2 * (size_t)n + i] = out;     // owner publishes to every rank
        }
    }
    dw_last_block_barrier(PT, epoch, timed_out, ticket);
}

// ---- materialisation / synthetic reset -------------------------------------------------------------------------------
// full reference grid [7, R, N] of the band, materialised by a literal forward from the post-graze state the last step
// started from: the other lattice buffer, or the fp64 planes when that step was the first one after a reset.
// T = float: the fp32 grid of that state, each value rounded in fp64 and then converted once (fp32 mode of a planes pre-state).
template <class Pre, class T>
__global__ void __launch_bounds__(256) k_band_materialise(DevParams P, double SL, BandGeom G, Pre pre, T *__restrict__ out) {
    const size_t RN = (size_t)G.R * G.N;
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < RN; i += (size_t)gridDim.x * blockDim.x) {
        const int r = (int)(i / G.N), y = (int)(i - (size_t)r * G.N);
        double l9[9], d9[9];
        pre.load9(G, r, y, l9, d9);
        const LitCell o = dw_literal_cell(P, SL, l9, d9);
        out[i] = (T)dw_round3(o.nb);
        out[RN + i] = (T)dw_round3(o.nl);
        out[2 * RN + i] = (T)dw_round3(o.nd);
        out[3 * RN + i] = (T)dw_round3(o.T);
        out[4 * RN + i] = (T)dw_round3(o.Tl);
        out[5 * RN + i] = (T)dw_round3(o.Td);
        out[6 * RN + i] = (T)0.0;
    }
}

// ---- fp32 mode: the band's grid [7, R, N] as float32, evaluated with fp32 arithmetic from the lattice ---------------------
// The per-cell arithmetic of k_forward_f32 (csrc/dw_f32.cuh) in the band geometry: the 3x3 neighbourhood of band row r comes
// from stored rows r .. r+2 of the post-graze pre-state, columns c0 + y - 1 .. c0 + y + W, all in place with the ghost rows
// and columns, so the kernel is a plain grid-stride walk over R x N cells without wrap arithmetic or tile masks. Traffic:
// 4 B of pre-state and 4 B of current state read, 28 B written per cell.
// fp64 tier of the cell at p of the padded lattice (out of line, after the thread's stores, like dw_f32_bare_slow)
__device__ __noinline__ float dwt_f32_bare_slow(const DevParams *Pp, const FastCoef *Fp, const StepCoef *Cp, const uint32_t *p, int pitch,
                                                unsigned *nlit) {
    const uint32_t *q0 = p - pitch, *q2 = p + pitch;
    const uint32_t pc = p[0];
    const uint32_t E = p[-1] + p[1] + q0[0] + q2[0];
    const uint32_t S = E + q0[-1] + q0[1] + q2[-1] + q2[1];
    return dw_f32_bare_tiers(*Pp, *Fp, *Cp, pc, E, S, [=](int a, int c) { return p[(a - 1) * pitch + (c - 1)]; }, nlit);
}
// W cells per thread: W = 2 (N even) loads 8 B and stores float2 -- a stored row starts 16 B aligned (pitch a multiple of 4
// words), c0 = 4 and y is even; W = 1 for odd N (3 CTAs per SM: at the 64 registers of 4 it spills around the fp64-tier call). pre: post-graze pre-state lattice, cur: the lattice after that step.
// out: float [7, R, N], channels 0..6 (4 before the agent stamp). stats[0] += cells sent to the fp64 tier, stats[1] += cells
// that needed the literal cell (per-warp sums).
struct BandF32Args { DevParams P; FastCoef F; StepCoef C; F32Coef Q; BandGeom G; };
template <int W>
__global__ void __launch_bounds__(256, W == 2 ? 4 : 3) k_band_forward_f32(const __grid_constant__ BandF32Args A, const uint32_t *__restrict__ pre,
                                                             const uint32_t *__restrict__ cur, float *__restrict__ out,
                                                             unsigned long long *stats) {
    const F32Coef &Q = A.Q;
    const int pitch = A.G.pitch;
    const unsigned N = (unsigned)A.G.N, gN = N / W;
    const size_t RN = (size_t)A.G.R * N, total = (size_t)A.G.R * gN, stride = (size_t)gridDim.x * blockDim.x;
    size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
    CellWalk w(i, stride, gN);                           // b: band row, c: group of W columns
    unsigned n64 = 0, nlit = 0;
    for (; i < total; i += stride, w.next()) {
        const unsigned r = w.b, y = W * w.c;
        const uint32_t *p = pre + (size_t)r * pitch + A.G.c0 + y;     // stored row r = the row above band row r
        uint32_t row[3][W + 2];                          // rows r-1, r, r+1 of the band; columns y-1 .. y+W
#pragma unroll
        for (int a = 0; a < 3; ++a) {
            const uint32_t *q = p + a * pitch;
            row[a][0] = q[-1];
            if (W == 2) {
                const uint2 v = *reinterpret_cast<const uint2 *>(q);
                row[a][1] = v.x; row[a][2] = v.y;
            } else row[a][1] = q[0];
            row[a][W + 1] = q[W];
        }
        const uint32_t *pc_cur = cur + (size_t)(r + 1) * pitch + A.G.c0 + y;
        uint32_t pn[W];
        if (W == 2) {
            const uint2 v = *reinterpret_cast<const uint2 *>(pc_cur);
            pn[0] = v.x; pn[W - 1] = v.y;
        } else pn[0] = pc_cur[0];
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
        float *ob = out + (size_t)r * N + y;
#pragma unroll
        for (int q = 0; q < 7; ++q) {
            if (W == 2) *reinterpret_cast<float2 *>(ob + (size_t)q * RN) = make_float2(ch[q][0], ch[q][W - 1]);
            else ob[(size_t)q * RN] = ch[q][0];
        }
        // cells whose fp32 bare fraction sits within its error bound of a rounding tie (or outside the accepted range):
        // fp64 tier, the stored channel 0 is overwritten
#pragma unroll
        for (int c = 0; c < W; ++c) {
            if (!ok[c]) {
                n64 += 1;
                ob[c] = dw_div1000f(dwt_f32_bare_slow(&A.P, &A.F, &A.C, p + pitch + c, pitch, &nlit));
            }
        }
    }
    if (stats) {
        n64 = __reduce_add_sync(__activemask(), n64);
        nlit = __reduce_add_sync(__activemask(), nlit);
        if ((threadIdx.x & 31) == 0 && n64) { atomicAdd(stats, (unsigned long long)n64); atomicAdd(stats + 1, (unsigned long long)nlit); }
    }
}
// lattice covers of the band as fp64 planes [2, R, N] (k/1000 exactly as np.round stores them)
__global__ void __launch_bounds__(256) k_band_covers(BandGeom G, const uint32_t *__restrict__ lat, double *__restrict__ out) {
    const size_t RN = (size_t)G.R * G.N;
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < RN; i += (size_t)gridDim.x * blockDim.x) {
        const int r = (int)(i / G.N), y = (int)(i - (size_t)r * G.N);
        const uint32_t w = lat[(size_t)(r + 1) * G.pitch + G.c0 + y];
        out[i] = dw_milli(w & 0xffffu);
        out[RN + i] = dw_milli(w >> 16);
    }
}
// Position-weighted checksum of the band's own cells (exact integer arithmetic on the milli-covers, wraps mod 2^64):
// out[0..3] += {sum kl, sum kd, sum kl * w, sum kd * w}, w = (global_row * 131 + column) % 977 + 1. Additive over bands,
// so the sum over the ranks of a banded world equals the checksum of the same world held as one band.
__global__ void __launch_bounds__(256) k_band_checksum(BandGeom G, const uint32_t *__restrict__ lat, unsigned long long *out) {
    const size_t RN = (size_t)G.R * G.N;
    unsigned long long a[4] = {0, 0, 0, 0};
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < RN; i += (size_t)gridDim.x * blockDim.x) {
        const int r = (int)(i / G.N), y = (int)(i - (size_t)r * G.N);
        const uint32_t w = lat[(size_t)(r + 1) * G.pitch + G.c0 + y];
        const unsigned long long wt = (unsigned long long)((((long long)(G.row0 + r) % G.N) * 131 + y) % 977 + 1);
        a[0] += w & 0xffffu; a[1] += w >> 16; a[2] += (w & 0xffffu) * wt; a[3] += (w >> 16) * wt;
    }
    for (int k = 0; k < 4; ++k) {
        unsigned long long v = a[k];
        for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
        if ((threadIdx.x & 31) == 0 && v) atomicAdd(out + k, v);
    }
}
// agent stamp of ch4 (forward :454-459): the highest agent index on a cell wins. claim holds INT_MAX outside a stamp.
__global__ void __launch_bounds__(256) k_band_stamp_claim(BandGeom G, const int32_t *__restrict__ xy, int n, int *claim) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int lr = band_owned_row(G, xy[2 * i]);
    if (lr >= 0) atomicMin(claim + (size_t)lr * G.N + xy[2 * i + 1], n - 1 - i);
}
// ch4: channel 4 of the fp64 grid, or of the fp32 grid (T = float: the agent's state converted once)
template <class T>
__global__ void __launch_bounds__(256) k_band_stamp_write(BandGeom G, const int32_t *__restrict__ xy, const double *__restrict__ st, int n,
                                                          int *claim, T *ch4, int pass) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int lr = band_owned_row(G, xy[2 * i]);
    if (lr < 0) return;
    const size_t c = (size_t)lr * G.N + xy[2 * i + 1];
    if (pass == 0) { if (claim[c] == n - 1 - i) ch4[(size_t)(lr - 1) * G.N + xy[2 * i + 1]] = (T)st[i]; }
    else claim[c] = 0x7fffffff;
}

// ---- observations (step()'s obs[0], daisy_world_rl.py:246-263, 494) ----------------------------------------------------
// The band's PARTIAL observation obs[n, 7, 3, 3]: one thread per (agent, window cell). A window cell whose row this band
// owns is evaluated whole, as k_obs_from_pre does it (screened, literal next to ties: what forward stored there), from the
// post-graze pre-state at SL = S * L_last; every other cell is 0. A ghost-row cell would need a pre-state row two away from
// the band, which is stored nowhere, so the owner always evaluates: the partial observations of all bands add up to the
// whole one with exactly one non-zero term per element (a caller with several bands sums them, like act).
// ch4 carries the agent stamp (highest index on the cell, dead agents included) from `claim`, filled by k_band_stamp_claim
// (n - 1 - i, smallest wins); a value >= n is idle.
// init != 0: the state right after a reset -- `pre` holds the reset covers themselves, SL = S * L, and the window shows
// initialize_grid's unrounded fields (no stamp; daisy_world_rl.py:304-324), like the init branch of k_obs_from_pre.
template <class Pre>
__global__ void __launch_bounds__(256) k_band_obs(DevParams P, double SL, BandGeom G, Pre pre, const int32_t *__restrict__ xy,
                                                  const double *__restrict__ st, int n, const int *__restrict__ claim,
                                                  double *__restrict__ obs, int init) {
    const size_t total = (size_t)n * 9;
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        const size_t ag = i / 9;
        const int w = (int)(i - ag * 9);
        double *o = obs + ag * 63 + w;
        int x = xy[2 * ag] + w / 3 - 1, y = xy[2 * ag + 1] + w % 3 - 1;
        x = x < 0 ? x + G.N : (x >= G.N ? x - G.N : x);
        y = y < 0 ? y + G.N : (y >= G.N ? y - G.N : y);
        const int lr = band_owned_row(G, x);
        if (lr < 0) {
#pragma unroll
            for (int ch = 0; ch < 7; ++ch) o[9 * ch] = 0.0;
            continue;
        }
        const double mk = P.mask[w];
        double l9[9], d9[9];
        pre.load9(G, lr - 1, y, l9, d9);
        if (init) {
            const LitCell c = dw_literal_cell(P, SL, l9, d9);
            o[0] = c.b0 * mk; o[9] = l9[4] * mk; o[18] = d9[4] * mk; o[27] = c.T * mk; o[36] = c.Tl * mk; o[45] = c.Td * mk;
            o[54] = 0.0 * mk;
            continue;
        }
        ScrCell c;
        if (!(P.screen && dw_screened_cell(P, SL / P.sigma, l9, d9, c))) dw_literal_rounded(P, SL, l9, d9, c);
        const int s = claim[(size_t)lr * G.N + y];
        const double ch4 = (s >= 0 && s < n) ? st[n - 1 - s] : dw_k2v(c.k[4]);
        o[0] = dw_k2v(c.k[0]) * mk;
        o[9] = dw_k2v(c.k[1]) * mk;
        o[18] = dw_k2v(c.k[2]) * mk;
        o[27] = dw_k2v(c.k[3]) * mk;
        o[36] = ch4 * mk;
        o[45] = dw_k2v(c.k[5]) * mk;
        o[54] = 0.0 * mk;
    }
}

// device-side synthetic reset of the band (+ its ghost rows) and of the replicated agents: same distribution as
// initialize_grid / initialize_agents (daisy_world_rl.py:285-302, 173-179), counter RNG keyed by the GLOBAL cell index,
// so any banding of the same world draws the same state.
__global__ void __launch_bounds__(256) k_band_init_random(BandGeom Gp, uint64_t seed, double prop_l, double prop_d, double init_l,
                                                          double init_d, double *l, double *d, int32_t *agent_xy, double *agent_state, int n) {
    const size_t total = (size_t)(Gp.R + 2) * Gp.N;
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        const int r = (int)(i / Gp.N), y = (int)(i - (size_t)r * Gp.N);
        int x = Gp.row0 + r - 1;
        x = x < 0 ? x + Gp.N : (x >= Gp.N ? x - Gp.N : x);
        const uint64_t gidx = (uint64_t)x * Gp.N + y;
        d[i] = dw_u01(seed, gidx, 0) < prop_d ? init_d * dw_u01(seed, gidx, 1) : 0.0;
        l[i] = dw_u01(seed, gidx, 2) < prop_l ? init_l * dw_u01(seed, gidx, 3) : 0.0;
    }
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < (size_t)n; i += (size_t)gridDim.x * blockDim.x) {
        agent_xy[2 * i] = (int)(dw_u01(seed ^ 0xA5A5A5A5ull, i, 0) * Gp.N);
        agent_xy[2 * i + 1] = (int)(dw_u01(seed ^ 0xA5A5A5A5ull, i, 1) * Gp.N);
        agent_state[i] = 1.0;
    }
}

// ---- diagnostics and plot feed (the unrounded fields of the last forward, their statistics, block-averaged images) ------
// Every field is evaluated like k_band_materialise: dw_literal_cell on the post-graze pre-state at SL = S * L_last. Field
// selectors are those of dwt_pool (include/daisyworld_b200_tiled.h): 0..6 equal DW_DIAG_TEMP..DW_DIAG_BETA_D, then the two
// growth planes and the grid channels 0, 1, 2, 3, 5 as dwt_get_grid holds them. The one mapping all field kernels share:
__device__ __forceinline__ double dwt_field_value(const LitCell &o, int field) {
    switch (field) {
        case DWT_FIELD_TEMP: return o.T;
        case DWT_FIELD_TEMP_LIGHT: return o.Tl;
        case DWT_FIELD_TEMP_DARK: return o.Td;
        case DWT_FIELD_TEMP_EFFECTIVE: return o.Te;
        case DWT_FIELD_BETA: return o.beta;
        case DWT_FIELD_BETA_L: return o.beta_l;
        case DWT_FIELD_BETA_D: return o.beta_d;
        case DWT_FIELD_GROWTH_L: return o.dl;
        case DWT_FIELD_GROWTH_D: return o.dd;
        case DWT_FIELD_GRID_BARE: return dw_round3(o.nb);
        case DWT_FIELD_GRID_LIGHT: return dw_round3(o.nl);
        case DWT_FIELD_GRID_DARK: return dw_round3(o.nd);
        case DWT_FIELD_GRID_TEMP: return dw_round3(o.T);
        default: return dw_round3(o.Td);                 // DWT_FIELD_GRID_TEMP_DARK
    }
}
// the cell (r, y) of the band (band row r, 0-based), evaluated from the pre-state
template <class Pre>
__device__ __forceinline__ LitCell dwt_band_cell(const DevParams &P, double SL, const BandGeom &G, const Pre &pre, int r, int y) {
    double l9[9], d9[9];
    pre.load9(G, r, y, l9, d9);
    return dw_literal_cell(P, SL, l9, d9);
}

// One DW_DIAG_* field of the band [R, N] (DW_DIAG_GROWTH: [2, R, N], dl then dd), as k_diag computes it.
template <class Pre>
__global__ void __launch_bounds__(256) k_band_diag(DevParams P, double SL, BandGeom G, Pre pre, int which, double *__restrict__ out) {
    const size_t RN = (size_t)G.R * G.N;
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < RN; i += (size_t)gridDim.x * blockDim.x) {
        const int r = (int)(i / G.N), y = (int)(i - (size_t)r * G.N);
        const LitCell o = dwt_band_cell(P, SL, G, pre, r, y);
        if (which == DW_DIAG_GROWTH) {
            out[i] = dwt_field_value(o, DWT_FIELD_GROWTH_L);
            out[RN + i] = dwt_field_value(o, DWT_FIELD_GROWTH_D);
        } else {
            out[i] = dwt_field_value(o, which);
        }
    }
}

// Statistics of one DW_DIAG_* field over the band's own cells, evaluated and reduced without storing the field: per thread
// {sum, sum of squares} of (x - shift), min and max, then dw_stats_block_reduce -> partial[4 * blockIdx.x]. The shift is the
// field at the band's first cell (dl there for growth, whose two planes are reduced together); block 0 stores it at
// partial[4 * gridDim.x + 4], behind the 4 results of k_band_partials_final. A fixed grid gives a fixed summation order.
template <class Pre>
__global__ void __launch_bounds__(256) k_band_field_stats(DevParams P, double SL, BandGeom G, Pre pre, int which, double *__restrict__ partial) {
    const bool growth = which == DW_DIAG_GROWTH;
    const int f0 = growth ? DWT_FIELD_GROWTH_L : which;
    const double shift = dwt_field_value(dwt_band_cell(P, SL, G, pre, 0, 0), f0);
    double s = 0.0, q = 0.0, mn = 1e300, mx = -1e300;
    const size_t RN = (size_t)G.R * G.N;
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < RN; i += (size_t)gridDim.x * blockDim.x) {
        const int r = (int)(i / G.N), y = (int)(i - (size_t)r * G.N);
        const LitCell o = dwt_band_cell(P, SL, G, pre, r, y);
        for (int k = 0; k < (growth ? 2 : 1); ++k) {
            const double v = dwt_field_value(o, f0 + k), d = v - shift;
            s += d; q += d * d; mn = fmin(mn, v); mx = fmax(mx, v);
        }
    }
    dw_stats_block_reduce(s, q, mn, mx, partial + 4 * blockIdx.x);
    if (blockIdx.x == 0 && threadIdx.x == 0) partial[4 * gridDim.x + 4] = shift;
}

// Covers of the band's own cells in the current state: per block {sum light, sum dark, min(-light), max dark} (the min slot
// of dw_stats_block_reduce carries the light maximum negated). On the lattice the values are the integer milli-covers, so
// every sum is exact (below 2^53) and independent of the order; on the fp64 planes of a reset the fixed grid fixes it.
__device__ __forceinline__ void dwt_cell_covers(const LatCells &C, size_t i, double &l, double &d) {
    const uint32_t w = C.p[i];
    l = (double)(w & 0xffffu);
    d = (double)(w >> 16);
}
__device__ __forceinline__ void dwt_cell_covers(const PlaneCells &C, size_t i, double &l, double &d) { l = C.l[i]; d = C.d[i]; }
template <class Cells>
__global__ void __launch_bounds__(256) k_band_cover_stats(BandGeom G, Cells C, double *__restrict__ partial) {
    double sl = 0.0, sd = 0.0, nml = 1e300, md = -1e300;
    const size_t RN = (size_t)G.R * G.N;
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < RN; i += (size_t)gridDim.x * blockDim.x) {
        const int r = (int)(i / G.N), y = (int)(i - (size_t)r * G.N);
        double l, d;
        dwt_cell_covers(C, (size_t)(r + 1) * G.pitch + G.c0 + y, l, d);
        sl += l; sd += d; nml = fmin(nml, -l); md = fmax(md, d);
    }
    dw_stats_block_reduce(sl, sd, nml, md, partial + 4 * blockIdx.x);
}

// Second stage of both: the `blocks` partials in a fixed order -> out[0..3] = {sum, sum, min, max}.
__global__ void __launch_bounds__(256) k_band_partials_final(const double *__restrict__ partial, int blocks, double *__restrict__ out) {
    double s = 0.0, q = 0.0, mn = 1e300, mx = -1e300;
    for (int i = threadIdx.x; i < blocks; i += blockDim.x) {
        s += partial[4 * i]; q += partial[4 * i + 1]; mn = fmin(mn, partial[4 * i + 2]); mx = fmax(mx, partial[4 * i + 3]);
    }
    dw_stats_block_reduce(s, q, mn, mx, out);
}

// Block sums of a field for a block-averaged image: output block (i, j) covers global rows and columns [i*b, min((i+1)*b, N))
// x [j*b, min((j+1)*b, N)); only the cells this band owns count, so the sum over the ranks is the whole world's. Work unit u =
// (output block, slice s of `slices`) -- the slice takes every slices-th row of the block -- is reduced by one warp in a
// fixed order (lane-strided, then a shuffle tree); out[u] is written for every unit, 0 where the band owns nothing.
// slices == 1: out is the [H, H] image; else [H * H, slices] partials for k_band_pool_final.
template <class Pre>
__global__ void __launch_bounds__(256) k_band_pool(DevParams P, double SL, BandGeom G, Pre pre, int field, int b, int H, int slices,
                                                   double *__restrict__ out) {
    const int lane = threadIdx.x & 31;
    const long long units = (long long)H * H * slices;
    for (long long u = (blockIdx.x * (long long)blockDim.x + threadIdx.x) >> 5; u < units; u += ((long long)gridDim.x * blockDim.x) >> 5) {
        const long long blk = u / slices;
        const int s = (int)(u - blk * slices);
        const int bi = (int)(blk / H), bj = (int)(blk - (long long)bi * H);
        const int x0 = bi * b, y0 = bj * b;
        const int bh = min(b, G.N - x0), bw = min(b, G.N - y0);
        const int sh = bh > s ? (bh - s + slices - 1) / slices : 0;    // rows s, s + slices, ... of the block
        double acc = 0.0;
        for (int k = lane; k < sh * bw; k += 32) {
            const int rr = k / bw, y = y0 + (k - rr * bw);
            const int lr = band_owned_row(G, x0 + s + rr * slices);
            if (lr >= 0) acc += dwt_field_value(dwt_band_cell(P, SL, G, pre, lr - 1, y), field);
        }
        for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
        if (lane == 0) out[u] = acc;
    }
}
__global__ void __launch_bounds__(256) k_band_pool_final(const double *__restrict__ partial, int slices, long long hh, double *__restrict__ out) {
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < hh; i += (long long)gridDim.x * blockDim.x) {
        double acc = 0.0;
        for (int s = 0; s < slices; ++s) acc += partial[i * slices + s];
        out[i] = acc;
    }
}
