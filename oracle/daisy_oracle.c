/*
 * CPU oracle (plain C) for the RLDaisyWorld simulation step -- TEST INFRASTRUCTURE ONLY.
 *
 * Restates the algorithm of the reference environment daisy/daisy_world_rl.py
 * (riveSunder/therldaisyworld) with the FFT convolution (daisy/nn/functional.py:12-49) replaced
 * by the 3x3 toroidal stencil it is mathematically equal to.  Arithmetic follows, operation for
 * operation, the canonical order documented in oracle/daisy_numpy.py (which is pinned against
 * trajectories recorded from the live reference, tests/golden/).  Build with
 *     gcc -O2 -ffp-contract=off -fopenmp -shared -fPIC   (see oracle/build_oracle.py)
 * -ffp-contract=off is REQUIRED: the canonical order has no fused multiply-adds.
 *
 * Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may
 * load this library.  The product (therldaisyworld_b200/) never does.
 *
 * Parity status: the reference ships no golden vectors for this path; this oracle is pinned
 * through tests/test_oracle_c.py (bit-equal to the NumPy oracle and to the reference-recorded
 * fixtures).
 */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

typedef struct {
    int32_t B, N, n_agents, ch;            /* ch is always 7 (reference :18) */
    double p, g, S, sigma, gamma, q, q2, temp_optimal, dt, agent_gamma;
    double albedo_bare, albedo_light, albedo_dark;
    double mask[9];                        /* observation neighbourhood, row-major 3x3 */
    double w[9];                           /* daisy-spread kernel (reference :270-273), computed by the
                                              caller with NumPy exactly as the reference does */
    double adj[9];                         /* adjacent-albedo kernel (reference :278-281), row-major 3x3 */
} dwo_params;

static inline double root4(double x) { return sqrt(sqrt(x)); }
static inline double pow4(double x) { double x2 = x * x; return x2 * x2; }
static inline double round3(double x) { return rint(x * 1000.0) / 1000.0; }
static inline double clip01(double x) { x = x < 0.0 ? 0.0 : x; return x > 1.0 ? 1.0 : x; }

/* diag (optional): [B,9,N,N] = T, Tl, Td, Te, beta, beta_l, beta_d, dl, dd (all unrounded) */
void dwo_forward(const dwo_params *P, double L, double *grid, const int64_t *agent_idx,
                 const double *agent_state, double *out, double *diag) {
    const int N = P->N, B = P->B;
    const size_t NN = (size_t)N * N;
    const double *w = P->w, *adj = P->adj;
    const int skip_centre = adj[4] == 0.0;   /* the default adjacent kernel: its zero centre term is not added */
    const double ab = P->albedo_bare, al = P->albedo_light, ad = P->albedo_dark;
    const double SL = P->S * L;
#pragma omp parallel for schedule(static)
    for (int bb = 0; bb < B; ++bb) {
        double *g = grid + (size_t)bb * 7 * NN;
        double *o = out + (size_t)bb * 7 * NN;
        double *bare = g, *lt = g + NN, *dk = g + 2 * NN;
        for (size_t i = 0; i < NN; ++i) bare[i] = (P->p - lt[i]) - dk[i];   /* :381, in place */
        for (int x = 0; x < N; ++x) {
            int xs[3] = {(x + N - 1) % N, x, (x + 1) % N};
            for (int y = 0; y < N; ++y) {
                int ys[3] = {(y + N - 1) % N, y, (y + 1) % N};
                size_t c = (size_t)x * N + y;
                double nb_b = 0, nb_l = 0, nb_d = 0, rho_l = 0, rho_d = 0;
                int first = 1, first9 = 1;
                /* circular convolution like ft_convolve (daisy/nn/functional.py:12-49): the neighbour at offset
                   (a-1, b-1), visited row-major, is weighted by the tap turned 180 degrees, w[2-a][2-b] */
                for (int a = 0; a < 3; ++a)
                    for (int b = 0; b < 3; ++b) {
                        size_t k = (size_t)xs[a] * N + ys[b];
                        const int t = 8 - (a * 3 + b);
                        double tl = w[t] * lt[k], td = w[t] * dk[k];
                        if (first9) { rho_l = tl; rho_d = td; first9 = 0; }
                        else { rho_l = rho_l + tl; rho_d = rho_d + td; }
                        if (a == 1 && b == 1 && skip_centre) continue;
                        double vb = adj[t] * bare[k], vl = adj[t] * lt[k], vd = adj[t] * dk[k];
                        if (first) { nb_b = vb; nb_l = vl; nb_d = vd; first = 0; }
                        else { nb_b = nb_b + vb; nb_l = nb_l + vl; nb_d = nb_d + vd; }
                    }
                double l = lt[c], d = dk[c], b0 = bare[c];
                double Al = (ab * b0 + al * l) + ad * d;
                double A = (ab * nb_b + al * nb_l) + ad * nb_d;
                double Te = root4((SL * (1 - A)) / P->sigma);
                double T = root4(P->q * (A - Al) + pow4(Te));
                double T4 = pow4(T);
                double Tl = root4(P->q2 * (Al - al) + T4);
                double Td = root4(P->q2 * (Al - ad) + T4);
                double dT = P->temp_optimal - T, dTl = P->temp_optimal - Tl, dTd = P->temp_optimal - Td;
                double beta = 1 - P->g * (dT * dT);
                double beta_l = 1 - P->g * (dTl * dTl);
                double beta_d = 1 - P->g * (dTd * dTd);
                double rb = (P->p - rho_l) - rho_d;
                double dl = rho_l * (rb * beta_l - P->gamma);
                double dd = rho_d * (rb * beta_d - P->gamma);
                double nl = clip01(l + P->dt * dl), nd = clip01(d + P->dt * dd);
                double nb = (P->p - nl) - nd;
                o[c] = round3(nb); o[NN + c] = round3(nl); o[2 * NN + c] = round3(nd);
                o[3 * NN + c] = round3(T); o[4 * NN + c] = round3(Tl); o[5 * NN + c] = round3(Td);
                o[6 * NN + c] = 0.0;
                if (diag) {
                    double *q = diag + (size_t)bb * 9 * NN + c;
                    q[0] = T; q[NN] = Tl; q[2 * NN] = Td; q[3 * NN] = Te; q[4 * NN] = beta;
                    q[5 * NN] = beta_l; q[6 * NN] = beta_d; q[7 * NN] = dl; q[8 * NN] = dd;
                }
            }
        }
        /* agent stamp: agent order, last wins, dead agents included (:454-459) */
        for (int nn = 0; nn < P->n_agents; ++nn) {
            const int64_t *xy = agent_idx + ((size_t)bb * P->n_agents + nn) * 2;
            o[4 * NN + (size_t)xy[0] * N + xy[1]] = agent_state[(size_t)bb * P->n_agents + nn];
        }
    }
}

/* action: [ab, am] (ab<=B, am<=n_agents), values 0..8; reference :181-244 (collision_mode 0) */
void dwo_update_agents(const dwo_params *P, double *grid, int64_t *agent_idx, double *agent_state,
                       const int64_t *action, int ab, int am) {
    const int N = P->N, n = P->n_agents;
    const size_t NN = (size_t)N * N;
#pragma omp parallel for schedule(static)
    for (int bb = 0; bb < P->B; ++bb) {
        double *st = agent_state + (size_t)bb * n;
        int64_t *ix = agent_idx + (size_t)bb * n * 2;
        double *g = grid + (size_t)bb * 7 * NN;
        for (int nn = 0; nn < n; ++nn) st[nn] = st[nn] - P->agent_gamma;
        if (bb < ab)
            for (int nn = 0; nn < am; ++nn) {
                if (!(st[nn] > 0.0)) continue;
                int a = (int)action[(size_t)bb * am + nn];
                int64_t x = ix[nn * 2], y = ix[nn * 2 + 1];
                if (a != 8) {
                    switch (a % 4) {
                        case 0: y -= 1; break;
                        case 1: x -= 1; break;
                        case 2: x += 1; break;
                        default: y += 1; break;
                    }
                }
                x = ((x % N) + N) % N; y = ((y % N) + N) % N;
                ix[nn * 2] = x; ix[nn * 2 + 1] = y;
                if (a > 4) {
                    size_t c = (size_t)x * N + y;
                    st[nn] = st[nn] + (g[NN + c] + g[2 * NN + c]);
                    g[NN + c] *= 0.0; g[2 * NN + c] *= 0.0;
                }
            }
        for (int nn = 0; nn < n; ++nn) st[nn] = clip01(st[nn]);
    }
}

/* obs: [B, n, 7, 3, 3]; reference :246-263 */
void dwo_get_obs(const dwo_params *P, const double *grid, const int64_t *agent_idx, double *obs) {
    const int N = P->N, n = P->n_agents;
    const size_t NN = (size_t)N * N;
#pragma omp parallel for schedule(static)
    for (int bb = 0; bb < P->B; ++bb)
        for (int nn = 0; nn < n; ++nn) {
            const int64_t *xy = agent_idx + ((size_t)bb * n + nn) * 2;
            double *o = obs + ((size_t)bb * n + nn) * 63;
            for (int c = 0; c < 7; ++c)
                for (int a = 0; a < 3; ++a)
                    for (int b = 0; b < 3; ++b) {
                        int x = (int)((xy[0] + a - 1 + N) % N), y = (int)((xy[1] + b - 1 + N) % N);
                        o[c * 9 + a * 3 + b] = grid[((size_t)bb * 7 + c) * NN + (size_t)x * N + y] * P->mask[a * 3 + b];
                    }
        }
}

/* Greedy policy, deterministic branch (reference daisy/agents/greedy.py:16-30). */
void dwo_greedy(const dwo_params *P, const double *obs, int greedy, int64_t *action) {
    static const int cand[4] = {3, 1, 7, 5};
    const int total = P->B * P->n_agents;
#pragma omp parallel for schedule(static)
    for (int i = 0; i < total; ++i) {
        const double *o = obs + (size_t)i * 63;
        int best = 0;
        double bv = o[9 + cand[0]] + o[18 + cand[0]];
        for (int k = 1; k < 4; ++k) {
            double v = o[9 + cand[k]] + o[18 + cand[k]];
            if (greedy ? (v > bv) : (v < bv)) { bv = v; best = k; }
        }
        action[i] = 4 + best;
    }
}

typedef struct {
    double L, dL, min_L, max_L, ddL;
    int64_t step_count, ramp_period;
    int32_t ramp_up_down, pad;
} dwo_clock;

static void update_L(dwo_clock *c) {   /* reference :463-473 */
    c->step_count += 1;
    if (c->ramp_up_down && c->step_count % c->ramp_period == 0) {
        c->dL *= -1; c->min_L -= c->ddL; c->max_L += c->ddL;
    }
    double L = c->L + c->dL;
    L = L < c->max_L ? L : c->max_L;
    c->L = L > c->min_L ? L : c->min_L;
}

/* One env.step (reference :475-497).  action==NULL with agents => all-zero action.
   grid is replaced in place; scratch must hold B*7*N*N doubles.
   reward[B,n] f64, done[B,n] u8 (n_agents>0) or reward[B,2]/done[B,2] as 0/1 (n_agents==0). */
void dwo_step(const dwo_params *P, dwo_clock *clk, double *grid, double *scratch, int64_t *agent_idx,
              double *agent_state, const int64_t *action, int ab, int am, double *obs, double *reward,
              uint8_t *done) {
    const int n = P->n_agents, N = P->N;
    const size_t NN = (size_t)N * N, G = (size_t)P->B * 7 * NN;
    if (n > 0) {
        if (action) dwo_update_agents(P, grid, agent_idx, agent_state, action, ab, am);
        else {
            int64_t *zero = (int64_t *)calloc((size_t)P->B * n, sizeof(int64_t));
            dwo_update_agents(P, grid, agent_idx, agent_state, zero, P->B, n);
            free(zero);
        }
    }
    dwo_forward(P, clk->L, grid, agent_idx, agent_state, scratch, NULL);
    memcpy(grid, scratch, G * sizeof(double));
    if (obs) dwo_get_obs(P, grid, agent_idx, obs);
    if (n > 0) {
        for (size_t i = 0; i < (size_t)P->B * n; ++i) {
            double r = agent_state[i];
            r = r * (r > 0 ? 1.0 : 0.0);
            if (reward) reward[i] = r;
            if (done) done[i] = r < 0.1;
        }
    } else {
        for (int bb = 0; bb < P->B; ++bb)
            for (int c = 0; c < 2; ++c) {
                double s = 0;
                const double *f = grid + ((size_t)bb * 7 + 1 + c) * NN;
                for (size_t i = 0; i < NN; ++i) s += f[i];
                int r = s > 0;
                if (reward) reward[bb * 2 + c] = r;
                if (done) done[bb * 2 + c] = r < 0.1;
            }
    }
    update_L(clk);
}

/* Lifespan experiment (notebooks/greedy_longevity_abatement.ipynb cell 2) with an on-host policy:
   policy 0 = none (action None), 1 = greedy, 2 = anti-greedy, 3 = replay actions[K,B,n].
   Runs until every world is grid_done in the same step (stop_all_done) or K steps.
   Returns the number of steps run.  done_at[B], agents_done_at[B,n] are incremented. */
int64_t dwo_run(const dwo_params *P, dwo_clock *clk, double *grid, int64_t *agent_idx, double *agent_state,
                int policy, const int64_t *actions, int64_t K, int stop_all_done, int64_t *done_at,
                int64_t *agents_done_at) {
    const int n = P->n_agents, N = P->N, B = P->B;
    const size_t NN = (size_t)N * N;
    double *scratch = (double *)malloc((size_t)B * 7 * NN * sizeof(double));
    double *obs = (double *)malloc(((size_t)B * (n ? n : 1)) * 63 * sizeof(double));
    int64_t *act = (int64_t *)malloc(((size_t)B * (n ? n : 1)) * sizeof(int64_t));
    uint8_t *done = (uint8_t *)malloc((size_t)B * (n ? n : 2));
    int64_t t = 0;
    if (n) dwo_get_obs(P, grid, agent_idx, obs);
    while (t < K) {
        const int64_t *a = NULL;
        if (n && (policy == 1 || policy == 2)) { dwo_greedy(P, obs, policy == 1, act); a = act; }
        else if (n && policy == 3) a = actions + (size_t)t * B * n;
        dwo_step(P, clk, grid, scratch, agent_idx, agent_state, a, B, n, obs, NULL, done);
        ++t;
        int all_done = 1;
#pragma omp parallel for schedule(static) reduction(&& : all_done)
        for (int bb = 0; bb < B; ++bb) {
            const double *f = grid + ((size_t)bb * 7 + 1) * NN;
            double m = f[0];
            for (size_t i = 1; i < 2 * NN; ++i) m = f[i] > m ? f[i] : m;
            int gd = m <= 0.005;
            done_at[bb] += 1 - gd;
            all_done = all_done && gd;
            for (int nn = 0; nn < n; ++nn) agents_done_at[(size_t)bb * n + nn] += 1 - done[(size_t)bb * n + nn];
        }
        if (stop_all_done && all_done) break;
    }
    free(scratch); free(obs); free(act); free(done);
    return t;
}

/* Test support: number of integers k in [0,kmax] for which Markstein's division-free k/1000
   (q = k*0.001; r = fma(-1000,q,k); q + r*0.001), used by the CUDA kernels, differs from k/1000.0. */
long dwo_check_markstein(long kmax) {
    long bad = 0;
    for (long k = 0; k <= kmax; ++k) {
        double kd = (double)k, q = kd * 0.001, r = fma(-1000.0, q, kd), f = fma(r, 0.001, q);
        if (f != kd / 1000.0) ++bad;
        kd = -kd; q = kd * 0.001; r = fma(-1000.0, q, kd); f = fma(r, 0.001, q);
        if (f != kd / 1000.0) ++bad;
    }
    return bad;
}

int dwo_sizeof_params(void) { return (int)sizeof(dwo_params); }
int dwo_sizeof_clock(void) { return (int)sizeof(dwo_clock); }
