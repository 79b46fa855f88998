/*
 * imx_oracle.c — TEST INFRASTRUCTURE: plain-C restatement of the MARL-for-IM environment step.
 *
 * This is the checker for full-size batches, not the product: only tests/, __graft_entry__.smoke()
 * and bench.py's CPU-baseline legs load it (through oracle/c_oracle.py).  It restates the same
 * algorithm as oracle/im_oracle.py (which is pinned bit-for-bit to the unmodified reference and to
 * tests/golden/) with scalar loops: one environment at a time, one stage at a time, in the order the
 * reference executes them.  Config derivation (order_max, demand_max, node prices, topology) is done
 * by oracle/im_oracle.py and passed in; this file only runs the dynamics.
 *
 * Reference lines followed (paths relative to the reference root):
 *   order clipping        IM_env.py:298-302  MAIM_env.py:340-347  IM_div_env.py:372-376  MAIM_div_env.py:451-456
 *   demand propagation    MAIM_env.py:351-353  MAIM_div_env.py:460-467
 *   update_acquisition    MAIM_env.py:438-476  MAIM_div_env.py:657-695
 *   ship / state update   MAIM_env.py:360-384  MAIM_div_env.py:474,582-603
 *   divergent split       MAIM_div_env.py:476-579  IM_div_env.py:396-502
 *   pipeline shift        MAIM_env.py:478-495  MAIM_div_env.py:697-715
 *   rewards               MAIM_env.py:413-436  IM_env.py:362-374  MAIM_div_env.py:632-655  IM_div_env.py:551-563
 *   observation           MAIM_env.py:242-328  IM_env.py:231-285  MAIM_div_env.py:343-439  IM_div_env.py:304-359
 *   base-stock policy     base_restock_policy.py:4-45
 *
 * Build: gcc -O2 -fPIC -shared -fopenmp -ffp-contract=off imx_oracle.c -lm   (no FMA contraction:
 * every product, quotient and sum is a separate IEEE-754 double rounding, like numpy).
 */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>
#ifdef _OPENMP
#include <omp.h>
#endif

#define ORC_MAX_NODES 32
#define ORC_MAX_CHILDREN 8
#define ORC_MAX_DELAY 16
#define ORC_MAX_HIST 16

typedef struct orc_cfg {
    int32_t multi, div, m, T, P, D, O, R;
    int32_t std_state, std_actions, cap_backlog, independent, share_network, td, pd, pa;
    int32_t wd_mult1, wd_mult;                 /* watchdog multipliers of the divergent split */
    double a, b;
    int32_t inv_init[ORC_MAX_NODES], inv_max[ORC_MAX_NODES], order_max[ORC_MAX_NODES], demand_max[ORC_MAX_NODES];
    int32_t delay[ORC_MAX_NODES], parent[ORC_MAX_NODES], nchild[ORC_MAX_NODES], retailer_idx[ORC_MAX_NODES];
    int32_t children[ORC_MAX_NODES][ORC_MAX_CHILDREN];
    double p[ORC_MAX_NODES], c[ORC_MAX_NODES], h[ORC_MAX_NODES], bc[ORC_MAX_NODES], target[ORC_MAX_NODES];
} orc_cfg;

typedef struct {
    int inv[ORC_MAX_NODES], backlog[ORC_MAX_NODES], order_u[ORC_MAX_NODES], carry[ORC_MAX_NODES];
    int pipe[ORC_MAX_NODES][ORC_MAX_DELAY];
    int hd[ORC_MAX_NODES][ORC_MAX_HIST], ho[ORC_MAX_NODES][ORC_MAX_HIST];
    int bt[ORC_MAX_NODES][ORC_MAX_CHILDREN];
} orc_state;

int orc_cfg_size(void) { return (int)sizeof(orc_cfg); }

static double rescale(double v, double vmax, double a, double b) { return a + (((v - 0.0) * (b - a)) / (vmax - 0.0)); }
static double rev_scale(double x, double vmax, double a, double b) { return (((x - a) * (vmax - 0.0)) / (b - a)) + 0.0; }

/* numpy pairwise_sum order (loops_utils.h.src): sequential below 8, eight accumulators up to 128, recursive split above */
static double np_sum(const double* v, int n) {
    if (n < 8) {
        double r = 0.0;
        for (int i = 0; i < n; ++i) r += v[i];
        return r;
    }
    if (n > 128) {
        int n2 = n / 2;
        n2 -= n2 % 8;
        return np_sum(v, n2) + np_sum(v + n2, n - n2);
    }
    double r[8];
    for (int j = 0; j < 8; ++j) r[j] = v[j];
    int i = 8;
    for (; i < n - (n % 8); i += 8)
        for (int j = 0; j < 8; ++j) r[j] += v[i + j];
    double res = ((r[0] + r[1]) + (r[2] + r[3])) + ((r[4] + r[5]) + (r[6] + r[7]));
    for (; i < n; ++i) res += v[i];
    return res;
}

static void reset_state(const orc_cfg* c, orc_state* s) {
    memset(s, 0, sizeof(*s));
    for (int i = 0; i < c->m; ++i) s->inv[i] = c->inv_init[i];
}

static void observe(const orc_cfg* c, const orc_state* s, int t, double* obs /* [m][O] */) {
    const int m = c->m, O = c->O, P = c->P, D = c->D;
    const double a = c->a, b = c->b;
    for (int i = 0; i < m; ++i) {
        double* row = obs + (size_t)i * O;
        for (int k = 0; k < O; ++k) row[k] = 0.0;
        const double inv_max = c->inv_max[i], order_max = c->order_max[i];
        const double dem_max = c->div ? (double)c->demand_max[i] : inv_max;
        const double ou_max = c->multi ? order_max : inv_max;
        if (c->std_state) {
            row[0] = rescale(s->inv[i], inv_max, a, b);
            row[1] = rescale(s->backlog[i], dem_max, a, b);
            row[2] = rescale(s->order_u[i], ou_max, a, b);
        } else {
            row[0] = s->inv[i]; row[1] = s->backlog[i]; row[2] = s->order_u[i];
        }
        if (c->multi && !c->std_state) {                 /* MAIM_env.py:319-324 */
            if (t >= 1 && c->td)
                for (int k = 0; k < D; ++k) row[3 + k] = s->pipe[i][k];
            continue;
        }
        int k0 = 3;
        if (c->multi && c->pd && !c->pa && !c->td) {
            k0 += P;                                     /* slot exists, never written */
        } else {
            if (c->pd) { for (int j = 0; j < P; ++j) row[k0 + j] = rescale(j < t ? s->hd[i][j] : 0, dem_max, a, b); k0 += P; }
            if (c->pa) { for (int j = 0; j < P; ++j) row[k0 + j] = rescale(j < t ? s->ho[i][j] : 0, order_max, a, b); k0 += P; }
        }
        if (c->td) {
            for (int k = 0; k < D; ++k) {
                const int raw = t >= 1 ? s->pipe[i][k] : 0;
                double v;
                if (!c->std_state) v = raw;
                else if (c->div && c->multi) v = rescale(raw < 2 * c->inv_max[i] ? raw : 2 * c->inv_max[i], 2.0 * inv_max, a, b);
                else v = rescale(raw, inv_max, a, b);
                row[k0 + k] = v;
            }
            k0 += D;
        }
        if (c->share_network) row[O - 1] = rescale(i, (double)m, a, b);
    }
}

static int decode_order(const orc_cfg* c, int i, double x) {
    const double om = c->order_max[i];
    if (c->std_actions) x = rev_scale(x, om, c->a, c->b);
    if (c->multi) {
        /* round, .astype(int), clip (MAIM_env.py:344-347): on the reference's x86-64 the float64 -> int64 conversion of NaN,
         * +-inf and anything outside [-2^63, 2^63) yields INT64_MIN, which the clip turns into 0 */
        x = rint(x);
        if (!(x >= -9223372036854775808.0 && x < 9223372036854775808.0)) x = -9223372036854775808.0;
        x = x < 0.0 ? 0.0 : x; x = x > om ? om : x;
    }
    else { x = x < 0.0 ? 0.0 : x; x = x > om ? om : x; x = rint(x); }
    return (int)x;
}

/* dm * mult saturated at INT32_MAX: a pass count never exceeds the int32 amount it hands out, so the saturated limit fires
 * exactly where the reference's unbounded product would */
static int wd_limit(int dm, int mult) { return dm > INT32_MAX / mult ? INT32_MAX : dm * mult; }

/* returns the watchdog code (0 ok) */
static int split(const orc_cfg* c, orc_state* s, int i, int ship, int demand, int backlog, const int* order, int* st) {
    const int nc = c->nchild[i];
    const int lim1 = wd_limit(c->demand_max[i], c->wd_mult1), lim = wd_limit(c->demand_max[i], c->wd_mult);
    int* bt = s->bt[i];
    int od[ORC_MAX_CHILDREN];
    int amt = ship;
    for (int k = 0; k < nc; ++k) { st[k] = 0; od[k] = order[c->children[i][k]]; }
    if (nc == 1) { st[0] = ship; return 0; }
    if (ship >= demand) {
        if (backlog > 0) {
            int cnt = 0;
            for (;;) {
                int sum = 0;
                for (int k = 0; k < nc; ++k) sum += bt[k];
                if (!(sum > 0 && amt > 0)) break;
                for (int k = 0; k < nc; ++k) if (bt[k] > 0) { st[k]++; bt[k]--; amt--; }
                if (++cnt > lim1) return 1;
            }
            if (amt > 0 && demand > 0) {
                int out[ORC_MAX_CHILDREN];
                for (int k = 0; k < nc; ++k) out[k] = od[k];
                cnt = 0;
                for (;;) {
                    int sum = 0;
                    for (int k = 0; k < nc; ++k) sum += out[k];
                    if (!(amt > 0 && sum > 0)) break;
                    for (int k = 0; k < nc; ++k) if (out[k] > 0) { st[k]++; out[k]--; amt--; }
                    if (++cnt > lim) return 2;
                }
                for (int k = 0; k < nc; ++k) bt[k] += out[k];
            }
        } else {
            for (int k = 0; k < nc; ++k) st[k] += od[k];
        }
    } else {
        if (backlog > 0) {
            int cnt = 0;
            for (;;) {
                int sum = 0;
                for (int k = 0; k < nc; ++k) sum += bt[k];
                if (!(sum > 0 && amt > 0)) break;
                for (int k = 0; k < nc; ++k) if (bt[k] > 0) { st[k]++; bt[k]--; amt--; }
                if (++cnt > lim) return 3;
            }
        } else {
            int cnt = 0;
            while (amt > 0) {
                int gave = 0;
                for (int k = 0; k < nc; ++k) if (st[k] < od[k] + bt[k]) { st[k]++; amt--; gave = 1; }
                if (!gave) return 4;                     /* nobody can take a unit: the reference spins into its watchdog */
                if (++cnt > lim) return 4;
            }
        }
        for (int k = 0; k < nc; ++k) bt[k] += od[k] - st[k];
    }
    return 0;
}

/* One period.  actions [m]; cust [R] this period's customer demand; mask [m] or NULL.
 * reward_out: [m] (multi) or [1].  Returns the watchdog code. */
static int step_env(const orc_cfg* c, orc_state* s, int t, const double* actions, const int* cust, const unsigned char* mask,
                    double* reward_out, double* profit_out, int* order_out) {
    const int m = c->m, P = c->P, D = c->D;
    int order[ORC_MAX_NODES], demand[ORC_MAX_NODES], acq[ORC_MAX_NODES], ship[ORC_MAX_NODES], incoming[ORC_MAX_NODES];
    int new_carry[ORC_MAX_NODES];
    int err = 0;
    for (int i = 0; i < m; ++i) order[i] = decode_order(c, i, actions[i]);
    for (int i = 0; i < m; ++i) {
        if (c->retailer_idx[i] >= 0) {
            const int d = cust[c->retailer_idx[i]];
            demand[i] = d < c->inv_max[i] ? d : c->inv_max[i];
        } else if (c->div) {
            int sum = 0;
            for (int k = 0; k < c->nchild[i]; ++k) sum += order[c->children[i][k]];
            demand[i] = sum;
        } else {
            demand[i] = order[i - 1];
        }
    }
    for (int i = 0; i < m; ++i) {
        int a = s->carry[i];
        new_carry[i] = 0;
        if (t >= c->delay[i]) {
            a += s->pipe[i][0];
            if (mask && mask[i] && t < c->T - 1) { new_carry[i] = a; a = 0; }
        }
        acq[i] = a;
        const int lhs = s->backlog[i] + demand[i], rhs = s->inv[i] + a;
        ship[i] = lhs < rhs ? lhs : rhs;
    }
    if (c->div) {
        incoming[0] = order[0];
        for (int i = 0; i < m; ++i) {
            if (c->nchild[i] > 0) {
                int st[ORC_MAX_CHILDREN];
                const int code = split(c, s, i, ship[i], demand[i], s->backlog[i], order, st);
                if (code && !err) err = code;
                for (int k = 0; k < c->nchild[i]; ++k) incoming[c->children[i][k]] = st[k];
            }
        }
    } else {
        incoming[m - 1] = order[m - 1];
        for (int i = 0; i < m - 1; ++i) incoming[i] = ship[i + 1];
    }
    double profit[ORC_MAX_NODES];
    for (int i = 0; i < m; ++i) {
        int bl = s->backlog[i] + demand[i] - ship[i];
        if (c->cap_backlog) { const int cap = c->div ? c->demand_max[i] : c->inv_max[i]; bl = bl < cap ? bl : cap; }
        int ou = s->order_u[i] + order[i] - acq[i];
        ou = ou < 0 ? 0 : ou; ou = ou > c->inv_max[i] ? c->inv_max[i] : ou;
        int iv = s->inv[i] + acq[i] - ship[i];
        iv = iv < 0 ? 0 : iv; iv = iv > c->inv_max[i] ? c->inv_max[i] : iv;
        s->backlog[i] = bl; s->order_u[i] = ou; s->inv[i] = iv;
        for (int k = 0; k < D - 1; ++k) s->pipe[i][k] = s->pipe[i][k + 1];
        s->pipe[i][D - 1] = 0;
        s->pipe[i][c->delay[i] - 1] = incoming[i];
        for (int j = P - 1; j > 0; --j) { s->hd[i][j] = s->hd[i][j - 1]; s->ho[i][j] = s->ho[i][j - 1]; }
        s->hd[i][0] = demand[i]; s->ho[i][0] = order[i];
        s->carry[i] = new_carry[i];
        profit[i] = c->p[i] * (double)ship[i] - c->c[i] * (double)order[i] - c->h[i] * fabs((double)iv - c->target[i])
                    - c->bc[i] * (double)bl;
        if (profit_out) profit_out[i] = profit[i];
        if (order_out) order_out[i] = order[i];
    }
    if (c->multi) {
        if (c->independent) {
            for (int i = 0; i < m; ++i) reward_out[i] = profit[i];
        } else {
            double sum = 0.0;
            for (int i = 0; i < m; ++i) sum += profit[i];
            for (int i = 0; i < m; ++i) reward_out[i] = sum / (double)m;
        }
    } else {
        reward_out[0] = np_sum(profit, m);
    }
    return err;
}

static void store_state(const orc_cfg* c, const orc_state* s, long n, int L, int NB, int32_t* inv, int32_t* backlog, int32_t* order_u,
                        int32_t* pipe, int32_t* bt, int32_t* hd, int32_t* ho) {
    const int m = c->m;
    int po = 0, bo = 0;
    for (int i = 0; i < m; ++i) {
        if (inv) inv[n * m + i] = s->inv[i];
        if (backlog) backlog[n * m + i] = s->backlog[i];
        if (order_u) order_u[n * m + i] = s->order_u[i];
        if (pipe) for (int k = 0; k < c->delay[i]; ++k) pipe[n * L + po + k] = s->pipe[i][k];
        po += c->delay[i];
        if (bt && c->nchild[i] > 1) { for (int k = 0; k < c->nchild[i]; ++k) bt[n * NB + bo + k] = s->bt[i][k]; bo += c->nchild[i]; }
        if (hd) for (int j = 0; j < c->P; ++j) hd[(n * m + i) * c->P + j] = s->hd[i][j];
        if (ho) for (int j = 0; j < c->P; ++j) ho[(n * m + i) * c->P + j] = s->ho[i][j];
    }
}

/* Runs `periods` periods for N envs from the reset state.
 *   demand  [N][R][T] int32      actions [periods][N][m] f64     mask [N][T][m] uint8 or NULL
 *   obs_all [periods+1][N][m][O] or NULL;  obs_last [N][m][O] or NULL
 *   reward  [periods][N][cols] (cols = m for multi, 1 otherwise) or NULL
 *   final state arrays may be NULL.  Returns the number of envs whose watchdog fired. */
long orc_run(const orc_cfg* c, long N, int periods, const int32_t* demand, const double* actions, const unsigned char* mask,
             double* obs_all, double* obs_last, double* reward, int32_t* inv, int32_t* backlog, int32_t* order_u,
             int32_t* pipe, int32_t* bt, int32_t* hd, int32_t* ho, int32_t* err, int nthreads) {
    const int m = c->m, O = c->O, T = c->T, R = c->R;
    const int cols = c->multi ? m : 1;
    int L = 0, NB = 0;
    for (int i = 0; i < m; ++i) { L += c->delay[i]; if (c->nchild[i] > 1) NB += c->nchild[i]; }
    long bad = 0;
#ifdef _OPENMP
    if (nthreads > 0) omp_set_num_threads(nthreads);
#endif
#pragma omp parallel for schedule(static) reduction(+ : bad)
    for (long n = 0; n < N; ++n) {
        orc_state s;
        reset_state(c, &s);
        double obs[ORC_MAX_NODES * 64];
        double rew[ORC_MAX_NODES];
        int cust[ORC_MAX_NODES];
        int e = 0;
        if (obs_all) { observe(c, &s, 0, obs); memcpy(obs_all + (size_t)n * m * O, obs, sizeof(double) * m * O); }
        for (int t = 0; t < periods; ++t) {
            for (int r = 0; r < R; ++r) cust[r] = demand[((size_t)n * R + r) * T + t];
            const int code = step_env(c, &s, t, actions + ((size_t)t * N + n) * m, cust, mask ? mask + ((size_t)n * T + t) * m : NULL,
                                      rew, NULL, NULL);
            if (code && !e) e = code;
            if (reward) memcpy(reward + ((size_t)t * N + n) * cols, rew, sizeof(double) * cols);
            if (obs_all) { observe(c, &s, t + 1, obs); memcpy(obs_all + ((size_t)(t + 1) * N + n) * m * O, obs, sizeof(double) * m * O); }
        }
        if (obs_last) { observe(c, &s, periods, obs); memcpy(obs_last + (size_t)n * m * O, obs, sizeof(double) * m * O); }
        store_state(c, &s, n, L, NB, inv, backlog, order_u, pipe, bt, hd, ho);
        if (err) err[n] = e;
        if (e) bad += 1;
    }
    return bad;
}

/* Base-stock rollout (dfo_func's loop): z [m] (z_stride 0) or [N][m]; demand [N][R][T]; mask [N][T][m] or NULL;
 * ret [N][cols]; step_reward [T][N][cols] or NULL; pmf [N][R][T] + dfo [N] or NULL (np.sum over the flattened
 * [R][T] product of pmf and the per-period rewards, base_restock_policy.py:41-45). */
long orc_rollout(const orc_cfg* c, long N, const double* z, int z_stride, const int32_t* demand, const unsigned char* mask,
                 const double* pmf, double* ret, double* step_reward, double* dfo, int32_t* inv, int32_t* backlog, int32_t* order_u,
                 int32_t* pipe, int32_t* bt, int nthreads) {
    const int m = c->m, T = c->T, R = c->R;
    const int cols = c->multi ? m : 1;
    int L = 0, NB = 0;
    for (int i = 0; i < m; ++i) { L += c->delay[i]; if (c->nchild[i] > 1) NB += c->nchild[i]; }
    long bad = 0;
#ifdef _OPENMP
    if (nthreads > 0) omp_set_num_threads(nthreads);
#endif
#pragma omp parallel for schedule(static) reduction(+ : bad)
    for (long n = 0; n < N; ++n) {
        orc_state s;
        reset_state(c, &s);
        double act[ORC_MAX_NODES], rew[ORC_MAX_NODES], acc[ORC_MAX_NODES];
        double* rew_t = dfo ? (double*)malloc(sizeof(double) * (size_t)T) : NULL;
        int cust[ORC_MAX_NODES];
        int e = 0;
        for (int k = 0; k < cols; ++k) acc[k] = 0.0;
        const double* zz = z + (z_stride ? (size_t)n * m : 0);
        for (int t = 0; t < T; ++t) {
            for (int i = 0; i < m; ++i) {        /* base_restock_policy.py:12-20 */
                const double inv_ech = (double)s.inv[i] + (double)s.order_u[i] - (double)s.backlog[i];
                double u = zz[i] - inv_ech;
                u = u > 0.0 ? u : 0.0;
                act[i] = (double)c->order_max[i] < u ? (double)c->order_max[i] : u;
            }
            for (int r = 0; r < R; ++r) cust[r] = demand[((size_t)n * R + r) * T + t];
            const int code = step_env(c, &s, t, act, cust, mask ? mask + ((size_t)n * T + t) * m : NULL, rew, NULL, NULL);
            if (code && !e) e = code;
            for (int k = 0; k < cols; ++k) acc[k] += rew[k];
            if (step_reward) memcpy(step_reward + ((size_t)t * N + n) * cols, rew, sizeof(double) * cols);
            if (dfo) rew_t[t] = rew[0];
        }
        memcpy(ret + (size_t)n * cols, acc, sizeof(double) * cols);
        if (dfo) {
            double* prod = (double*)malloc(sizeof(double) * (size_t)R * T);
            for (int r = 0; r < R; ++r)
                for (int t = 0; t < T; ++t) prod[(size_t)r * T + t] = pmf[((size_t)n * R + r) * T + t] * rew_t[t];
            dfo[n] = (-1.0 / (double)T) * np_sum(prod, R * T);
            free(prod);
            free(rew_t);
        }
        store_state(c, &s, n, L, NB, inv, backlog, order_u, pipe, bt, NULL, NULL);
        if (e) bad += 1;
    }
    return bad;
}

int orc_max_threads(void) {
#ifdef _OPENMP
    return omp_get_max_threads();
#else
    return 1;
#endif
}
