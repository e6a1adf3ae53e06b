/*
 * yagre_oracle.c -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.
 *
 * Plain-C, scalar, one-chain-at-a-time CPU restatement of the reference's
 * (rkutri/yagre-mcmc, pure Python) Metropolis-Hastings hot path.  Only tests/,
 * __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs
 * may load this library, and only as the checker / the CPU arm -- never as a
 * fallback of the product path.
 *
 * Parity status: PINNED for MRW and two-level MLDA on the Gaussian, linear and
 * Lotka-Volterra(RK4) problems against tests/golden/ fixtures, which were produced
 * by the unmodified reference under injected noise (oracle/make_golden.py;
 * the RK4 forward model is our SolverInterface plugin because the reference
 * integrates with scipy.solve_ivp -- see oracle/ref_harness.py).  PINNED for
 * Welford, IAT and dense-covariance operators against postprocessing.npz.
 * PINNED for adaptive Metropolis against tests/golden/am_*.npz: the unmodified
 * AdaptiveMRWProposal + MetropolisHastings.run (chain/adaptive.py:37-64) driving our concrete
 * AdaptiveCovarianceMatrix (oracle/ref_harness.py; the reference ships only the abstract class,
 * so the recurrence is ours, its call order / swap semantics / Cholesky are the reference's).
 * UNPINNED for split-R-hat (absent from the reference; checked against numpy).
 *
 * Compile with -ffp-contract=off: the reference is numpy (unfused arithmetic).
 *
 * Reference lines each function follows are cited at the function.
 */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>
#ifdef _OPENMP
#include <omp.h>
#endif

enum { YO_GAUSS = 0, YO_LINEAR = 1, YO_LV = 2 };
enum { YO_EQ_EXACT = 0, YO_EQ_ISCLOSE = 1 };
#define YO_MAX_DIM 64
#define YO_MAX_DATA 256

typedef struct yo_level {
    /* explicit Gaussian target: logp = -0.5 (t-m)' P (t-m) + logconst (testSetup.py:15-44) */
    const double *g_mean;      /* [d]   */
    const double *g_prec;      /* [d,d] */
    double g_logconst;
    /* regression posterior = likelihood + prior (chain/target.py:19-22) */
    int32_t n_data, data_dim;
    const double *data;        /* [n_data, data_dim] (statistics/data.py) */
    const double *noise_prec;  /* [data_dim, data_dim]; exact zeros are skipped */
    const double *prior_mean;  /* [d] */
    const double *prior_prec;  /* [d,d] */
    const double *G;           /* [data_dim, d]  exampleSetup.py:46 */
    const double *b;           /* [data_dim] */
    const double *design;      /* [n_data, 2]    testSetup.py:118-141 */
    double alpha, gamma, T;
    int32_t rk4_steps;
    int32_t tempered;          /* TemperedUnnormalisedPosterior (chain/target.py:25-43) */
    double tempering;
} yo_level;

typedef struct yo_problem {
    int32_t model, dim, n_levels, J, eq_mode, _pad;
    const double *prop_L;      /* [d,d] lower triangular, p = s + L z (gaussian.py:61-66) */
    /* level[n_levels-1] is the target; n_levels == 3 is MLDA with two surrogates AS THE REFERENCE RUNS
     * IT (mlda.py:12-43,60-71,112-117): MRW sub-chain of J = subChainLengths[1] steps on level[0],
     * screen with the finest surrogate level[1] */
    yo_level level[3];
    /* adaptive Metropolis (am_update below; pinned by tests/golden/am_*.npz) */
    int32_t adaptive, am_refresh;
    int64_t am_idle, am_collect;
    double am_eps, am_scale;
    /* preconditioned Crank-Nicolson (chain/method/pcn.py:9-57): prop_L is the PRIOR's factor,
     * p = sqrt(1-2h) s + sqrt(2h) (m + L z); the target is the likelihood alone */
    int32_t pcn, _pad2;
    double pcn_a, pcn_b;       /* sqrt(1 - 2h), sqrt(2h) */
    const double *pcn_mean;    /* [d] prior mean (zeros: pcn.py:44-46) */
    /* adaptive error model (chain/method/aem.py, statistics/likelihood.py:90-155, noise.py:25-61):
     * two levels, linear forward model, diagonal measurement noise */
    int32_t aem, aem_min_data, aem_heuristic, _pad3;
} yo_problem;

/* ---------------------------------------------------------------------- */
/* numpy's pairwise summation (np.sum over a contiguous double vector),   */
/* as used by likelihood.py:80 on the per-row norms.                      */
/* ---------------------------------------------------------------------- */
static double np_pairwise_sum(const double *a, long n)
{
    if (n < 8) {
        double res = 0.0;
        for (long i = 0; i < n; i++) res += a[i];
        return res;
    } else if (n <= 128) {
        double r[8];
        long i;
        for (i = 0; i < 8; i++) r[i] = a[i];
        for (i = 8; i < n - (n % 8); i += 8)
            for (int k = 0; k < 8; k++) r[k] += a[i + k];
        double res = ((r[0] + r[1]) + (r[2] + r[3])) + ((r[4] + r[5]) + (r[6] + r[7]));
        for (; i < n; i++) res += a[i];
        return res;
    } else {
        long n2 = n / 2;
        n2 -= n2 % 8;
        return np_pairwise_sum(a, n2) + np_pairwise_sum(a + n2, n - n2);
    }
}

/* x' P x with P applied first (covariance.py:19-22: Px = apply_inverse(x); dot(x, Px)).
 * Exact zeros of P are skipped so a diagonal precision behaves exactly like
 * DiagonalCovarianceMatrix (prec * x, covariance.py:54-55) even for x = inf. */
static double quad_form(const double *P, const double *x, int n)
{
    double acc = 0.0;
    for (int k = 0; k < n; k++) {
        double pk = 0.0;
        int first = 1;
        for (int l = 0; l < n; l++) {
            double p = P[k * n + l];
            if (p != 0.0) {
                double t = p * x[l];
                pk = first ? t : pk + t;
                first = 0;
            }
        }
        double t = x[k] * pk;
        acc = (k == 0) ? t : acc + t;
    }
    return acc;
}

/* ---------------------------------------------------------------------- */
/* forward models                                                         */
/* ---------------------------------------------------------------------- */

/* One LV integration; arithmetic order of oracle/ref_harness.py
 * RK4LotkaVolterraSolver.invoke (flow association: testSetup.py:98-99). */
static void lv_rk4(double alpha, double beta, double gamma, double delta,
                   double T, int N, double *px, double *py)
{
    double x = *px, y = *py;
    const double h = T / (double)N, h2 = 0.5 * h, h6 = h / 6.0;
    for (int i = 0; i < N; i++) {
        double k1x = alpha * x - beta * x * y,        k1y = delta * x * y - gamma * y;
        double xa = x + h2 * k1x,                     ya = y + h2 * k1y;
        double k2x = alpha * xa - beta * xa * ya,     k2y = delta * xa * ya - gamma * ya;
        double xb = x + h2 * k2x,                     yb = y + h2 * k2y;
        double k3x = alpha * xb - beta * xb * yb,     k3y = delta * xb * yb - gamma * yb;
        double xc = x + h * k3x,                      yc = y + h * k3y;
        double k4x = alpha * xc - beta * xc * yc,     k4y = delta * xc * yc - gamma * yc;
        x = x + h6 * (((k1x + 2.0 * k2x) + 2.0 * k3x) + k4x);
        y = y + h6 * (((k1y + 2.0 * k2y) + 2.0 * k3y) + k4y);
    }
    *px = isfinite(x) ? x : INFINITY;
    *py = isfinite(y) ? y : INFINITY;
}

/* chain/target.py:19-22 -> likelihood.py:33-39,74-84 + gaussian.py:19-24 */
double yo_logpost(const yo_problem *pb, int lvl, const double *theta, int64_t *n_evals)
{
    const yo_level *L = &pb->level[lvl];
    const int d = pb->dim;
    double x[YO_MAX_DIM];
    if (n_evals) (*n_evals)++;
    if (pb->model == YO_GAUSS) {
        for (int i = 0; i < d; i++) x[i] = theta[i] - L->g_mean[i];
        return -0.5 * quad_form(L->g_prec, x, d) + L->g_logconst;
    }
    const int nD = L->n_data, dd = L->data_dim;
    double *q = (double *)malloc(sizeof(double) * (size_t)nD);
    double r[YO_MAX_DATA], F[YO_MAX_DATA];
    if (pb->model == YO_LINEAR) {
        for (int k = 0; k < dd; k++) {               /* A @ theta + b  (exampleSetup.py:46) */
            double acc = 0.0;
            for (int j = 0; j < d; j++) {
                double t = L->G[k * d + j] * theta[j];
                acc = (j == 0) ? t : acc + t;
            }
            F[k] = acc + L->b[k];
        }
        for (int n = 0; n < nD; n++) {               /* broadcast against rows (likelihood.py:74-75) */
            for (int k = 0; k < dd; k++) r[k] = F[k] - L->data[n * dd + k];
            q[n] = quad_form(L->noise_prec, r, dd);
        }
    } else {                                          /* YO_LV */
        const double beta = exp(theta[0]), delta = exp(theta[1]);   /* testSetup.py:57-58,101-107 */
        for (int n = 0; n < nD; n++) {
            double X = L->design[2 * n], Y = L->design[2 * n + 1];
            lv_rk4(L->alpha, beta, L->gamma, delta, L->T, L->rk4_steps, &X, &Y);
            r[0] = X - L->data[2 * n];
            r[1] = Y - L->data[2 * n + 1];
            q[n] = quad_form(L->noise_prec, r, 2);
        }
    }
    double logL = -0.5 * np_pairwise_sum(q, nD);      /* likelihood.py:80 */
    free(q);
    if (L->tempered) logL = L->tempering * logL;      /* target.py:40-43 */
    for (int i = 0; i < d; i++) x[i] = theta[i] - L->prior_mean[i];
    double lp = -0.5 * quad_form(L->prior_prec, x, d); /* gaussian.py:19-24 */
    return logL + lp;
}

/* ---------------------------------------------------------------------- */
/* step primitives                                                        */
/* ---------------------------------------------------------------------- */

/* statistics/gaussian.py:61-66, covariance.py:51-52,84-86 */
static void propose(const yo_problem *pb, const double *L, const double *s, const double *z, double *p)
{
    const int d = pb->dim;
    for (int i = 0; i < d; i++) {
        double acc = 0.0;
        int first = 1;
        for (int j = 0; j <= i; j++) {
            double l = L[i * d + j];
            if (l != 0.0 || j == i) {
                double t = l * z[j];
                acc = first ? t : acc + t;
                first = 0;
            }
        }
        if (pb->pcn) {
            /* pcn.py:30-35: xi = mean + L z (gaussian.py:63-66), sqrt(1-t)*state + sqrt(t)*xi */
            double xi = (pb->pcn_mean ? pb->pcn_mean[i] : 0.0) + acc;
            p[i] = pb->pcn_a * s[i] + pb->pcn_b * xi;
        } else {
            p[i] = s[i] + acc;
        }
    }
}

/* parameter/vector.py:37-45 (array_equal) and parameter/scalar.py:38-43 (math.isclose) */
static int param_equal(const yo_problem *pb, const double *a, const double *b)
{
    if (pb->eq_mode == YO_EQ_ISCLOSE) {
        double x = a[0], y = b[0];
        if (x == y) return 1;
        if (isinf(x) || isinf(y)) return 0;
        double diff = fabs(y - x);
        return (diff <= fabs(1e-9 * y)) || (diff <= fabs(1e-9 * x)) || (diff <= 0.0);
    }
    for (int i = 0; i < pb->dim; i++)
        if (!(a[i] == b[i])) return 0;
    return 1;
}

/* mrw.py:54-57 / mlda.py:148-154 + metropolisHastings.py:68-73.
 * NaN ratio: (r < 1.) is false -> a = 1 -> accepted. */
static int accept_rule(double delta, double u)
{
    double r = exp(delta);
    double a = (r < 1.0) ? r : 1.0;
    return u <= a;
}

/* ---------------------------------------------------------------------- */
/* Philox4x32-10 (Salmon, Moraes, Dror, Shaw, SC'11; Random123 v1.14)     */
/* ---------------------------------------------------------------------- */
void yo_philox4x32_10(const uint32_t ctr[4], const uint32_t key[2], uint32_t out[4])
{
    uint32_t c0 = ctr[0], c1 = ctr[1], c2 = ctr[2], c3 = ctr[3];
    uint32_t k0 = key[0], k1 = key[1];
    for (int r = 0; r < 10; r++) {
        uint64_t p0 = (uint64_t)0xD2511F53u * c0;
        uint64_t p1 = (uint64_t)0xCD9E8D57u * c2;
        uint32_t n0 = (uint32_t)(p1 >> 32) ^ c1 ^ k0;
        uint32_t n1 = (uint32_t)p1;
        uint32_t n2 = (uint32_t)(p0 >> 32) ^ c3 ^ k1;
        uint32_t n3 = (uint32_t)p0;
        c0 = n0; c1 = n1; c2 = n2; c3 = n3;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
    out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}

/* Stream keying shared with the CUDA kernels (DESIGN.md "Noise streams"):
 *   key = (seed lo, seed hi)
 *   ctr = (chain lo32, step lo32, step hi32, chain_hi8<<24 | sub<<8 | slot)
 *   sub  = coarse sub-step j, or 0xFFFF for the fine / single-level screen
 *   slot = b for the b-th pair of normals, 0xFF for the accept uniform */
#define YO_SUB_FINE 0xFFFFu
#define YO_SLOT_U 0xFFu
static void philox_block(uint64_t seed, uint64_t chain, uint64_t step, uint32_t sub, uint32_t slot,
                         uint32_t out[4])
{
    uint32_t key[2] = { (uint32_t)seed, (uint32_t)(seed >> 32) };
    uint32_t ctr[4] = { (uint32_t)chain, (uint32_t)step, (uint32_t)(step >> 32),
                        (uint32_t)(((chain >> 32) & 0xFFu) << 24) | (sub << 8) | slot };
    yo_philox4x32_10(ctr, key, out);
}

static double u53(uint32_t hi, uint32_t lo)
{
    return (double)((((uint64_t)hi << 32) | lo) >> 11) * 0x1.0p-53;
}

double yo_philox_uniform(uint64_t seed, uint64_t chain, uint64_t step, uint32_t sub)
{
    uint32_t w[4];
    philox_block(seed, chain, step, sub, YO_SLOT_U, w);
    return u53(w[0], w[1]);                                   /* [0,1) like numpy's uniform */
}

void yo_philox_normals(uint64_t seed, uint64_t chain, uint64_t step, uint32_t sub, int d, double *z)
{
    for (int b = 0; 2 * b < d; b++) {                         /* Box-Muller, one block per pair */
        uint32_t w[4];
        philox_block(seed, chain, step, sub, (uint32_t)b, w);
        double u1 = u53(w[0], w[1]) + 0x1.0p-53;              /* (0,1] */
        double u2 = u53(w[2], w[3]);
        double R = sqrt(-2.0 * log(u1));
        double a = 6.283185307179586476925286766559 * u2;
        z[2 * b] = R * cos(a);
        if (2 * b + 1 < d) z[2 * b + 1] = R * sin(a);
    }
}

/* ---------------------------------------------------------------------- */
/* one chain                                                              */
/* ---------------------------------------------------------------------- */
typedef struct {
    const double *z, *u_c, *u_f;   /* injected noise for this chain, or NULL -> Philox */
    uint64_t seed, chain_id, step0;
} noise_src;

static void get_z(const yo_problem *pb, const noise_src *ns, int64_t n, int j, double *z)
{
    const int d = pb->dim;
    if (ns->z) memcpy(z, ns->z + ((size_t)n * pb->J + j) * d, sizeof(double) * d);
    else yo_philox_normals(ns->seed, ns->chain_id, ns->step0 + (uint64_t)n, (uint32_t)j, d, z);
}
static double get_uc(const yo_problem *pb, const noise_src *ns, int64_t n, int j)
{
    if (ns->z) return ns->u_c[(size_t)n * pb->J + j];
    return yo_philox_uniform(ns->seed, ns->chain_id, ns->step0 + (uint64_t)n, (uint32_t)j);
}
static double get_uf(const noise_src *ns, int64_t n)
{
    if (ns->z) return ns->u_f[n];
    return yo_philox_uniform(ns->seed, ns->chain_id, ns->step0 + (uint64_t)n, YO_SUB_FINE);
}

typedef struct {
    double theta[YO_MAX_DIM];
    double lp[3];                  /* log-posterior of theta per level */
    int64_t n_accept;
    int64_t n_coarse_accept;       /* accepted coarse sub-steps (the device's coarse_accepted counter) */
    int64_t n_evals[3];
    int64_t w_n;                   /* Welford (estimation.py:36-53), fed the PRE-transition state */
    double w_mean[YO_MAX_DIM], w_m2[YO_MAX_DIM];
    /* adaptive Metropolis: full-matrix Welford of the states from step am_idle on + current factor */
    double am_mean[YO_MAX_DIM], am_m2[YO_MAX_DIM * YO_MAX_DIM], L[YO_MAX_DIM * YO_MAX_DIM];
    /* adaptive error model: Welford of F_f - F_c on accepted fine steps (estimation.py:36-53), the
     * inflated noise precision, and the coarse likelihood's LRU(3) cache of (parameter -> logL)
     * (utility/memoisation.py:76-149), entries ordered oldest .. newest */
    int64_t aem_n;
    double aem_mean[YO_MAX_DATA], aem_m2[YO_MAX_DATA], aem_prec[YO_MAX_DATA];
    int aem_have_noise, lru_n;
    double lru_key[3][YO_MAX_DIM], lru_ll[3];
    int64_t aem_model_evals;
} chain_state;

int yo_cholesky(const double *C, int d, double *L);

/* chain/adaptive.py:55-60: update() runs in AdaptiveMRWProposal.set_state(), i.e. BEFORE each
 * proposal of the MRW chain it drives, with that chain's current state x: the chain state for a
 * single level, the sub-chain state for the coarse MRW of two-level delayed acceptance.  t_idx =
 * number of update() calls before this one.  The recurrence (Welford, C = s (Cov + eps I) once
 * am_collect states were collected) is ours; its arithmetic is pinned to oracle/ref_harness.py
 * HaarioAdaptiveCovariance driven by the unmodified reference (tests/golden/am_*.npz). */
static void am_update(const yo_problem *pb, chain_state *cs, const double *x, int64_t t_idx)
{
    const int d = pb->dim;
    if (t_idx < pb->am_idle) return;
    const int64_t n_am = t_idx - pb->am_idle + 1;
    double dl[YO_MAX_DIM], e[YO_MAX_DIM];
    for (int i = 0; i < d; i++) {
        dl[i] = x[i] - cs->am_mean[i];
        cs->am_mean[i] += dl[i] / (double)n_am;
        e[i] = x[i] - cs->am_mean[i];
    }
    for (int i = 0; i < d; i++)
        for (int j = 0; j < d; j++) cs->am_m2[i * d + j] += dl[i] * e[j];
    if (n_am >= pb->am_collect && n_am >= 2 && ((n_am - pb->am_collect) % pb->am_refresh) == 0) {
        double C[YO_MAX_DIM * YO_MAX_DIM], Ln[YO_MAX_DIM * YO_MAX_DIM];
        for (int i = 0; i < d; i++)
            for (int j = 0; j < d; j++) {
                double cov = 0.5 * (cs->am_m2[i * d + j] + cs->am_m2[j * d + i]) / (double)(n_am - 1);
                C[i * d + j] = pb->am_scale * (cov + ((i == j) ? pb->am_eps : 0.0));
            }
        if (yo_cholesky(C, d, Ln) == 0) memcpy(cs->L, Ln, sizeof(double) * d * d);
    }
}

static void welford_update(chain_state *cs, int d)
{
    cs->w_n += 1;
    for (int i = 0; i < d; i++) {
        double delta = cs->theta[i] - cs->w_mean[i];
        cs->w_mean[i] += delta / (double)cs->w_n;
        double delta2 = cs->theta[i] - cs->w_mean[i];
        cs->w_m2[i] += delta * delta2;
    }
}


/* ---------------------------------------------------------------------- */
/* adaptive error model                                                   */
/* ---------------------------------------------------------------------- */
static int lru_find(const yo_problem *pb, const chain_state *cs, const double *x)
{
    for (int i = 0; i < cs->lru_n; i++) {
        int eq = 1;
        for (int k = 0; k < pb->dim; k++) eq = eq && (cs->lru_key[i][k] == x[k]);   /* vector.py:37-45 */
        if (eq) return i;
    }
    return -1;
}
/* AEMCache._move_to_back (memoisation.py:95-100) */
static void lru_touch(const yo_problem *pb, chain_state *cs, int idx)
{
    double key[YO_MAX_DIM], ll = cs->lru_ll[idx];
    memcpy(key, cs->lru_key[idx], sizeof(double) * pb->dim);
    for (int i = idx; i + 1 < cs->lru_n; i++) {
        memcpy(cs->lru_key[i], cs->lru_key[i + 1], sizeof(double) * pb->dim);
        cs->lru_ll[i] = cs->lru_ll[i + 1];
    }
    memcpy(cs->lru_key[cs->lru_n - 1], key, sizeof(double) * pb->dim);
    cs->lru_ll[cs->lru_n - 1] = ll;
}
/* AEMCache.add (memoisation.py:102-116): evict the oldest of three */
static void lru_add(const yo_problem *pb, chain_state *cs, const double *x, double ll)
{
    if (cs->lru_n >= 3) {
        for (int i = 0; i + 1 < 3; i++) {
            memcpy(cs->lru_key[i], cs->lru_key[i + 1], sizeof(double) * pb->dim);
            cs->lru_ll[i] = cs->lru_ll[i + 1];
        }
        cs->lru_n = 2;
    }
    memcpy(cs->lru_key[cs->lru_n], x, sizeof(double) * pb->dim);
    cs->lru_ll[cs->lru_n] = ll;
    cs->lru_n++;
}
static void linear_forward(const yo_level *L, int d, const double *theta, double *F)
{
    for (int k = 0; k < L->data_dim; k++) {          /* A @ theta + b  (exampleSetup.py:46) */
        double acc = 0.0;
        for (int j = 0; j < d; j++) {
            double t = L->G[k * d + j] * theta[j];
            acc = (j == 0) ? t : acc + t;
        }
        F[k] = acc + L->b[k];
    }
}
/* AEMLikelihood.compute_log_likelihood (likelihood.py:74-84,140-145) + prior (target.py:19-22) */
static double aem_coarse_logpost(const yo_problem *pb, chain_state *cs, const double *x)
{
    const yo_level *L = &pb->level[0];
    const int d = pb->dim, dd = L->data_dim;
    double F[YO_MAX_DATA], q[64];
    linear_forward(L, d, x, F);
    cs->aem_model_evals++;
    for (int n = 0; n < L->n_data; n++) {
        double acc = 0.0;
        for (int k = 0; k < dd; k++) {
            double r = F[k] - L->data[n * dd + k];
            if (cs->aem_n >= pb->aem_min_data) r = r + cs->aem_mean[k];              /* likelihood.py:140-145 */
            const double prec = cs->aem_have_noise ? cs->aem_prec[k] : L->noise_prec[k * dd + k];
            const double t = r * (prec * r);                                         /* covariance.py:19-22,54-55 */
            acc = (k == 0) ? t : acc + t;
        }
        q[n] = acc;
    }
    const double logL = -0.5 * np_pairwise_sum(q, L->n_data);
    double xx[YO_MAX_DIM];
    for (int i = 0; i < d; i++) xx[i] = x[i] - L->prior_mean[i];
    return logL + (-0.5 * quad_form(L->prior_prec, xx, d));
}
/* AEMLikelihood.query_log_likelihood (likelihood.py:126-131): a cached value is NOT invalidated
 * when the error model changes */
static double aem_query_coarse(const yo_problem *pb, chain_state *cs, const double *x)
{
    /* the cache stores logL; the prior term is deterministic, so caching the sum is equivalent */
    int idx = lru_find(pb, cs, x);
    if (idx >= 0) {
        const double ll = cs->lru_ll[idx];
        lru_touch(pb, cs, idx);
        return ll;
    }
    const double lp = aem_coarse_logpost(pb, cs, x);
    lru_add(pb, cs, x, lp);
    return lp;
}
/* AdaptiveErrorModel._process_transition on an accepted fine step (aem.py:25-58) +
 * AEMLikelihood.update_error_estimate (likelihood.py:147-155) + AEMNoise (noise.py:41-54) */
static void aem_update(const yo_problem *pb, chain_state *cs, const double *P)
{
    const yo_level *Lc = &pb->level[0], *Lf = &pb->level[1];
    const int d = pb->dim, dd = Lc->data_dim;
    double Fc[YO_MAX_DATA], Ff[YO_MAX_DATA];
    int idx = lru_find(pb, cs, P);                    /* query_model_evaluation: a hit moves the entry back */
    if (idx >= 0) lru_touch(pb, cs, idx); else cs->aem_model_evals++;
    linear_forward(Lc, d, P, Fc);
    linear_forward(Lf, d, P, Ff);
    cs->aem_n++;
    for (int k = 0; k < dd; k++) {                    /* Welford, estimation.py:36-53 */
        const double e = Ff[k] - Fc[k];
        const double delta = e - cs->aem_mean[k];
        cs->aem_mean[k] += delta / (double)cs->aem_n;
        cs->aem_m2[k] += delta * (e - cs->aem_mean[k]);
    }
    if (cs->aem_n > pb->aem_min_data) {
        double mv[YO_MAX_DATA], mn = INFINITY, mx = -INFINITY;
        for (int k = 0; k < dd; k++) {
            mv[k] = cs->aem_m2[k] / (double)(cs->aem_n - 1);
            if (mv[k] < mn) mn = mv[k];
            if (mv[k] > mx) mx = mv[k];
        }
        double scaling = 1.0;
        if (pb->aem_heuristic) {                      /* noise.py:41-46 */
            const double minVal = mn > 1e-6 ? mn : 1e-6;
            scaling = 2. * mx / minVal;
            if (scaling > 100.) scaling = 100.;
        }
        for (int k = 0; k < dd; k++) {
            const double dataVar = 1.0 / Lc->noise_prec[k * dd + k];     /* covariance.py:33-34 */
            cs->aem_prec[k] = 1.0 / (scaling * mv[k] + dataVar);         /* noise.py:51-53, covariance.py:37-38 */
        }
        cs->aem_have_noise = 1;
    }
}

/* One AEM transition (two level): aem.py + mlda.py:100-110,146-154 with the coarse likelihood's
 * cache semantics.  Returns 1 if accepted. */
static int chain_step_aem(const yo_problem *pb, chain_state *cs, const noise_src *ns, int64_t n)
{
    const int d = pb->dim;
    double z[YO_MAX_DIM], p[YO_MAX_DIM], s[YO_MAX_DIM];
    welford_update(cs, d);
    memcpy(s, cs->theta, sizeof(double) * d);
    for (int j = 0; j < pb->J; j++) {
        get_z(pb, ns, n, j, z);
        propose(pb, cs->L, s, z, p);
        if (param_equal(pb, p, s)) continue;
        const double lpp = aem_query_coarse(pb, cs, p);      /* mrw.py:53: proposal first, then state */
        const double lps = aem_query_coarse(pb, cs, s);
        if (accept_rule(lpp - lps, get_uc(pb, ns, n, j))) {
            memcpy(s, p, sizeof(double) * d);
            cs->n_coarse_accept++;
        }
    }
    if (param_equal(pb, s, cs->theta)) return 0;
    /* mlda.py:148-152: pi_f(P) + pi_c(theta) - pi_c(P) - pi_f(theta), evaluated in this order */
    const double lpf_s = yo_logpost(pb, 1, s, &cs->n_evals[1]);
    const double lpc_t = aem_query_coarse(pb, cs, cs->theta);
    const double lpc_s = aem_query_coarse(pb, cs, s);
    const double delta = lpf_s + lpc_t - lpc_s - cs->lp[1];
    if (accept_rule(delta, get_uf(ns, n))) {
        aem_update(pb, cs, s);
        memcpy(cs->theta, s, sizeof(double) * d);
        cs->lp[1] = lpf_s;
        cs->n_accept++;
        return 1;
    }
    return 0;
}

static void chain_init(const yo_problem *pb, chain_state *cs, const double *theta0)
{
    memset(cs, 0, sizeof(*cs));
    memcpy(cs->theta, theta0, sizeof(double) * pb->dim);
    memcpy(cs->L, pb->prop_L, sizeof(double) * pb->dim * pb->dim);
    for (int l = 0; l < pb->n_levels; l++)
        cs->lp[l] = yo_logpost(pb, l, cs->theta, &cs->n_evals[l]);
}

/* One transition.  Single level: metropolisHastings.py:112-120 with mrw.py.
 * Two level: mlda.py:100-110 (sub-chain) + mlda.py:146-154 (screen);
 * SURVEY Appendix A.  Returns 1 if accepted. */
static int chain_step(const yo_problem *pb, chain_state *cs, const noise_src *ns, int64_t n)
{
    const int d = pb->dim;
    double z[YO_MAX_DIM], p[YO_MAX_DIM];
    if (pb->aem) return chain_step_aem(pb, cs, ns, n);
    welford_update(cs, d);                               /* diagnostics.py:91-94 */
    if (pb->n_levels == 1) {
        if (pb->adaptive) am_update(pb, cs, cs->theta, n);        /* n counts from chain_init, where the moments were reset */
        get_z(pb, ns, n, 0, z);
        propose(pb, cs->L, cs->theta, z, p);
        if (param_equal(pb, p, cs->theta)) return 0;     /* metropolisHastings.py:60-61 */
        double lpp = yo_logpost(pb, 0, p, &cs->n_evals[0]);
        if (accept_rule(lpp - cs->lp[0], get_uf(ns, n))) {
            memcpy(cs->theta, p, sizeof(double) * d);
            cs->lp[0] = lpp;
            cs->n_accept++;
            return 1;
        }
        return 0;
    }
    double s[YO_MAX_DIM], lpc_s = cs->lp[0];
    memcpy(s, cs->theta, sizeof(double) * d);
    for (int j = 0; j < pb->J; j++) {                    /* coarse MRW sub-chain */
        if (pb->adaptive) am_update(pb, cs, s, n * pb->J + j);
        get_z(pb, ns, n, j, z);
        propose(pb, cs->L, s, z, p);
        if (param_equal(pb, p, s)) continue;
        double lpp = yo_logpost(pb, 0, p, &cs->n_evals[0]);
        if (accept_rule(lpp - lpc_s, get_uc(pb, ns, n, j))) {
            memcpy(s, p, sizeof(double) * d);
            lpc_s = lpp;
            cs->n_coarse_accept++;
        }
    }
    if (param_equal(pb, s, cs->theta)) return 0;         /* no fine evaluation, no uniform */
    if (pb->n_levels == 3) {
        /* two surrogates: MLDA._acceptance_probability (mlda.py:146-154) with _finestTarget = level 1,
         * while the sub-chain above ran on level 0 (SurrogateTransition.generate_proposal, mlda.py:23-33) */
        double lpt_s = yo_logpost(pb, 2, s, &cs->n_evals[2]);
        double lpm_s = yo_logpost(pb, 1, s, &cs->n_evals[1]);
        double delta = lpt_s + cs->lp[1] - lpm_s - cs->lp[2];
        if (accept_rule(delta, get_uf(ns, n))) {
            memcpy(cs->theta, s, sizeof(double) * d);
            cs->lp[0] = lpc_s; cs->lp[1] = lpm_s; cs->lp[2] = lpt_s;
            cs->n_accept++;
            return 1;
        }
        return 0;
    }
    double lpf_s = yo_logpost(pb, 1, s, &cs->n_evals[1]);
    double delta = lpf_s + cs->lp[0] - lpc_s - cs->lp[1]; /* mlda.py:148-152, this order */
    if (accept_rule(delta, get_uf(ns, n))) {
        memcpy(cs->theta, s, sizeof(double) * d);
        cs->lp[0] = lpc_s;
        cs->lp[1] = lpf_s;
        cs->n_accept++;
        return 1;
    }
    return 0;
}

/* ---------------------------------------------------------------------- */
/* exported drivers                                                       */
/* ---------------------------------------------------------------------- */

/* Injected-noise run, chain-major layouts:
 *   theta0[nc,d]  z[nc,ns,J,d]  u_c[nc,ns,J]  u_f[nc,ns]
 *   traj[nc,ns+1,d]  accepted[nc,ns]  lp0/lp1[nc,ns+1]  w_mean/w_var[nc,d] */
int yo_run_injected(const yo_problem *pb, int64_t nc, int64_t ns,
                    const double *theta0, const double *z, const double *u_c, const double *u_f,
                    double *traj, uint8_t *accepted, double *lp0, double *lp1, double *lp2,
                    double *w_mean, double *w_var, int64_t *n_evals, int n_threads, double *aem_out, double *am_out,
                    int64_t *coarse_accepted)
{   /* aem_out[nc, 2 + 2 data_dim]: error samples, coarse model evaluations, error mean, error variance
     * am_out[nc, d + 2 d d]: adaptive Metropolis mean, M2, proposal factor L after the last transition
     * coarse_accepted[nc] (may be NULL): accepted sub-steps of the coarse sub-chain, summed over all transitions */
    const int d = pb->dim, J = pb->J;
    if (d > YO_MAX_DIM || pb->n_levels < 1 || pb->n_levels > 3) return -1;
    for (int l = 0; l < pb->n_levels; l++) if (pb->model != YO_GAUSS && pb->level[l].data_dim > YO_MAX_DATA) return -1;
    int64_t ev0 = 0, ev1 = 0, ev2 = 0;
#ifdef _OPENMP
    if (n_threads > 0) omp_set_num_threads(n_threads);
#endif
    #pragma omp parallel for schedule(dynamic, 1) reduction(+:ev0, ev1, ev2)
    for (int64_t c = 0; c < nc; c++) {
        chain_state cs;
        noise_src nsrc = { z + (size_t)c * ns * J * d, u_c + (size_t)c * ns * J, u_f + (size_t)c * ns, 0, 0, 0 };
        chain_init(pb, &cs, theta0 + c * d);
        for (int64_t n = 0; n <= ns; n++) {
            if (traj) memcpy(traj + ((size_t)c * (ns + 1) + n) * d, cs.theta, sizeof(double) * d);
            if (lp0) lp0[(size_t)c * (ns + 1) + n] = cs.lp[0];
            if (lp1 && pb->n_levels >= 2) lp1[(size_t)c * (ns + 1) + n] = cs.lp[1];
            if (lp2 && pb->n_levels == 3) lp2[(size_t)c * (ns + 1) + n] = cs.lp[2];
            if (n == ns) break;
            int a = chain_step(pb, &cs, &nsrc, n);
            if (accepted) accepted[(size_t)c * ns + n] = (uint8_t)a;
        }
        for (int i = 0; i < d; i++) {
            if (w_mean) w_mean[c * d + i] = cs.w_mean[i];
            if (w_var) w_var[c * d + i] = cs.w_n > 1 ? cs.w_m2[i] / (double)(cs.w_n - 1) : NAN;
        }
        ev0 += cs.n_evals[0]; ev1 += cs.n_evals[1]; ev2 += cs.n_evals[2];
        if (coarse_accepted) coarse_accepted[c] = cs.n_coarse_accept;
        if (am_out && pb->adaptive) {
            double *o = am_out + (size_t)c * (d + 2 * d * d);
            memcpy(o, cs.am_mean, sizeof(double) * d);
            memcpy(o + d, cs.am_m2, sizeof(double) * d * d);
            memcpy(o + d + d * d, cs.L, sizeof(double) * d * d);
        }
        if (aem_out && pb->aem) {
            const int dd = pb->level[0].data_dim;
            double *o = aem_out + (size_t)c * (2 + 2 * dd);
            o[0] = (double)cs.aem_n;
            o[1] = (double)cs.aem_model_evals;
            for (int k = 0; k < dd; k++) {
                o[2 + k] = cs.aem_mean[k];
                o[2 + dd + k] = cs.aem_n > 1 ? cs.aem_m2[k] / (double)(cs.aem_n - 1) : 0.0;
            }
        }
    }
    if (n_evals) { n_evals[0] = ev0; n_evals[1] = ev1; n_evals[2] = ev2; }
    return 0;
}

/* Philox-noise run (the CPU baseline arm and the stream-parity checker).
 *   theta[nc,d] in/out; traj[nc, ns/thin, d] optional (state after every thin-th step);
 *   n_accept[nc]; n_evals[2] totals.  Global chain id = chain_offset + c. */
int yo_run_philox(const yo_problem *pb, int64_t nc, int64_t chain_offset, uint64_t seed,
                  uint64_t step0, int64_t ns, int64_t thin,
                  double *theta, double *traj, int64_t *n_accept, int64_t *n_evals, int n_threads)
{
    const int d = pb->dim;
    if (d > YO_MAX_DIM || pb->n_levels < 1 || pb->n_levels > 3) return -1;
    for (int l = 0; l < pb->n_levels; l++) if (pb->model != YO_GAUSS && pb->level[l].data_dim > YO_MAX_DATA) return -1;
    if (thin < 1) thin = 1;
    const int64_t n_out = ns / thin;
    int64_t ev0 = 0, ev1 = 0;
#ifdef _OPENMP
    if (n_threads > 0) omp_set_num_threads(n_threads);
#endif
    #pragma omp parallel for schedule(dynamic, 1) reduction(+:ev0, ev1)
    for (int64_t c = 0; c < nc; c++) {
        chain_state cs;
        noise_src nsrc = { NULL, NULL, NULL, seed, (uint64_t)(chain_offset + c), step0 };
        chain_init(pb, &cs, theta + c * d);
        for (int64_t n = 0; n < ns; n++) {
            chain_step(pb, &cs, &nsrc, n);
            if (traj && (n + 1) % thin == 0)
                memcpy(traj + ((size_t)c * n_out + (n + 1) / thin - 1) * d, cs.theta, sizeof(double) * d);
        }
        memcpy(theta + c * d, cs.theta, sizeof(double) * d);
        if (n_accept) n_accept[c] = cs.n_accept;
        ev0 += cs.n_evals[0]; ev1 += cs.n_evals[1] + cs.n_evals[2];
    }
    if (n_evals) { n_evals[0] = ev0; n_evals[1] = ev1; }
    return 0;
}

/* Forward-model evaluation alone (tests of the RK4 restatement). F[n_data, data_dim] */
int yo_forward(const yo_problem *pb, int lvl, const double *theta, double *F)
{
    const yo_level *L = &pb->level[lvl];
    if (pb->model == YO_LV) {
        const double beta = exp(theta[0]), delta = exp(theta[1]);
        for (int n = 0; n < L->n_data; n++) {
            double X = L->design[2 * n], Y = L->design[2 * n + 1];
            lv_rk4(L->alpha, beta, L->gamma, delta, L->T, L->rk4_steps, &X, &Y);
            F[2 * n] = X; F[2 * n + 1] = Y;
        }
        return 0;
    }
    if (pb->model == YO_LINEAR) {
        for (int k = 0; k < L->data_dim; k++) {
            double acc = 0.0;
            for (int j = 0; j < pb->dim; j++) {
                double t = L->G[k * pb->dim + j] * theta[j];
                acc = (j == 0) ? t : acc + t;
            }
            F[k] = acc + L->b[k];
        }
        return 0;
    }
    return -1;
}

/* ---------------------------------------------------------------------- */
/* post-processing: postprocessing/autocorrelation.py:5-140               */
/* ---------------------------------------------------------------------- */

/* ACF by direct summation (the reference uses scipy.signal.correlate, FFT or
 * direct chosen automatically; same quantity up to rounding), :20-29 */
static void acf_1d(const double *x, int64_t n, int64_t stride, double *acf)
{
    double mean = 0.0;
    for (int64_t i = 0; i < n; i++) mean += x[i * stride];
    mean /= (double)n;
    double *c = (double *)malloc(sizeof(double) * (size_t)n);
    for (int64_t i = 0; i < n; i++) c[i] = x[i * stride] - mean;
    for (int64_t k = 0; k < n; k++) {
        double s = 0.0;
        for (int64_t i = 0; i + k < n; i++) s += c[i] * c[i + k];
        acf[k] = s;
    }
    double a0 = acf[0];
    for (int64_t k = 0; k < n; k++) acf[k] /= a0;
    free(c);
}

/* :62-89 with sokal_heuristic :32-59.  np.argmin over the boolean
 * "M < c*iat[M]" returns the first False; all-True returns index 0 (!),
 * none-True returns n-1. */
static int64_t iat_from_acf(const double *acf, int64_t n, double sokal)
{
    double *iat = (double *)malloc(sizeof(double) * (size_t)n);
    double cum = 0.0;
    int any = 0;
    int64_t first_false = -1;
    for (int64_t m = 0; m < n; m++) {
        cum += acf[m];
        iat[m] = 2.0 * cum - 1.0;
        int sat = (double)m < sokal * iat[m];
        if (sat) any = 1;
        else if (first_false < 0) first_false = m;
    }
    int64_t lag = any ? (first_false < 0 ? 0 : first_false) : n - 1;
    double v = rint(iat[lag]);
    free(iat);
    return (int64_t)v;
}

/* integrated_autocorrelation(seq[n,d], 'max'|'mean'), :92-140. method: 0 mean, 1 max */
int64_t yo_iat(const double *seq, int64_t n, int d, int method, double sokal)
{
    double *acf = (double *)malloc(sizeof(double) * (size_t)n);
    int64_t res = 0;
    if (method == 0) {
        double *m = (double *)malloc(sizeof(double) * (size_t)n);
        for (int64_t i = 0; i < n; i++) {
            double s = 0.0;
            for (int k = 0; k < d; k++) s += seq[i * d + k];
            m[i] = s / (double)d;
        }
        acf_1d(m, n, 1, acf);
        res = iat_from_acf(acf, n, sokal);
        free(m);
    } else {
        for (int k = 0; k < d; k++) {
            acf_1d(seq + k, n, d, acf);
            int64_t v = iat_from_acf(acf, n, sokal);
            if (k == 0 || v > res) res = v;
        }
    }
    free(acf);
    return res;
}

void yo_acf(const double *x, int64_t n, double *acf) { acf_1d(x, n, 1, acf); }

/* WelfordAccumulator over rows x[n,d] (estimation.py:36-53) */
void yo_welford(const double *x, int64_t n, int d, double *mean, double *var)
{
    double *m2 = (double *)calloc((size_t)d, sizeof(double));
    for (int i = 0; i < d; i++) mean[i] = 0.0;
    for (int64_t k = 0; k < n; k++)
        for (int i = 0; i < d; i++) {
            double delta = x[k * d + i] - mean[i];
            mean[i] += delta / (double)(k + 1);
            m2[i] += delta * (x[k * d + i] - mean[i]);
        }
    for (int i = 0; i < d; i++) var[i] = m2[i] / (double)(n - 1);
    free(m2);
}

/* DenseCovarianceMatrix (covariance.py:69-94): lower Cholesky, L x, C^-1 x.
 * scipy.linalg.cholesky -> LAPACK dpotrf; for these sizes the unblocked column algorithm (dpotf2):
 * a_jj = sqrt(c_jj - dot(l_j, l_j)); column below = (c_ij - dot(l_i, l_j)) * (1 / a_jj)  -- the
 * RECIPROCAL is formed once and multiplied (DSCAL), which rounds differently from a division. */
int yo_cholesky(const double *C, int d, double *L)
{
    memset(L, 0, sizeof(double) * d * d);
    for (int j = 0; j < d; j++) {
        double dot = 0.0;
        for (int k = 0; k < j; k++) dot += L[j * d + k] * L[j * d + k];
        double s = C[j * d + j] - dot;
        if (!(s > 0.0)) return -1;
        const double ajj = sqrt(s);
        L[j * d + j] = ajj;
        const double rcp = 1.0 / ajj;
        for (int i = j + 1; i < d; i++) {
            double dt = 0.0;
            for (int k = 0; k < j; k++) dt += L[i * d + k] * L[j * d + k];
            L[i * d + j] = (C[i * d + j] - dt) * rcp;
        }
    }
    return 0;
}

void yo_chol_apply(const double *L, int d, const double *x, double *y)
{
    for (int i = 0; i < d; i++) {
        double acc = 0.0;
        for (int j = 0; j <= i; j++) acc += L[i * d + j] * x[j];
        y[i] = acc;
    }
}

void yo_chol_solve(const double *L, int d, const double *x, double *y)
{
    double t[YO_MAX_DIM];
    for (int i = 0; i < d; i++) {                    /* L t = x */
        double s = x[i];
        for (int j = 0; j < i; j++) s -= L[i * d + j] * t[j];
        t[i] = s / L[i * d + i];
    }
    for (int i = d - 1; i >= 0; i--) {               /* L' y = t */
        double s = t[i];
        for (int j = i + 1; j < d; j++) s -= L[j * d + i] * y[j];
        y[i] = s / L[i * d + i];
    }
}

int yo_num_threads(void)
{
#ifdef _OPENMP
    return omp_get_max_threads();
#else
    return 1;
#endif
}
