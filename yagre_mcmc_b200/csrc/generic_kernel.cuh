// generic_kernel.cuh -- one chain per thread, everything in registers: the
// Metropolis-Hastings step for cheap targets (explicit Gaussian densities and the
// linear model G.theta + b), single level or two-level delayed acceptance, with
// optional per-chain adaptive Metropolis.  Also the log-posterior evaluator used
// by yg_set_state / yg_logpost for every model (LV included).
//
// Reference semantics restated (rkutri/yagre-mcmc):
//   Gaussian targets     test/testSetup.py:15-44
//   linear forward       exampleSetup.py:42-52 (A @ theta + b)
//   likelihood / prior   statistics/likelihood.py:33-39,74-84, statistics/gaussian.py:19-24
//   proposal             statistics/gaussian.py:61-66, statistics/covariance.py:51-52,84-86,
//                        pCN: chain/method/pcn.py:23-35
//   MRW / MLDA ratios    chain/method/mrw.py:51-57, chain/method/mlda.py:146-154
//   step loop            chain/metropolisHastings.py:55-120
//   adaptive interface   chain/adaptive.py:37-64 (update() before each proposal);
//                        recurrence: DESIGN.md "Adaptive Metropolis" (the reference's
//                        own AM, chain/method/deprecated/am.py, does not run)
//
// These targets cost a few hundred FP64 instructions per step, dominated by the
// transcendental sequences of Box-Muller and exp; the kernel is bound by FP64
// issue with the sample write-back (8 d bytes per chain-step, coalesced SoA) as
// the secondary bound.
#pragma once
#include "ensemble.h"
#include "lv_model.cuh"
#include "smem_plan.h"
#include <math_constants.h>
#include <algorithm>

namespace {

// numpy-ordered streaming sum of q_0..q_{n-1} produced by `next(i)` (np.sum, n <= 128 exact)
// UNROLL_SMALL: for n < 8 the terms are evaluated as seven independent (predicated) copies before they are
// added in the same order -- the dependent shared-memory loads and FP64 chains of the rows overlap instead of
// running one row after the other (one chain per thread has nothing else to hide them behind).
template <bool UNROLL_SMALL = false, typename F>
YG_DEVFN double np_stream_sum(int n, F next)
{
    if (n < 8) {
        double res = 0.0;
        if (UNROLL_SMALL) {
            double v[7];
#pragma unroll
            for (int i = 0; i < 7; i++) v[i] = (i < n) ? next(i) : 0.0;
#pragma unroll
            for (int i = 0; i < 7; i++)
                if (i < n) res += v[i];
            return res;
        }
        for (int i = 0; i < n; i++) res += next(i);
        return res;
    }
    double r[8];
#pragma unroll
    for (int k = 0; k < 8; k++) r[k] = next(k);
    const int n8 = n - (n % 8);
    for (int i = 8; i < n8; i += 8) {
#pragma unroll
        for (int k = 0; k < 8; k++) r[k] += next(i + k);
    }
    double res = ((r[0] + r[1]) + (r[2] + r[3])) + ((r[4] + r[5]) + (r[6] + r[7]));
    for (int i = n8; i < n; i++) res += next(i);
    return res;
}

// log-posterior of one parameter vector at `lvl` (chain/target.py:19-22)
template <int D, int DD>
YG_DEVFN double logpost_any(const DevProblemHeader *pb, int lvl, const double (&t)[D])
{
    const DevLevel &Lv = pb->lvl[lvl];
    const int d = pb->dim;
    double x[D];
    if (pb->model == YG_MODEL_GAUSS) {
#pragma unroll
        for (int i = 0; i < D; i++) x[i] = (i < d) ? t[i] - Lv.g_mean[i] : 0.0;
        return -0.5 * quad_form<D>(Lv.g_prec, d, x, d) + Lv.g_logconst;
    }
    const double *tail = dev_tail(pb);
    const double *data = tail + Lv.data_off;
    const int nD = Lv.n_data, dd = Lv.data_dim;
    double sum;
    if (pb->model == YG_MODEL_LINEAR) {
        double F[DD];
#pragma unroll
        for (int k = 0; k < DD; k++) {
            double acc = 0.0;
            if (k < dd) {
#pragma unroll
                for (int j = 0; j < D; j++)
                    if (j < d) acc = (j == 0) ? Lv.G[k * d] * t[0] : fma(Lv.G[k * d + j], t[j], acc);
                acc += Lv.b[k];
            }
            F[k] = acc;
        }
        sum = np_stream_sum<true>(nD, [&](int n) {
            double r[DD];
#pragma unroll
            for (int k = 0; k < DD; k++) r[k] = (k < dd) ? F[k] - data[n * dd + k] : 0.0;
            return quad_form<DD>(Lv.noise_prec, dd, r, dd);
        });
    } else {   // YG_MODEL_LV_RK4 (thread-per-parameter evaluation; the hot path is lv_kernel.cu)
        const double *design = tail + Lv.design_off;
        const double h = Lv.T / (double)Lv.rk4_steps;
        const LvStepConsts kc = lv_step_consts(Lv.alpha, Lv.gamma, h);
        const LvRates rates = lv_rates(h, exp(t[0]), exp(t[D > 1 ? 1 : 0]));
        sum = np_stream_sum(nD, [&](int n) {
            double X = design[2 * n], Y = design[2 * n + 1];
            lv_integrate(kc, rates, Lv.rk4_steps, X, Y);
            lv_finite_or_inf(X, Y);
            const double r[2] = {X - data[2 * n], Y - data[2 * n + 1]};
            return quad_form<2>(Lv.noise_prec, 2, r, 2);
        });
    }
    // tempering = 1 (an exact identity) unless the level is a TemperedUnnormalisedPosterior (target.py:40-43)
    const double logL = __dmul_rn(Lv.tempering, -0.5 * sum);
#pragma unroll
    for (int i = 0; i < D; i++) x[i] = (i < d) ? t[i] - Lv.prior_mean[i] : 0.0;
    return logL + (-0.5 * quad_form<D>(Lv.prior_prec, d, x, d));
}

__device__ void stage_blob(unsigned char *smem, const DevProblemHeader *g, uint32_t bytes)
{
    const uint4 *src = reinterpret_cast<const uint4 *>(g);
    uint4 *dst = reinterpret_cast<uint4 *>(smem);
    for (uint32_t i = threadIdx.x; i < (bytes + 15) / 16; i += blockDim.x) dst[i] = src[i];
    __syncthreads();
}

template <int D, int DD>
__global__ void logpost_kernel(const DevProblemHeader *gpb, uint32_t bytes, int lvl, const double *theta,
                               int64_t n, double *out)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    stage_blob(smem_raw, gpb, bytes);
    const DevProblemHeader *pb = reinterpret_cast<const DevProblemHeader *>(smem_raw);
    const int d = pb->dim;
    for (int64_t g = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; g < n; g += (int64_t)gridDim.x * blockDim.x) {
        double t[D];
#pragma unroll
        for (int i = 0; i < D; i++) t[i] = (i < d) ? theta[i * n + g] : 0.0;
        out[g] = logpost_any<D, DD>(pb, lvl, t);
    }
}

// In-register Cholesky of the d x d leading block; returns false if not positive definite.
// Operation order of LAPACK's unblocked dpotf2 (what scipy.linalg.cholesky runs for the reference's
// DenseCovarianceMatrix, statistics/covariance.py:78): a_jj = sqrt(c_jj - dot), and the column below is
// scaled by the RECIPROCAL 1 / a_jj (DSCAL), not divided.  Unfused, so that the factor equals the host's
// bit for bit for d <= 3 (tests/golden/am_*.npz).
template <int D>
YG_DEVFN bool cholesky_lower(const double (&C)[D][D], double (&L)[D][D], int d)
{
#pragma unroll
    for (int j = 0; j < D; j++) {
        if (j < d) {
            double dot = 0.0;
#pragma unroll
            for (int k = 0; k < D; k++)
                if (k < j) dot = __dadd_rn(dot, __dmul_rn(L[j][k], L[j][k]));
            const double s = __dsub_rn(C[j][j], dot);
            if (!(s > 0.0)) return false;
            const double ljj = sqrt(s);
            L[j][j] = ljj;
            const double rcp = 1.0 / ljj;
#pragma unroll
            for (int i = 0; i < D; i++) {
                if (i > j && i < d) {
                    double dt = 0.0;
#pragma unroll
                    for (int k = 0; k < D; k++)
                        if (k < j) dt = __dadd_rn(dt, __dmul_rn(L[i][k], L[j][k]));
                    L[i][j] = __dmul_rn(__dsub_rn(C[i][j], dt), rcp);
                }
                if (i < j) L[i][j] = 0.0;
            }
        }
    }
    return true;
}

// Warp-specialised variant (WS, d <= 2, Philox noise, small ensembles).  An ensemble of a few thousand
// chains leaves most SM sub-partitions without a warp, and a chain step is one long dependent sequence
// (Philox rounds -> log / sqrt / sincospi of Box-Muller -> proposal -> log-posterior -> exp -> compare): with
// one warp per sub-partition nothing hides its latency.  The noise does not depend on the chain state
// (counter-based Philox, keyed by chain / step / sub-step), so a CTA of three warps splits the sequence:
// warps 1 and 2 PRODUCE the normals and uniforms of the coming sub-steps into a shared-memory ring, warp 0
// CONSUMES them and runs only the state-dependent half.  Same streams, same arithmetic: trajectories are
// bit-identical to the unspecialised kernel (tests/test_backend_gpu.py).
constexpr int WS_THREADS = 64;             // 1 consumer warp + 1 producer warp (more producers measured no gain)
constexpr int64_t WS_MAX_CHAINS = 32768;   // beyond this the plain kernel has enough warps per sub-partition

template <int D, int DD, bool TWO_LEVEL, bool WS>
__global__ void __launch_bounds__(WS ? WS_THREADS : 128) generic_mh_kernel(const RunArgs a)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    double *ws_ring = nullptr;
    volatile unsigned long long *ws_ready = nullptr, *ws_consumed = nullptr;
    if (WS) {
        ws_ring = reinterpret_cast<double *>(smem_raw + ((a.problem_bytes + 15u) & ~15u));       // [WS_RING][3][32]
        ws_ready = reinterpret_cast<volatile unsigned long long *>(ws_ring + WS_RING * 96);     // [WS_RING]
        ws_consumed = ws_ready + WS_RING;
        YG_CHK(((a.problem_bytes + 15u) & ~15u) + WS_RING_BYTES - 1, yg_dynamic_smem_bytes());  // the ring fits the launch
        if (threadIdx.x <= WS_RING) ws_ready[threadIdx.x] = 0ull;                               // incl. ws_consumed
    }
    stage_blob(smem_raw, a.problem, a.problem_bytes);
    const DevProblemHeader *pb = reinterpret_cast<const DevProblemHeader *>(smem_raw);
    const int d = pb->dim;
    const int J = TWO_LEVEL ? pb->J : 1;
    // TWO_LEVEL covers delayed acceptance with one surrogate and MLDA with two surrogates as the reference runs
    // it (mlda.py:12-43,60-71,112-117): sub-chain on level 0, screen with the finest surrogate (level 1) against
    // the target (level 2)
    const int n_lvl = TWO_LEVEL ? pb->n_levels : 1;
    const bool three = TWO_LEVEL && n_lvl == 3;
    const int64_t N = a.n_chains;
    const bool isclose_eq = pb->eq_mode == YG_EQ_ISCLOSE;
    const bool pcn = pb->proposal == YG_PROPOSAL_PCN;
    unsigned long long cnt_acc = 0ull, cnt_ev0 = 0ull, cnt_ev1 = 0ull, cnt_ev2 = 0ull, cnt_tr = 0ull, cnt_cacc = 0ull;

    const int ws_lane = threadIdx.x & 31;
    const int ws_per_step = TWO_LEVEL ? J + 1 : 1;       // ring entries per transition
    if (WS && threadIdx.x >= 32) {
        // ---- producer warps: entry q = (transition n, sub-step j); warp w fills q = w, w + 2, ... ----
        const uint64_t gid = (uint64_t)(a.chain_offset + blockIdx.x * 32ll + ws_lane);
        const unsigned long long Q = (unsigned long long)a.n_steps * (unsigned long long)ws_per_step;
        const unsigned n_prod = (blockDim.x >> 5) - 1;
        int64_t n = 0;
        int j = (int)(threadIdx.x >> 5) - 1;                  // (n, j) = divmod(q, ws_per_step), kept incrementally
        for (unsigned long long q = (threadIdx.x >> 5) - 1; q < Q; q += n_prod, j += (int)n_prod) {
            while (j >= ws_per_step) { j -= ws_per_step; n++; }
            while (*ws_consumed + WS_RING <= q) __nanosleep(20);
            const uint64_t step = (uint64_t)(a.step0 + n);
            double z0 = 0.0, z1 = 0.0, u;
            if (!TWO_LEVEL || j < J) philox_normal_pair(a.seed, gid, step, (uint32_t)j, 0u, z0, z1);
            u = philox_uniform(a.seed, gid, step, (!TWO_LEVEL || j == J) ? YG_SUB_FINE : (uint32_t)j);
            YG_CHK((q % WS_RING) * 96 + ws_lane + 64, WS_RING * 96);
            double *slot = ws_ring + (q % WS_RING) * 96 + ws_lane;
            slot[0] = z0; slot[32] = z1; slot[64] = u;
            __threadfence_block();
            __syncwarp();
            if (ws_lane == 0) ws_ready[q % WS_RING] = q + 1ull;
        }
        return;
    }
    unsigned ws_mask = 0xffffffffu;
    unsigned long long ws_q = 0ull;
    double ws_z0 = 0.0, ws_z1 = 0.0, ws_u = 0.0;
    // consumer: the noise of ring entry ws_q (all live lanes of the warp call this together)
    auto ws_fetch = [&]() {
        __syncwarp(ws_mask);
        const int e = (int)(ws_q % WS_RING);
        while (ws_ready[e] != ws_q + 1ull) { }
        __threadfence_block();
        YG_CHK(e * 96 + ws_lane + 64, WS_RING * 96);
        const volatile double *slot = ws_ring + e * 96 + ws_lane;
        ws_z0 = slot[0]; ws_z1 = slot[32]; ws_u = slot[64];
        __syncwarp(ws_mask);
        ws_q += 1ull;
        if (ws_lane == __ffs(ws_mask) - 1) *ws_consumed = ws_q;
    };
    if (WS) {
        ws_mask = __ballot_sync(0xffffffffu, blockIdx.x * 32ll + ws_lane < N);
        if (blockIdx.x * 32ll + ws_lane >= N) return;
    }

    const int64_t g_first = WS ? blockIdx.x * 32ll + ws_lane : blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    const int64_t g_stride = WS ? N : (int64_t)gridDim.x * blockDim.x;      // WS: one chain per consumer lane
    for (int64_t g = g_first; g < N; g += g_stride) {
        const uint64_t gid = (uint64_t)(a.chain_offset + g);
        double th[D], wm[D], w2[D][D], L[D][D];
        double am_m[D], am_2[D][D];
#pragma unroll
        for (int i = 0; i < D; i++) {
            th[i] = (i < d) ? a.theta[i * N + g] : 0.0;
            wm[i] = (i < d) ? a.w_mean[i * N + g] : 0.0;
#pragma unroll
            for (int j = 0; j < D; j++) {
                w2[i][j] = (i < d && j < d) ? a.w_m2[(i * d + j) * N + g] : 0.0;
                L[i][j] = (i < d && j < d) ? (a.adaptive ? a.prop_L[(i * d + j) * N + g] : pb->prop_L[i * d + j]) : 0.0;
                am_2[i][j] = (a.adaptive && i < d && j < d) ? a.am_m2[(i * d + j) * N + g] : 0.0;
            }
            am_m[i] = (a.adaptive && i < d) ? a.am_mean[i * N + g] : 0.0;
        }
        double lp0 = a.logpost[g], lp1 = TWO_LEVEL ? a.logpost[N + g] : 0.0;
        double lp2 = three ? a.logpost[2 * N + g] : 0.0;
        unsigned long long nacc = a.n_accept[g];

        auto equal = [&](const double (&p)[D], const double (&s)[D]) {
            if (isclose_eq) return isclose_rule(p[0], s[0]);
            bool eq = true;
#pragma unroll
            for (int i = 0; i < D; i++)
                if (i < d) eq = eq && (p[i] == s[i]);
            return eq;
        };
        // p = s + L z, unfused, exact zeros of L skipped (covariance.py:51-52,84-86)
        auto propose = [&](const double (&s)[D], int64_t n, int j, uint64_t step, double (&p)[D]) {
            double z[D];
            if (WS) {
#pragma unroll
                for (int i = 0; i < D; i++) z[i] = (i == 0) ? ws_z0 : (i == 1 ? ws_z1 : 0.0);
            } else if (a.noise_mode == YG_NOISE_INJECT) {
#pragma unroll
                YG_CHK(((n * J + j) * d + d - 1) * N + g, a.n_steps * J * d * N);
                for (int i = 0; i < D; i++) z[i] = (i < d) ? a.z[((n * J + j) * d + i) * N + g] : 0.0;
            } else {
#pragma unroll
                for (int b = 0; b < (D + 1) / 2; b++) {
                    if (2 * b < d) {
                        double z0, z1;
                        philox_normal_pair(a.seed, gid, step, (uint32_t)j, (uint32_t)b, z0, z1);
                        z[2 * b] = z0;
                        if (2 * b + 1 < D) z[2 * b + 1] = z1;
                    }
                }
                if (a.noise_mode == YG_NOISE_RECORD) {
#pragma unroll
                    for (int i = 0; i < D; i++)
                        if (i < d) a.z[((n * J + j) * d + i) * N + g] = z[i];
                }
            }
#pragma unroll
            for (int i = 0; i < D; i++) {
                double acc = 0.0;
                bool first = true;
#pragma unroll
                for (int k = 0; k < D; k++) {
                    if (k <= i && i < d) {
                        const double l = L[i][k];
                        if (l != 0.0 || k == i) {
                            const double t = __dmul_rn(l, z[k]);
                            acc = first ? t : __dadd_rn(acc, t);
                            first = false;
                        }
                    }
                }
                if (pcn)      // pcn.py:30-35: sqrt(1-t) * state + sqrt(t) * (mean + L z), unfused like numpy
                    p[i] = (i < d) ? __dadd_rn(__dmul_rn(pb->pcn_a, s[i]), __dmul_rn(pb->pcn_b, __dadd_rn(pb->pcn_mean[i], acc)))
                                   : 0.0;
                else
                    p[i] = (i < d) ? __dadd_rn(s[i], acc) : 0.0;
            }
        };

        // ---- adaptive Metropolis: AdaptiveMRWProposal.set_state -> update() (adaptive.py:55-60) runs before
        // every proposal of the MRW chain it drives, with that chain's current state x (the sub-chain state in
        // the two-level case); t_idx = number of earlier updates.  Recurrence: DESIGN.md section 5, arithmetic
        // pinned to oracle/ref_harness.py HaarioAdaptiveCovariance (unfused, numpy order).
        auto am_update = [&](const double (&x)[D], const int64_t t_idx) {
            if (t_idx < a.am_idle) return;
            const int64_t n_am = t_idx - a.am_idle + 1;
            double dl[D], e[D];
#pragma unroll
            for (int i = 0; i < D; i++) {
                dl[i] = __dsub_rn(x[i], am_m[i]);
                am_m[i] = __dadd_rn(am_m[i], dl[i] / (double)n_am);
                e[i] = __dsub_rn(x[i], am_m[i]);
            }
#pragma unroll
            for (int i = 0; i < D; i++)
#pragma unroll
                for (int j = 0; j < D; j++) am_2[i][j] = __dadd_rn(am_2[i][j], __dmul_rn(dl[i], e[j]));
            if (n_am >= a.am_collect && n_am >= 2 && (a.am_refresh == 1 || ((n_am - a.am_collect) % a.am_refresh) == 0)) {
                double Cm[D][D], Ln[D][D];
#pragma unroll
                for (int i = 0; i < D; i++)
#pragma unroll
                    for (int j = 0; j < D; j++) {
                        // symmetrised sample covariance, C = s (Cov + eps I)
                        const double cov = __dmul_rn(0.5, __dadd_rn(am_2[i][j], am_2[j][i])) / (double)(n_am - 1);
                        Cm[i][j] = __dmul_rn(a.am_scale, (i == j) ? __dadd_rn(cov, a.am_eps) : cov);
                        Ln[i][j] = 0.0;
                    }
                if (cholesky_lower<D>(Cm, Ln, d)) {
#pragma unroll
                    for (int i = 0; i < D; i++)
#pragma unroll
                        for (int j = 0; j < D; j++) L[i][j] = Ln[i][j];
                }
            }
        };

        int64_t thin_left = a.thin, thin_out = 0;
        for (int64_t n = 0; n < a.n_steps; n++) {
            const uint64_t step = (uint64_t)(a.step0 + n);
            // ---- diagnostics Welford of the pre-transition state (diagnostics.py:91-94) ----
            {
                const double wn = (double)(a.welford_n0 + n + 1);
                double dl[D], e[D];
#pragma unroll
                for (int i = 0; i < D; i++) {
                    dl[i] = th[i] - wm[i];
                    wm[i] += dl[i] / wn;
                    e[i] = th[i] - wm[i];
                }
#pragma unroll
                for (int i = 0; i < D; i++)
#pragma unroll
                    for (int j = 0; j < D; j++) w2[i][j] += dl[i] * e[j];
            }
            bool accepted = false;
            if (!TWO_LEVEL) {
                double p[D];
                if (a.adaptive) am_update(th, a.am_t0 + n);
                if (WS) ws_fetch();
                propose(th, n, 0, step, p);
                if (!equal(p, th)) {                                    // metropolisHastings.py:60-61
                    const double lpp = logpost_any<D, DD>(pb, 0, p);
                    cnt_ev0++;
                    double u;
                    if (WS) u = ws_u;
                    else if (a.noise_mode == YG_NOISE_INJECT) u = a.u_f[n * N + g];
                    else {
                        u = philox_uniform(a.seed, gid, step, YG_SUB_FINE);
                        if (a.noise_mode == YG_NOISE_RECORD) a.u_f[n * N + g] = u;
                    }
                    if (accept_rule(lpp - lp0, u)) {
#pragma unroll
                        for (int i = 0; i < D; i++) th[i] = p[i];
                        lp0 = lpp;
                        accepted = true;
                    }
                }
            } else {
                double s[D], p[D];
#pragma unroll
                for (int i = 0; i < D; i++) s[i] = th[i];
                double lps = lp0;
                for (int j = 0; j < J; j++) {                           // coarse sub-chain, mlda.py:100-110
                    if (a.adaptive) am_update(s, (a.am_t0 + n) * J + j);
                    if (WS) ws_fetch();
                    propose(s, n, j, step, p);
                    if (equal(p, s)) continue;
                    const double lpp = logpost_any<D, DD>(pb, 0, p);
                    cnt_ev0++;
                    double u;
                    const int64_t ui = (n * J + j) * N + g;
                    if (WS) u = ws_u;
                    else if (a.noise_mode == YG_NOISE_INJECT) u = a.u_c[ui];
                    else {
                        u = philox_uniform(a.seed, gid, step, (uint32_t)j);
                        if (a.noise_mode == YG_NOISE_RECORD) a.u_c[ui] = u;
                    }
                    if (accept_rule(lpp - lps, u)) {
#pragma unroll
                        for (int i = 0; i < D; i++) s[i] = p[i];
                        lps = lpp;
                        cnt_cacc++;
                    }
                }
                if (WS) ws_fetch();
                if (!equal(s, th)) {
                    // levels above the sub-chain's: one (the target) or two (finest surrogate, target)
                    double lpm_s = 0.0, lpf_s = 0.0;
                    for (int lv = 1; lv < n_lvl; lv++) {
                        const double v = logpost_any<D, DD>(pb, lv, s);
                        if (lv == n_lvl - 1) { lpf_s = v; cnt_ev1++; } else { lpm_s = v; cnt_ev2++; }
                    }
                    double u;
                    if (WS) u = ws_u;
                    else if (a.noise_mode == YG_NOISE_INJECT) u = a.u_f[n * N + g];
                    else {
                        u = philox_uniform(a.seed, gid, step, YG_SUB_FINE);
                        if (a.noise_mode == YG_NOISE_RECORD) a.u_f[n * N + g] = u;
                    }
                    // mlda.py:148-152, this order: pi_f(p) + pi_c(s) - pi_c(p) - pi_f(s); with two surrogates
                    // pi_c is the FINEST surrogate although the sub-chain ran on the base one (mlda.py:130,146-154)
                    const double delta = three ? lpf_s + lp1 - lpm_s - lp2 : lpf_s + lp0 - lps - lp1;
                    if (accept_rule(delta, u)) {
#pragma unroll
                        for (int i = 0; i < D; i++) th[i] = s[i];
                        lp0 = lps;
                        if (three) { lp1 = lpm_s; lp2 = lpf_s; } else lp1 = lpf_s;
                        accepted = true;
                    }
                }
            }
            if (accepted) { nacc++; cnt_acc++; }
            cnt_tr++;
            if (a.accepted) a.accepted[n * N + g] = accepted ? 1 : 0;
            YG_CHK(g, N); YG_CHK(n, a.n_steps);
            if (--thin_left == 0) {                 // (n + 1) % thin == 0 without a 64-bit division per step
                thin_left = a.thin;
                const int64_t o = thin_out++;
                YG_CHK(o, a.n_steps / a.thin);
                if (a.samples) {
#pragma unroll
                    for (int i = 0; i < D; i++)
                        if (i < d) a.samples[(o * d + i) * N + g] = th[i];
                }
                if (a.lp_out) {
                    a.lp_out[(o * n_lvl) * N + g] = lp0;
                    if (TWO_LEVEL) a.lp_out[(o * n_lvl + 1) * N + g] = lp1;
                    if (three) a.lp_out[(o * n_lvl + 2) * N + g] = lp2;
                }
            }
        }
        // ---- store chain state ---------------------------------------------------------
#pragma unroll
        for (int i = 0; i < D; i++) {
            if (i < d) {
                a.theta[i * N + g] = th[i];
                a.w_mean[i * N + g] = wm[i];
                if (a.adaptive) a.am_mean[i * N + g] = am_m[i];
#pragma unroll
                for (int j = 0; j < D; j++) {
                    if (j < d) {
                        a.w_m2[(i * d + j) * N + g] = w2[i][j];
                        if (a.adaptive) {
                            a.am_m2[(i * d + j) * N + g] = am_2[i][j];
                            a.prop_L[(i * d + j) * N + g] = L[i][j];
                        }
                    }
                }
            }
        }
        a.logpost[g] = lp0;
        if (TWO_LEVEL) a.logpost[N + g] = lp1;
        if (three) a.logpost[2 * N + g] = lp2;
        a.n_accept[g] = nacc;
    }
    // ---- counters: warp-shuffle reduction, one atomic per warp ------------------------------
    unsigned long long v[6] = {cnt_tr, cnt_acc, cnt_ev0, cnt_ev1, cnt_ev2, cnt_cacc};
#pragma unroll
    for (int k = 0; k < 6; k++) {
        if (WS) {                                   // exited lanes (chains beyond N, producers) cannot shuffle
            if (v[k]) atomicAdd(&a.counters[k], v[k]);
            continue;
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v[k] += __shfl_xor_sync(0xffffffffu, v[k], o);
        if ((threadIdx.x & 31) == 0 && v[k]) atomicAdd(&a.counters[k], v[k]);
    }
}

// ---------------------------------------------------------------------------------------------
// Adaptive error model (two-level delayed acceptance on the linear model): reference
// chain/method/aem.py:25-58, statistics/likelihood.py:90-155, statistics/noise.py:25-61,
// utility/memoisation.py:76-149.  One chain per thread.  Per chain: Welford of F_fine - F_coarse
// on accepted fine steps; the coarse residual is shifted by the error mean once min_data errors
// were seen; the noise variance is inflated from min_data + 1 errors on; and the coarse
// likelihood's LRU(3) cache is reproduced entry for entry, because the reference does NOT
// invalidate cached log-likelihoods when the error model changes: which value a chain sees for
// pi_c(state) depends on whether the state is still among the last three parameters queried.
// ISCLOSE: proposals of a scalar chain are compared with math.isclose (parameter/scalar.py:38-43); a
// separate instance, launched only for eq_mode == YG_EQ_ISCLOSE (d = 1, capacity 2), so that the
// exact-equality instances compile as if the rule did not exist.  The cache keys stay exact.
// ---------------------------------------------------------------------------------------------
template <int D>
struct Lru3 {
    double key[3][D], val[3];
    int n;
};

template <int D>
YG_DEVFN int lru_find(const Lru3<D> &c, const double (&x)[D], int d)
{
    int idx = -1;
#pragma unroll
    for (int i = 2; i >= 0; i--) {
        bool eq = i < c.n;
#pragma unroll
        for (int k = 0; k < D; k++)
            if (k < d) eq = eq && (c.key[i][k] == x[k]);            // parameter/vector.py:37-45
        if (eq) idx = i;
    }
    return idx;
}

// AEMCache._move_to_back (memoisation.py:95-100): bubble entry idx to the newest position
template <int D>
YG_DEVFN void lru_touch(Lru3<D> &c, int idx)
{
#pragma unroll
    for (int i = 0; i < 2; i++) {
        if (i >= idx && i + 1 < c.n) {
#pragma unroll
            for (int k = 0; k < D; k++) { const double t = c.key[i][k]; c.key[i][k] = c.key[i + 1][k]; c.key[i + 1][k] = t; }
            const double t = c.val[i]; c.val[i] = c.val[i + 1]; c.val[i + 1] = t;
        }
    }
}

// AEMCache.add (memoisation.py:102-116): evict the oldest of three, append
template <int D>
YG_DEVFN void lru_add(Lru3<D> &c, const double (&x)[D], double v)
{
    if (c.n >= 3) {
#pragma unroll
        for (int i = 0; i < 2; i++) {
#pragma unroll
            for (int k = 0; k < D; k++) c.key[i][k] = c.key[i + 1][k];
            c.val[i] = c.val[i + 1];
        }
        c.n = 2;
    }
#pragma unroll
    for (int i = 0; i < 3; i++) {
        if (i == c.n) {
#pragma unroll
            for (int k = 0; k < D; k++) c.key[i][k] = x[k];
            c.val[i] = v;
        }
    }
    c.n++;
}

template <int D, int DD, bool ISCLOSE>
__global__ void __launch_bounds__(128) aem_mh_kernel(const RunArgs a)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    stage_blob(smem_raw, a.problem, a.problem_bytes);
    const DevProblemHeader *pb = reinterpret_cast<const DevProblemHeader *>(smem_raw);
    const int d = pb->dim, J = pb->J;
    const DevLevel &Lc = pb->lvl[0], &Lf = pb->lvl[1];
    const int dd = Lc.data_dim, nD = Lc.n_data;
    const double *data = dev_tail(pb) + Lc.data_off;
    const int64_t N = a.n_chains;
    unsigned long long cnt_acc = 0ull, cnt_ev0 = 0ull, cnt_ev1 = 0ull, cnt_tr = 0ull, cnt_cacc = 0ull;

    for (int64_t g = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; g < N; g += (int64_t)gridDim.x * blockDim.x) {
        const uint64_t gid = (uint64_t)(a.chain_offset + g);
        double th[D], wm[D], w2[D][D];
#pragma unroll
        for (int i = 0; i < D; i++) {
            th[i] = (i < d) ? a.theta[i * N + g] : 0.0;
            wm[i] = (i < d) ? a.w_mean[i * N + g] : 0.0;
#pragma unroll
            for (int j = 0; j < D; j++) w2[i][j] = (i < d && j < d) ? a.w_m2[(i * d + j) * N + g] : 0.0;
        }
        double lp0 = a.logpost[g], lp1 = a.logpost[N + g];
        unsigned long long nacc = a.n_accept[g];
        // ---- error model + cache state -----------------------------------------------------------
        unsigned long long en = a.aem_n[g];
        double em[DD], e2[DD], eprec[DD];
        bool have_noise = false;
#pragma unroll
        for (int k = 0; k < DD; k++) {
            em[k] = (k < dd) ? a.aem_mean[k * N + g] : 0.0;
            e2[k] = (k < dd) ? a.aem_m2[k * N + g] : 0.0;
            eprec[k] = 0.0;
        }
        Lru3<D> cache;
        {
            const int stride = d + 1;
            cache.n = (int)a.aem_cache[(int64_t)(3 * stride) * N + g];
#pragma unroll
            for (int i = 0; i < 3; i++) {
#pragma unroll
                for (int k = 0; k < D; k++) cache.key[i][k] = (k < d) ? a.aem_cache[(int64_t)(i * stride + k) * N + g] : 0.0;
                cache.val[i] = a.aem_cache[(int64_t)(i * stride + d) * N + g];
            }
        }
        // noise.py:41-54 (+ covariance.py:33-38): precision of the inflated noise from the current moments
        auto refresh_noise = [&]() {
            if (en > (unsigned long long)a.aem_min_data) {
                double mv[DD], mn = CUDART_INF, mx = -CUDART_INF;
#pragma unroll
                for (int k = 0; k < DD; k++) {
                    mv[k] = (k < dd) ? e2[k] / (double)(en - 1ull) : 0.0;
                    if (k < dd) { mn = fmin(mn, mv[k]); mx = fmax(mx, mv[k]); }
                }
                double scaling = 1.0;
                if (a.aem_heuristic) {
                    const double minVal = mn > 1e-6 ? mn : 1e-6;
                    scaling = 2.0 * mx / minVal;
                    if (scaling > 100.0) scaling = 100.0;
                }
#pragma unroll
                for (int k = 0; k < DD; k++)
                    if (k < dd) eprec[k] = 1.0 / (scaling * mv[k] + 1.0 / Lc.noise_prec[k * dd + k]);
                have_noise = true;
            }
        };
        refresh_noise();
        auto forward = [&](const DevLevel &Lv, const double (&x)[D], double (&F)[DD]) {
#pragma unroll
            for (int k = 0; k < DD; k++) {
                double acc = 0.0;
                if (k < dd) {
#pragma unroll
                    for (int j = 0; j < D; j++)
                        if (j < d) acc = (j == 0) ? Lv.G[k * d] * x[0] : fma(Lv.G[k * d + j], x[j], acc);
                    acc += Lv.b[k];
                }
                F[k] = acc;
            }
        };
        // AEMLikelihood.compute_log_likelihood (likelihood.py:74-84,140-145) + prior (target.py:19-22)
        auto coarse_logpost = [&](const double (&x)[D]) {
            double F[DD];
            forward(Lc, x, F);
            cnt_ev0++;
            const bool shift = en >= (unsigned long long)a.aem_min_data;
            const double sum = np_stream_sum(nD, [&](int n) {
                double acc = 0.0;
#pragma unroll
                for (int k = 0; k < DD; k++) {
                    if (k < dd) {
                        double r = F[k] - data[n * dd + k];
                        if (shift) r = r + em[k];
                        const double prec = have_noise ? eprec[k] : Lc.noise_prec[k * dd + k];
                        acc = (k == 0) ? r * (prec * r) : fma(r, prec * r, acc);
                    }
                }
                return acc;
            });
            double xx[D];
#pragma unroll
            for (int i = 0; i < D; i++) xx[i] = (i < d) ? x[i] - Lc.prior_mean[i] : 0.0;
            return -0.5 * sum + (-0.5 * quad_form<D>(Lc.prior_prec, d, xx, d));
        };
        // AEMLikelihood.query_log_likelihood (likelihood.py:126-131)
        auto query_coarse = [&](const double (&x)[D]) {
            const int idx = lru_find<D>(cache, x, d);
            if (idx >= 0) {
                const double v = (idx == 0) ? cache.val[0] : (idx == 1 ? cache.val[1] : cache.val[2]);
                lru_touch<D>(cache, idx);
                return v;
            }
            const double v = coarse_logpost(x);
            lru_add<D>(cache, x, v);
            return v;
        };
        auto propose = [&](const double (&s)[D], int64_t n, int j, uint64_t step, double (&p)[D]) {
            double z[D];
#pragma unroll
            for (int i = 0; i < D; i++) z[i] = 0.0;
            if (a.noise_mode == YG_NOISE_INJECT) {
#pragma unroll
                YG_CHK(((n * J + j) * d + d - 1) * N + g, a.n_steps * J * d * N);
                for (int i = 0; i < D; i++) z[i] = (i < d) ? a.z[((n * J + j) * d + i) * N + g] : 0.0;
            } else {
#pragma unroll
                for (int b = 0; b < (D + 1) / 2; b++) {
                    if (2 * b < d) {
                        double z0, z1;
                        philox_normal_pair(a.seed, gid, step, (uint32_t)j, (uint32_t)b, z0, z1);
                        z[2 * b] = z0;
                        if (2 * b + 1 < D) z[2 * b + 1] = z1;
                    }
                }
                if (a.noise_mode == YG_NOISE_RECORD) {
#pragma unroll
                    for (int i = 0; i < D; i++)
                        if (i < d) a.z[((n * J + j) * d + i) * N + g] = z[i];
                }
            }
#pragma unroll
            for (int i = 0; i < D; i++) {
                double acc = 0.0;
                bool first = true;
#pragma unroll
                for (int k = 0; k < D; k++) {
                    if (k <= i && i < d) {
                        const double l = pb->prop_L[i * d + k];
                        if (l != 0.0 || k == i) {
                            const double t = __dmul_rn(l, z[k]);
                            acc = first ? t : __dadd_rn(acc, t);
                            first = false;
                        }
                    }
                }
                p[i] = (i < d) ? __dadd_rn(s[i], acc) : 0.0;
            }
        };
        auto equal = [&](const double (&p)[D], const double (&s)[D]) {
            if (ISCLOSE) return isclose_rule(p[0], s[0]);
            bool eq = true;
#pragma unroll
            for (int i = 0; i < D; i++)
                if (i < d) eq = eq && (p[i] == s[i]);
            return eq;
        };

        int64_t thin_left = a.thin, thin_out = 0;
        for (int64_t n = 0; n < a.n_steps; n++) {
            const uint64_t step = (uint64_t)(a.step0 + n);
            {   // diagnostics Welford of the pre-transition state (diagnostics.py:91-94)
                const double wn = (double)(a.welford_n0 + n + 1);
                double dl[D], e[D];
#pragma unroll
                for (int i = 0; i < D; i++) {
                    dl[i] = th[i] - wm[i];
                    wm[i] += dl[i] / wn;
                    e[i] = th[i] - wm[i];
                }
#pragma unroll
                for (int i = 0; i < D; i++)
#pragma unroll
                    for (int j = 0; j < D; j++) w2[i][j] += dl[i] * e[j];
            }
            bool accepted = false;
            double s[D], p[D];
#pragma unroll
            for (int i = 0; i < D; i++) s[i] = th[i];
            for (int j = 0; j < J; j++) {                               // coarse sub-chain, mlda.py:100-110
                propose(s, n, j, step, p);
                if (equal(p, s)) continue;
                const double lpp = query_coarse(p);                     // mrw.py:53: proposal first, then state
                const double lps = query_coarse(s);
                double u;
                const int64_t ui = (n * J + j) * N + g;
                if (a.noise_mode == YG_NOISE_INJECT) u = a.u_c[ui];
                else {
                    u = philox_uniform(a.seed, gid, step, (uint32_t)j);
                    if (a.noise_mode == YG_NOISE_RECORD) a.u_c[ui] = u;
                }
                if (accept_rule(lpp - lps, u)) {
#pragma unroll
                    for (int i = 0; i < D; i++) s[i] = p[i];
                    cnt_cacc++;
                }
            }
            if (!equal(s, th)) {
                // mlda.py:148-152: pi_f(P) + pi_c(theta) - pi_c(P) - pi_f(theta), evaluated in this order
                const double lpf_s = logpost_any<D, DD>(pb, 1, s);
                cnt_ev1++;
                const double lpc_t = query_coarse(th);
                const double lpc_s = query_coarse(s);
                double u;
                if (a.noise_mode == YG_NOISE_INJECT) u = a.u_f[n * N + g];
                else {
                    u = philox_uniform(a.seed, gid, step, YG_SUB_FINE);
                    if (a.noise_mode == YG_NOISE_RECORD) a.u_f[n * N + g] = u;
                }
                const double delta = lpf_s + lpc_t - lpc_s - lp1;
                if (accept_rule(delta, u)) {
                    // aem.py:44-56 + likelihood.py:147-155: feed F_f(P) - F_c(P) to the coarse error model
                    const int idx = lru_find<D>(cache, s, d);           // query_model_evaluation: a hit moves the entry back
                    if (idx >= 0) lru_touch<D>(cache, idx); else cnt_ev0++;
                    double Fc[DD], Ff[DD];
                    forward(Lc, s, Fc);
                    forward(Lf, s, Ff);
                    en += 1ull;
#pragma unroll
                    for (int k = 0; k < DD; k++) {
                        if (k < dd) {                                    // estimation.py:36-53
                            const double e = Ff[k] - Fc[k];
                            const double dl = e - em[k];
                            em[k] += dl / (double)en;
                            e2[k] += dl * (e - em[k]);
                        }
                    }
                    refresh_noise();
#pragma unroll
                    for (int i = 0; i < D; i++) th[i] = s[i];
                    lp0 = lpc_s;
                    lp1 = lpf_s;
                    accepted = true;
                }
            }
            if (accepted) { nacc++; cnt_acc++; }
            cnt_tr++;
            if (a.accepted) a.accepted[n * N + g] = accepted ? 1 : 0;
            YG_CHK(g, N); YG_CHK(n, a.n_steps);
            if (--thin_left == 0) {                 // (n + 1) % thin == 0 without a 64-bit division per step
                thin_left = a.thin;
                const int64_t o = thin_out++;
                YG_CHK(o, a.n_steps / a.thin);
                if (a.samples) {
#pragma unroll
                    for (int i = 0; i < D; i++)
                        if (i < d) a.samples[(o * d + i) * N + g] = th[i];
                }
                if (a.lp_out) {
                    a.lp_out[(o * 2) * N + g] = lp0;        // coarse value as last evaluated (may be stale, see above)
                    a.lp_out[(o * 2 + 1) * N + g] = lp1;
                }
            }
        }
        // ---- store chain state ---------------------------------------------------------------------
#pragma unroll
        for (int i = 0; i < D; i++) {
            if (i < d) {
                a.theta[i * N + g] = th[i];
                a.w_mean[i * N + g] = wm[i];
#pragma unroll
                for (int j = 0; j < D; j++)
                    if (j < d) a.w_m2[(i * d + j) * N + g] = w2[i][j];
            }
        }
        a.logpost[g] = lp0;
        a.logpost[N + g] = lp1;
        a.n_accept[g] = nacc;
        a.aem_n[g] = en;
#pragma unroll
        for (int k = 0; k < DD; k++) {
            if (k < dd) { a.aem_mean[k * N + g] = em[k]; a.aem_m2[k * N + g] = e2[k]; }
        }
        {
            const int stride = d + 1;
            a.aem_cache[(int64_t)(3 * stride) * N + g] = (double)cache.n;
#pragma unroll
            for (int i = 0; i < 3; i++) {
#pragma unroll
                for (int k = 0; k < D; k++)
                    if (k < d) a.aem_cache[(int64_t)(i * stride + k) * N + g] = cache.key[i][k];
                a.aem_cache[(int64_t)(i * stride + d) * N + g] = cache.val[i];
            }
        }
    }
    unsigned long long v[5] = {cnt_tr, cnt_acc, cnt_ev0, cnt_ev1, cnt_cacc};
#pragma unroll
    for (int k = 0; k < 5; k++) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v[k] += __shfl_xor_sync(0xffffffffu, v[k], o);
        if ((threadIdx.x & 31) == 0 && v[k]) atomicAdd(&a.counters[k == 4 ? 5 : k], v[k]);
    }
}

template <int D, int DD>
int launch_aem_t(yg_ensemble *e, const RunArgs &a, cudaStream_t st)
{
    const int threads = 128;
    const int64_t want = (a.n_chains + threads - 1) / threads;
    const int grid = (int)std::max<int64_t>(1, std::min<int64_t>(want, (int64_t)e->sm_count * 16));
    const size_t smem = (e->h_problem.size() + 15) & ~size_t(15);
    auto kern = aem_mh_kernel<D, DD, false>;
    if constexpr (D == 2) {                                   // abi.cu: isclose needs d = 1
        if (e->cfg.eq_mode == YG_EQ_ISCLOSE) kern = aem_mh_kernel<2, DD, true>;
    }
    YG_CUDA_CHECK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    kern<<<grid, threads, smem, st>>>(a);
    YG_CUDA_CHECK(cudaGetLastError());
    e->last_grid = grid;
    e->last_block = threads;
    e->last_smem = (int)smem;
    e->launches += 1;
    return YG_OK;
}

template <int D, int DD>
int launch_generic_t(yg_ensemble *e, const RunArgs &a, cudaStream_t st)
{
    int threads = 128;
    const int64_t want = (a.n_chains + threads - 1) / threads;
    int grid = (int)std::max<int64_t>(1, std::min<int64_t>(want, (int64_t)e->sm_count * 16));
    size_t smem = (e->h_problem.size() + 15) & ~size_t(15);
    auto kern = e->cfg.n_levels >= 2 ? generic_mh_kernel<D, DD, true, false> : generic_mh_kernel<D, DD, false, false>;
    // small ensembles with Philox noise: warp-specialised variant (see WS above); the parity modes
    // (injected / recorded noise) stay on the plain kernel, which the WS variant equals bit for bit
    if (D == 2 && a.noise_mode == YG_NOISE_PHILOX && a.n_chains <= WS_MAX_CHAINS && a.n_steps > 0) {
        kern = e->cfg.n_levels >= 2 ? generic_mh_kernel<D, DD, true, D == 2> : generic_mh_kernel<D, DD, false, D == 2>;
        threads = WS_THREADS;
        grid = (int)((a.n_chains + 31) / 32);
        smem += WS_RING_BYTES;
    }
    YG_CUDA_CHECK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    kern<<<grid, threads, smem, st>>>(a);
    YG_CUDA_CHECK(cudaGetLastError());
    e->last_grid = grid;
    e->last_block = threads;
    e->last_smem = (int)smem;
    e->launches += 1;
    return YG_OK;
}

template <int D, int DD>
int launch_logpost_t(yg_ensemble *e, int level, const double *theta, int64_t n, double *out, cudaStream_t st)
{
    const int threads = 128;
    const int64_t want = (n + threads - 1) / threads;
    const int grid = (int)std::max<int64_t>(1, std::min<int64_t>(want, (int64_t)e->sm_count * 16));
    const size_t smem = (e->h_problem.size() + 15) & ~size_t(15);
    auto kern = logpost_kernel<D, DD>;
    YG_CUDA_CHECK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    kern<<<grid, threads, smem, st>>>(static_cast<const DevProblemHeader *>(e->d_problem), (uint32_t)e->h_problem.size(),
                                      level, theta, n, out);
    YG_CUDA_CHECK(cudaGetLastError());
    e->launches += 1;
    return YG_OK;
}

}  // namespace

// One translation unit per parameter-dimension capacity D (generic_d2.cu, generic_d4.cu, generic_d8.cu): the 42
// kernel instances compile in parallel instead of in one eight-minute nvcc run.  Each unit defines
//   int yg_launch_generic_d<D>(e, a, st, cdd)   and   int yg_launch_logpost_d<D>(e, level, theta, n, out, st, cdd)
// with cdd the data-dimension capacity (2, 4 or 8); generic_kernel.cu dispatches on D.
#ifdef YG_DEV_22      /* dev build (make dev): data_dim <= 2 only, compiles in seconds */
#define YG_GENERIC_UNIT(D)                                                                                         \
    int yg_launch_generic_d##D(yg_ensemble *e, const RunArgs &a, cudaStream_t st, int cdd)                         \
    {                                                                                                              \
        if (cdd == 2) return a.aem ? launch_aem_t<D, 2>(e, a, st) : launch_generic_t<D, 2>(e, a, st);              \
        return YG_ERR_UNSUPPORTED;                                                                                 \
    }                                                                                                              \
    int yg_launch_logpost_d##D(yg_ensemble *e, int level, const double *theta, int64_t n, double *out,             \
                               cudaStream_t st, int cdd)                                                           \
    {                                                                                                              \
        if (cdd == 2) return launch_logpost_t<D, 2>(e, level, theta, n, out, st);                                  \
        return YG_ERR_UNSUPPORTED;                                                                                 \
    }
#else
#define YG_GENERIC_UNIT(D)                                                                                         \
    int yg_launch_generic_d##D(yg_ensemble *e, const RunArgs &a, cudaStream_t st, int cdd)                         \
    {                                                                                                              \
        switch (cdd) {                                                                                             \
        case 2: return a.aem ? launch_aem_t<D, 2>(e, a, st) : launch_generic_t<D, 2>(e, a, st);                    \
        case 4: return a.aem ? launch_aem_t<D, 4>(e, a, st) : launch_generic_t<D, 4>(e, a, st);                    \
        case 8: return a.aem ? launch_aem_t<D, 8>(e, a, st) : launch_generic_t<D, 8>(e, a, st);                    \
        default: return YG_ERR_UNSUPPORTED;                                                                        \
        }                                                                                                          \
    }                                                                                                              \
    int yg_launch_logpost_d##D(yg_ensemble *e, int level, const double *theta, int64_t n, double *out,             \
                               cudaStream_t st, int cdd)                                                           \
    {                                                                                                              \
        switch (cdd) {                                                                                             \
        case 2: return launch_logpost_t<D, 2>(e, level, theta, n, out, st);                                        \
        case 4: return launch_logpost_t<D, 4>(e, level, theta, n, out, st);                                        \
        case 8: return launch_logpost_t<D, 8>(e, level, theta, n, out, st);                                        \
        default: return YG_ERR_UNSUPPORTED;                                                                        \
        }                                                                                                          \
    }
#endif
