// common.cuh -- device-side building blocks shared by the sm_100a kernels of
// libyagre_b200: problem blob layout, Philox4x32-10 streams, Box-Muller,
// the reference's acceptance / equality rules and its summation orders.
//
// Reference (rkutri/yagre-mcmc) lines are cited where a rule is restated.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <math.h>
#include <math_constants.h>
#include "../../include/yagre_b200.h"

#define YG_DEVFN __device__ __forceinline__
#define YG_HDFN __host__ __device__ __forceinline__

// Bounds-checked development build (`make -C yagre_mcmc_b200/csrc checked`, -DYG_BOUNDS_CHECK): every computed index
// into a shared-memory carve-up or a caller-provided device buffer is asserted against the extent of that array
// (compute-sanitizer is not available on the B200 pool, profiles/r02_summary.md).  In the product build the macro
// expands to nothing and the SASS is unchanged.
#ifdef YG_BOUNDS_CHECK
#include <cassert>
#define YG_CHK(idx, limit) assert((long long)(idx) >= 0 && (long long)(idx) < (long long)(limit))
YG_DEVFN uint32_t yg_dynamic_smem_bytes()
{
    uint32_t v;
    asm volatile("mov.u32 %0, %%dynamic_smem_size;" : "=r"(v));
    return v;
}
#else
#define YG_CHK(idx, limit) ((void)0)
#endif

// ---------------------------------------------------------------------------
// Device problem blob: one contiguous, 16-byte aligned buffer per handle that
// kernels stage into shared memory (one TMA bulk copy in the LV kernel).
// ---------------------------------------------------------------------------
struct DevLevel {
    double g_mean[YG_MAX_DIM];
    double g_prec[YG_MAX_DIM * YG_MAX_DIM];
    double g_logconst;
    double noise_prec[YG_MAX_DATA_DIM * YG_MAX_DATA_DIM];
    double prior_mean[YG_MAX_DIM];
    double prior_prec[YG_MAX_DIM * YG_MAX_DIM];
    double G[YG_MAX_DATA_DIM * YG_MAX_DIM];
    double b[YG_MAX_DATA_DIM];
    double alpha, gamma, T;
    double tempering;      // logL multiplier: 1 unless the level is a TemperedUnnormalisedPosterior (target.py:25-43)
    double _padt;
    int32_t rk4_steps, n_data, data_dim;
    int32_t data_off;      // offsets (in doubles) into DevProblem::tail
    int32_t design_off;
    int32_t _pad[3];
};

struct DevProblemHeader {
    int32_t model, dim, n_levels, J, eq_mode, tail_len;
    int32_t proposal;          // yg_proposal
    int32_t _pad;
    double pcn_a, pcn_b;       // sqrt(1 - 2h), sqrt(2h)   (pcn.py:30-35)
    double pcn_mean[YG_MAX_DIM];
    double prop_L[YG_MAX_DIM * YG_MAX_DIM];
    DevLevel lvl[YG_MAX_LEVELS];
    // followed by double tail[tail_len]: per level data[n_data*data_dim], design[n_data*2]
};
static_assert(sizeof(DevLevel) % 16 == 0, "DevLevel must keep 16-byte alignment");
static_assert(sizeof(DevProblemHeader) % 16 == 0, "header must keep 16-byte alignment");

YG_DEVFN const double *dev_tail(const DevProblemHeader *h)
{
    return reinterpret_cast<const double *>(h + 1);
}

// ---------------------------------------------------------------------------
// Philox4x32-10 (Salmon et al., SC'11).  Stream keying (DESIGN.md):
//   key = (seed lo, seed hi)
//   ctr = (chain lo32, step lo32, step hi32, chain_hi8<<24 | sub<<8 | slot)
//   sub  = coarse sub-step j, or 0xFFFF for the fine / single-level screen
//   slot = b for the b-th pair of normals, 0xFF for the accept uniform
// ---------------------------------------------------------------------------
#define YG_SUB_FINE 0xFFFFu
#define YG_SLOT_U 0xFFu

YG_DEVFN uint4 philox4x32_10(uint4 c, uint2 k)
{
#pragma unroll
    for (int r = 0; r < 10; r++) {
        const uint32_t hi0 = __umulhi(0xD2511F53u, c.x), lo0 = 0xD2511F53u * c.x;
        const uint32_t hi1 = __umulhi(0xCD9E8D57u, c.z), lo1 = 0xCD9E8D57u * c.z;
        c = make_uint4(hi1 ^ c.y ^ k.x, lo1, hi0 ^ c.w ^ k.y, lo0);
        k.x += 0x9E3779B9u;
        k.y += 0xBB67AE85u;
    }
    return c;
}

YG_DEVFN uint4 philox_block(uint64_t seed, uint64_t chain, uint64_t step, uint32_t sub, uint32_t slot)
{
    const uint2 key = make_uint2((uint32_t)seed, (uint32_t)(seed >> 32));
    const uint4 ctr = make_uint4((uint32_t)chain, (uint32_t)step, (uint32_t)(step >> 32),
                                 (uint32_t)(((chain >> 32) & 0xFFu) << 24) | (sub << 8) | slot);
    return philox4x32_10(ctr, key);
}

YG_DEVFN double u53(uint32_t hi, uint32_t lo)
{
    return (double)((((uint64_t)hi << 32) | lo) >> 11) * 0x1.0p-53;
}

YG_DEVFN double philox_uniform(uint64_t seed, uint64_t chain, uint64_t step, uint32_t sub)
{
    const uint4 w = philox_block(seed, chain, step, sub, YG_SLOT_U);
    return u53(w.x, w.y);                                   // [0,1), like numpy.random.uniform
}

// Box-Muller on one Philox block -> two standard normals.
YG_DEVFN void philox_normal_pair(uint64_t seed, uint64_t chain, uint64_t step, uint32_t sub, uint32_t b,
                                 double &z0, double &z1)
{
    const uint4 w = philox_block(seed, chain, step, sub, b);
    const double u1 = u53(w.x, w.y) + 0x1.0p-53;            // (0,1]
    const double u2 = u53(w.z, w.w);
    const double R = sqrt(-2.0 * log(u1));
    double s, c;
    sincospi(2.0 * u2, &s, &c);
    z0 = R * c;
    z1 = R * s;
}

// ---------------------------------------------------------------------------
// Rules of the reference step
// ---------------------------------------------------------------------------

// mrw.py:54-57, mlda.py:148-154, metropolisHastings.py:68-73:
//   r = exp(delta); a = r if r < 1. else 1.; accept iff u <= a   (NaN -> a = 1 -> accept)
YG_HDFN bool accept_rule(double delta, double u)
{
    const double r = exp(delta);
    const double a = (r < 1.0) ? r : 1.0;
    return u <= a;
}

// Misfit budget of a proposal whose acceptance is accept_rule(t * (-S / 2) + lp - lps, u), S = sum of the
// misfits q_n >= 0: a partial sum of q above the budget certifies the rejection, so the remaining forward
// evaluations can be skipped.  The margin (relative 1e-9 of every term) covers the rounding of log / exp,
// of the product by t, of the sums and of summing S in another order than np_sum_le128.  Returns +inf (never
// skip) when the rule is not monotone in S or a term is not finite: u == 0 always accepts, and a NaN delta
// (lps = -inf) accepts too.
YG_HDFN double reject_budget(double lp, double lps, double u, double t)
{
    if (!(u > 0.0) || !(t > 0.0) || !isfinite(t)) return (double)INFINITY;
    const double lu = log(u);
    const double d = lp - lps - lu;
    const double m = fabs(lp) + fabs(lps) + fabs(lu) + 1.0;
    if (!isfinite(d) || !isfinite(m)) return (double)INFINITY;
    const double b = 2.0 * (d + 1e-9 * m) / t;
    return b > 0.0 ? b * (1.0 + 1e-9) : b;
}

// parameter/scalar.py:38-43: math.isclose(a, b) with rel_tol = 1e-9, abs_tol = 0
YG_DEVFN bool isclose_rule(double x, double y)
{
    if (x == y) return true;
    if (isinf(x) || isinf(y)) return false;
    const double diff = fabs(y - x);
    return (diff <= fabs(1e-9 * y)) || (diff <= fabs(1e-9 * x));
}

// numpy's pairwise summation over a contiguous vector (np.sum in likelihood.py:80).
// stride lets the caller walk a shared-memory column.
YG_HDFN double np_sum_le128(const double *a, int n, int stride)
{
    if (n < 8) {
        double res = 0.0;
        for (int i = 0; i < n; i++) res += a[i * stride];
        return res;
    }
    double r0 = a[0], r1 = a[stride], r2 = a[2 * stride], r3 = a[3 * stride];
    double r4 = a[4 * stride], r5 = a[5 * stride], r6 = a[6 * stride], r7 = a[7 * stride];
    int i = 8;
    for (; i < n - (n % 8); i += 8) {
        r0 += a[(i + 0) * stride]; r1 += a[(i + 1) * stride]; r2 += a[(i + 2) * stride]; r3 += a[(i + 3) * stride];
        r4 += a[(i + 4) * stride]; r5 += a[(i + 5) * stride]; r6 += a[(i + 6) * stride]; r7 += a[(i + 7) * stride];
    }
    double res = ((r0 + r1) + (r2 + r3)) + ((r4 + r5) + (r6 + r7));
    for (; i < n; i++) res += a[i * stride];
    return res;
}

__device__ inline double np_pairwise_sum(const double *a, int n, int stride)
{
    if (n <= 128) return np_sum_le128(a, n, stride);
    int n2 = n / 2;
    n2 -= n2 % 8;
    return np_pairwise_sum(a, n2, stride) + np_pairwise_sum(a + (size_t)n2 * stride, n - n2, stride);
}

// x' P x, P applied first (covariance.py:19-22); exact zeros of P are skipped so a
// diagonal precision reproduces DiagonalCovarianceMatrix (covariance.py:54-55) for x = inf.
template <int CAP>
YG_DEVFN double quad_form(const double *P, int ld, const double (&x)[CAP], int n)
{
    double acc = 0.0;
#pragma unroll
    for (int k = 0; k < CAP; k++) {
        if (k < n) {
            double pk = 0.0;
            bool first = true;
#pragma unroll
            for (int l = 0; l < CAP; l++) {
                if (l < n) {
                    const double p = P[k * ld + l];
                    if (p != 0.0) {
                        pk = first ? p * x[l] : fma(p, x[l], pk);
                        first = false;
                    }
                }
            }
            acc = (k == 0) ? x[k] * pk : fma(x[k], pk, acc);
        }
    }
    return acc;
}

// ---------------------------------------------------------------------------
// host-side error plumbing (abi.cu)
// ---------------------------------------------------------------------------
void yg_set_error(const char *fmt, ...);

#define YG_CUDA_CHECK(expr)                                                           \
    do {                                                                              \
        cudaError_t _e = (expr);                                                      \
        if (_e != cudaSuccess) {                                                      \
            yg_set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e),      \
                         __FILE__, __LINE__);                                         \
            return YG_ERR_CUDA;                                                       \
        }                                                                             \
    } while (0)
