// diag_kernels.cu -- post-processing on the device: integrated autocorrelation time /
// ESS per chain, pooled sufficient statistics, split-half moments (R-hat inputs) and
// the DFMA micro-benchmark that provides the FP64 roofline denominator.
//
// Reference semantics restated (rkutri/yagre-mcmc):
//   ACF                   postprocessing/autocorrelation.py:5-29 (centre, correlate, / lag 0)
//   Sokal window + IAT    postprocessing/autocorrelation.py:32-89
//   'mean' / 'max'        postprocessing/autocorrelation.py:92-140
//   ESS idiom             example_inference_lotkaVolterra_twoLevel.py:117-118,132
//   Welford moments       statistics/estimation.py:4-58
// R-hat and pooling do not exist in the reference (single chain); they are new.
#include "ensemble.h"
#include "lv_model.cuh"
#include <math_constants.h>

namespace {

constexpr int IAT_THREADS = 128;
constexpr int IAT_LAGS = 4;

// block-wide sums of IAT_LAGS values, fixed tree -> deterministic
__device__ void block_sum4(double (&v)[IAT_LAGS], double *red /* [4][IAT_LAGS] */)
{
#pragma unroll
    for (int k = 0; k < IAT_LAGS; k++)
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v[k] += __shfl_xor_sync(0xffffffffu, v[k], o);
    const int w = threadIdx.x >> 5;
    __syncthreads();
    if ((threadIdx.x & 31) == 0) {
#pragma unroll
        for (int k = 0; k < IAT_LAGS; k++) red[w * IAT_LAGS + k] = v[k];
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < IAT_LAGS; k++) {
        double s = 0.0;
        for (int ww = 0; ww < IAT_THREADS / 32; ww++) s += red[ww * IAT_LAGS + k];
        v[k] = s;
    }
}

// One CTA per chain.  The series is staged contiguously -- in shared memory, or for series longer
// than 25,600 samples (C2 / C3 run 100,000 / 50,000 steps) in a per-CTA slice of a global scratch
// buffer that stays L2 resident; lags are produced four at a time until Sokal's criterion
// M >= c * tau(M) is met (autocorrelation.py:53-59: argmin of the boolean "M < c*tau[M]" = first
// False; all True -> index 0).
__global__ void __launch_bounds__(IAT_THREADS) iat_kernel(const double *samples, int64_t ns, int d, int64_t nc,
                                                          int method, double sokal, int64_t *iat_out,
                                                          int64_t *ess_out, double *scratch)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    double *x = scratch ? scratch + (size_t)blockIdx.x * (size_t)ns : reinterpret_cast<double *>(smem_raw);   // [ns]
    __shared__ double red[(IAT_THREADS / 32) * IAT_LAGS];
    const int tid = threadIdx.x;
    for (int64_t chain = blockIdx.x; chain < nc; chain += gridDim.x) {
        long long best = 0;
        bool degenerate = false;         // block-uniform: derived from block_sum4 results only
        const int n_series = (method == 0) ? 1 : d;
        for (int k = 0; k < n_series; k++) {
            __syncthreads();
            for (int64_t i = tid; i < ns; i += IAT_THREADS) {
                if (method == 0) {                               // np.mean(seq, axis=1)
                    double s = 0.0;
                    for (int kk = 0; kk < d; kk++) s += samples[(i * d + kk) * nc + chain];
                    x[i] = s / (double)d;
                } else {
                    x[i] = samples[(i * d + k) * nc + chain];
                }
            }
            __syncthreads();
            double v[IAT_LAGS] = {0.0, 0.0, 0.0, 0.0};
            for (int64_t i = tid; i < ns; i += IAT_THREADS) v[0] += x[i];
            block_sum4(v, red);
            const double mean = v[0] / (double)ns;
            __syncthreads();
            for (int64_t i = tid; i < ns; i += IAT_THREADS) x[i] -= mean;
            __syncthreads();
            double acf0 = 0.0, cum = 0.0;
            long long result = 1;                                // all-True window -> tau[0] = 1
            bool done = false;
            for (int64_t M0 = 0; M0 < ns && !done; M0 += IAT_LAGS) {
#pragma unroll
                for (int l = 0; l < IAT_LAGS; l++) v[l] = 0.0;
                for (int64_t i = tid; i + M0 < ns; i += IAT_THREADS) {
                    const double xi = x[i];
#pragma unroll
                    for (int l = 0; l < IAT_LAGS; l++)
                        if (i + M0 + l < ns) v[l] = fma(xi, x[i + M0 + l], v[l]);
                }
                block_sum4(v, red);
                if (M0 == 0) {
                    acf0 = v[0];
                    // A constant (stuck / never accepted) or non-finite series has no autocorrelation function:
                    // 0/0 in the reference (autocorrelation.py:26-29; it fails on the NaNs).  A batched call cannot
                    // raise per chain, so such a chain reports IAT = n_samples and ESS = 0 -- never a full ESS.
                    if (!(acf0 > 0.0) || !isfinite(acf0)) { degenerate = true; break; }
                }
#pragma unroll
                for (int l = 0; l < IAT_LAGS; l++) {
                    const int64_t M = M0 + l;
                    if (!done && M < ns) {
                        cum += v[l] / acf0;
                        const double tau = 2.0 * cum - 1.0;
                        if (!isfinite(tau)) { degenerate = true; done = true; }
                        else if (!((double)M < sokal * tau)) {
                            result = (long long)rint(tau);
                            done = true;
                        }
                    }
                }
            }
            if (k == 0 || result > best) best = result;
        }
        if (tid == 0) {
            if (iat_out) iat_out[chain] = degenerate ? (long long)ns : best;
            if (ess_out) ess_out[chain] = degenerate ? 0 : ns / (best > 0 ? best : 1);
        }
    }
}

// Per-chain mean / unbiased variance of the two halves of the stored series.
__global__ void split_moments_kernel(const double *samples, int64_t ns, int d, int64_t nc, double *hm, double *hv)
{
    const int64_t total = (int64_t)d * nc;
    const int64_t half = ns / 2;
    for (int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; t < total; t += (int64_t)gridDim.x * blockDim.x) {
        const int64_t chain = t % nc;
        const int k = (int)(t / nc);
        for (int h = 0; h < 2; h++) {
            double mean = 0.0, m2 = 0.0;
            const int64_t lo = h * half;
            for (int64_t i = 0; i < half; i++) {
                const double x = samples[((lo + i) * d + k) * nc + chain];
                const double dl = x - mean;
                mean += dl / (double)(i + 1);
                m2 = fma(dl, x - mean, m2);
            }
            hm[((int64_t)h * d + k) * nc + chain] = mean;
            hv[((int64_t)h * d + k) * nc + chain] = half > 1 ? m2 / (double)(half - 1) : CUDART_NAN;
        }
    }
}

// Pooled sufficient statistics: stage 1 writes one partial vector per CTA, stage 2 adds the
// partials in index order -- deterministic, no floating-point atomics.
constexpr int POOL_THREADS = 256;

__global__ void __launch_bounds__(POOL_THREADS) pooled_stage1(const double *w_mean, const double *w_m2,
                                                              const unsigned long long *n_accept, int d, int64_t nc,
                                                              double welford_n, double *partials, int len)
{
    extern __shared__ double sh[];                     // [POOL_THREADS/32][len]
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int q = 0; q < len; q++) {
        double v = 0.0;
        for (int64_t c = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; c < nc; c += (int64_t)gridDim.x * blockDim.x) {
            if (q == 0) v += 1.0;
            else if (q == 1) v = welford_n;            // not a sum: identical on every chain
            else if (q == 2) v += (double)n_accept[c];
            else {
                int r = q - 3;
                if (r < d) v += w_mean[(int64_t)r * nc + c];
                else if ((r -= d) < d * d) v += w_mean[(int64_t)(r / d) * nc + c] * w_mean[(int64_t)(r % d) * nc + c];
                else if ((r -= d * d) < d * d) v += w_m2[(int64_t)r * nc + c];
                else {
                    r -= d * d;
                    v += welford_n > 1.0 ? w_m2[(int64_t)(r * d + r) * nc + c] / (welford_n - 1.0) : 0.0;
                }
            }
        }
        if (q != 1) {
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
        }
        if (lane == 0) sh[warp * len + q] = v;
    }
    __syncthreads();
    for (int q = threadIdx.x; q < len; q += blockDim.x) {
        double s = 0.0;
        if (q == 1) s = welford_n;
        else for (int w = 0; w < POOL_THREADS / 32; w++) s += sh[w * len + q];
        partials[(int64_t)blockIdx.x * len + q] = s;
    }
}

__global__ void pooled_stage2(const double *partials, int n_part, int len, double *out)
{
    for (int q = blockIdx.x * blockDim.x + threadIdx.x; q < len; q += gridDim.x * blockDim.x) {
        double s = 0.0;
        if (q == 1) s = partials[q];
        else for (int b = 0; b < n_part; b++) s += partials[(int64_t)b * len + q];
        out[q] = s;
    }
}

// Pooled sufficient statistics of a stored sample buffer x[ns, d, nc] (yg_pooled_samples), for any d <= 64.
//
// Each warp takes groups of 4 consecutive chains; the K dimension of a symmetric rank-K update is the (sample, chain)
// pairs of a group, 4 per m16n8k4 DMMA.  Lane (g = lane / 4, q = lane % 4) holds coordinates 8 m + g (m < G) of chain
// 4 gi + q, which is at once its A fragment (rows 16 I + g and 16 I + 8 + g: values m = 2 I, 2 I + 1) and its B fragment
// (column 8 J + g: value m = J) -- no shuffles, no shared-memory staging.  Only the output tiles (I, J) with
// J <= 2 I + 1 are issued: those cover the lower triangle (20 of 32 at d = 64); the diagonal tiles' upper halves are
// computed and dropped, the lower triangle is mirrored on write.
//
// Centred one-pass form: chain c is shifted by its first stored sample s_c, y = x - s_c, and
//   M2_c = sum_t y y' - S1_c S1_c' / ns,  S1_c = sum_t y,  mean_c = s_c + S1_c / ns,
// so the cancellation is relative to the chain's own spread, not to |x| (tests/pooled_samples_reference.py derives
// the bound).  The correction is one more DMMA step per group with B = -S1 / ns.
//
// Pass 1 reads the buffer once and writes each chain's mean to the workspace; pass 2 re-reads the means (d doubles
// per chain: 1 / ns of pass 1) for sum_c mean_c mean_c' with the same accumulator registers.  ns == 1 skips pass 1:
// the means are row 0 of the buffer.  Per-CTA partial vectors, warps added in a fixed order, then pooled_stage2:
// deterministic, no atomics.
constexpr int PS_WARPS = 4;
constexpr int PS_CHAINS_PER_CTA = 4 * PS_WARPS;
constexpr int PS_MAX_PARTS = 4 * 148;       // at most 4 CTAs on each of the B200's 148 SMs

YG_DEVFN void dmma_m16n8k4(double (&c)[4], double a0, double a1, double b0)
{
    asm volatile("mma.sync.aligned.m16n8k4.row.col.f64.f64.f64.f64 {%0,%1,%2,%3}, {%4,%5}, {%6}, {%0,%1,%2,%3};"
                 : "+d"(c[0]), "+d"(c[1]), "+d"(c[2]), "+d"(c[3])
                 : "d"(a0), "d"(a1), "d"(b0));
}

// acc[I][J] += A B over the 4 pairs of one k-step, lower tiles only.
template <int G>
YG_DEVFN void syrk_step(double (&acc)[(G + 1) / 2][G][4], const double (&a)[G], const double (&b)[G])
{
#pragma unroll
    for (int I = 0; I < (G + 1) / 2; I++)
#pragma unroll
        for (int J = 0; J < G; J++)
            if (J <= 2 * I + 1) dmma_m16n8k4(acc[I][J], a[2 * I], 2 * I + 1 < G ? a[2 * I + 1] : 0.0, b[J]);
}

// R[r * d + col] (col <= r) = sum over the CTA's warps, in warp order, of the accumulators.
template <int G>
YG_DEVFN void flush_lower(double (&acc)[(G + 1) / 2][G][4], double *R, int d, int smem_len)
{
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, g = lane >> 2, q = lane & 3;
    for (int w = 0; w < PS_WARPS; w++) {
        if (warp == w) {
#pragma unroll
            for (int I = 0; I < (G + 1) / 2; I++)
#pragma unroll
                for (int J = 0; J < G; J++)
                    if (J <= 2 * I + 1) {
#pragma unroll
                        for (int e = 0; e < 4; e++) {
                            const int r = 16 * I + g + (e >= 2 ? 8 : 0), col = 8 * J + 2 * q + (e & 1);
                            if (r < d && col <= r) {
                                YG_CHK(r * d + col, smem_len);
                                R[r * d + col] = (w == 0 ? 0.0 : R[r * d + col]) + acc[I][J][e];
                            }
                        }
                    }
        }
        __syncthreads();
    }
}

template <int G>
__global__ void __launch_bounds__(PS_WARPS * 32) pooled_samples_kernel(const double *__restrict__ x, int64_t ns, int d,
                                                                       int64_t nc, double *partials, int len,
                                                                       double *means)
{
    constexpr int RB = (G + 1) / 2;
    constexpr int U = G >= 8 ? 1 : 8 / G;          // samples per iteration: about 8 loads in flight per lane
    constexpr int DP = 8 * G;
    extern __shared__ double sm[];                  // R[d * d] | sum of means [warp][q][DP] | sum of variances, same
    [[maybe_unused]] const int smem_len = d * d + 2 * PS_WARPS * 4 * DP;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, g = lane >> 2, q = lane & 3;
    double *R = sm;
    const int slot = d * d + (warp * 4 + q) * DP;   // this lane's slots (coordinates 8 m + g of its chains)
    const int vslot = slot + PS_WARPS * 4 * DP;
#pragma unroll
    for (int m = 0; m < G; m++) {
        YG_CHK(vslot + 8 * m + g, smem_len);
        sm[slot + 8 * m + g] = 0.0;
        sm[vslot + 8 * m + g] = 0.0;
    }
    __syncthreads();
    const int64_t n_groups = (nc + 3) / 4, tw = (int64_t)gridDim.x * PS_WARPS;
    [[maybe_unused]] const int64_t x_len = ns * d * nc, m_len = (int64_t)d * nc;     // YG_CHK extents
    double *part = partials + (int64_t)blockIdx.x * len;
    [[maybe_unused]] const int part_len = gridDim.x * len;
    const int o_mean = 3, o_mm = o_mean + d, o_m2 = o_mm + d * d, o_var = o_m2 + d * d;
    double acc[RB][G][4];

    if (ns > 1) {
#pragma unroll
        for (int I = 0; I < RB; I++)
#pragma unroll
            for (int J = 0; J < G; J++) acc[I][J][0] = acc[I][J][1] = acc[I][J][2] = acc[I][J][3] = 0.0;
        const double inv_n = 1.0 / (double)ns;
        for (int64_t gi = (int64_t)blockIdx.x * PS_WARPS + warp; gi < n_groups; gi += tw) {
            const int64_t c = 4 * gi + q;
            const bool ok = c < nc;
            double s[G], S1[G], Q[G];
#pragma unroll
            for (int m = 0; m < G; m++) {
                const int i = 8 * m + g;
                if (ok && i < d) YG_CHK((int64_t)i * nc + c, x_len);
                s[m] = (ok && i < d) ? __ldg(x + (int64_t)i * nc + c) : 0.0;
                S1[m] = Q[m] = 0.0;
            }
            // software pipeline: the loads of iteration t + U are in flight during the DMMAs of iteration t
            double xn[U][G];
            auto load = [&](int64_t t0) {
#pragma unroll
                for (int u = 0; u < U; u++)
#pragma unroll
                    for (int m = 0; m < G; m++) {
                        const int i = 8 * m + g;
                        const int64_t idx = ((t0 + u) * d + i) * nc + c;
                        const bool in = ok && i < d && t0 + u < ns;
                        if (in) YG_CHK(idx, x_len);
                        xn[u][m] = in ? __ldg(x + idx) : s[m];
                    }
            };
            load(0);
            for (int64_t t = 0; t < ns; t += U) {
                double y[U][G];
#pragma unroll
                for (int u = 0; u < U; u++)
#pragma unroll
                    for (int m = 0; m < G; m++) y[u][m] = xn[u][m] - s[m];
                load(t + U);
#pragma unroll
                for (int u = 0; u < U; u++) {
#pragma unroll
                    for (int m = 0; m < G; m++) {
                        S1[m] += y[u][m];
                        Q[m] = fma(y[u][m], y[u][m], Q[m]);
                    }
                    syrk_step<G>(acc, y[u], y[u]);
                }
            }
            double nS[G];
#pragma unroll
            for (int m = 0; m < G; m++) nS[m] = -(S1[m] * inv_n);
            syrk_step<G>(acc, S1, nS);                              // - sum_c S1_c S1_c' / ns
#pragma unroll
            for (int m = 0; m < G; m++) {
                const int i = 8 * m + g;
                if (ok && i < d) {
                    YG_CHK((int64_t)i * nc + c, m_len);
                    means[(int64_t)i * nc + c] = s[m] + S1[m] * inv_n;
                    sm[vslot + 8 * m + g] += (Q[m] - S1[m] * (S1[m] * inv_n)) / (double)(ns - 1);
                }
            }
        }
        flush_lower<G>(acc, R, d, smem_len);
    }
    for (int k = tid; k < d * d; k += blockDim.x) {
        const int r = max(k / d, k % d), col = min(k / d, k % d);
        YG_CHK(r * d + col, smem_len);
        YG_CHK((int64_t)blockIdx.x * len + o_m2 + k, part_len);
        part[o_m2 + k] = ns > 1 ? R[r * d + col] : 0.0;
    }
    for (int i = tid; i < d; i += blockDim.x) {
        double v = 0.0;
        for (int w = 0; w < PS_WARPS * 4; w++) {
            YG_CHK(d * d + PS_WARPS * 4 * DP + w * DP + i, smem_len);
            v += sm[d * d + PS_WARPS * 4 * DP + w * DP + i];
        }
        YG_CHK((int64_t)blockIdx.x * len + o_var + i, part_len);
        part[o_var + i] = v;
    }
    __syncthreads();                                    // R is reused below

    // pass 2: sum_c mean_c mean_c' and sum_c mean_c
    const double *mb = ns > 1 ? means : x;             // [d, nc]; for ns == 1 row 0 of the buffer
#pragma unroll
    for (int I = 0; I < RB; I++)
#pragma unroll
        for (int J = 0; J < G; J++) acc[I][J][0] = acc[I][J][1] = acc[I][J][2] = acc[I][J][3] = 0.0;
    for (int64_t gi = (int64_t)blockIdx.x * PS_WARPS + warp; gi < n_groups; gi += tw) {
        const int64_t c = 4 * gi + q;
        const bool ok = c < nc;
        double mv[G];
#pragma unroll
        for (int m = 0; m < G; m++) {
            const int i = 8 * m + g;
            if (ok && i < d) YG_CHK((int64_t)i * nc + c, m_len);
            mv[m] = (ok && i < d) ? mb[(int64_t)i * nc + c] : 0.0;     // pass 1 of this thread wrote `means`
            if (ok && i < d) sm[slot + 8 * m + g] += mv[m];
        }
        syrk_step<G>(acc, mv, mv);
    }
    flush_lower<G>(acc, R, d, smem_len);
    for (int k = tid; k < d * d; k += blockDim.x) {
        const int r = max(k / d, k % d), col = min(k / d, k % d);
        YG_CHK(r * d + col, smem_len);
        YG_CHK((int64_t)blockIdx.x * len + o_mm + k, part_len);
        part[o_mm + k] = R[r * d + col];
    }
    for (int i = tid; i < d; i += blockDim.x) {
        double v = 0.0;
        for (int w = 0; w < PS_WARPS * 4; w++) {
            YG_CHK(d * d + w * DP + i, smem_len);
            v += sm[d * d + w * DP + i];
        }
        YG_CHK((int64_t)blockIdx.x * len + o_mean + i, part_len);
        part[o_mean + i] = v;
    }
    if (tid == 0) {
        YG_CHK((int64_t)blockIdx.x * len + 2, part_len);
        int64_t chains = 0;
        for (int w = 0; w < PS_WARPS; w++)
            for (int64_t gi = (int64_t)blockIdx.x * PS_WARPS + w; gi < n_groups; gi += tw)
                chains += min((int64_t)4, nc - 4 * gi);
        part[0] = (double)chains;
        part[1] = (double)ns;
        part[2] = 0.0;
    }
}

int64_t ps_parts_max(int64_t nc)
{
    return std::min<int64_t>(PS_MAX_PARTS, (nc + PS_CHAINS_PER_CTA - 1) / PS_CHAINS_PER_CTA);
}

template <int G>
int launch_pooled_samples(const double *x, int64_t ns, int d, int64_t nc, double *ws, double *out, cudaStream_t st)
{
    const int len = (int)yg_pooled_len(d);
    const size_t smem = sizeof(double) * ((size_t)d * d + 2 * PS_WARPS * 4 * 8 * G);     // <= 48 KiB at d = 64
    int dev = 0, sms = 148, per_sm = 1;
    YG_CUDA_CHECK(cudaGetDevice(&dev));
    YG_CUDA_CHECK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    YG_CUDA_CHECK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, pooled_samples_kernel<G>, PS_WARPS * 32, smem));
    const int64_t parts_max = ps_parts_max(nc);
    const int grid = (int)std::max<int64_t>(1, std::min<int64_t>(parts_max, (int64_t)sms * std::min(per_sm, 4)));
    double *means = ws + parts_max * len;
    pooled_samples_kernel<G><<<grid, PS_WARPS * 32, smem, st>>>(x, ns, d, nc, ws, len, means);
    YG_CUDA_CHECK(cudaGetLastError());
    pooled_stage2<<<(len + 127) / 128, 128, 0, st>>>(ws, grid, len, out);
    YG_CUDA_CHECK(cudaGetLastError());
    return YG_OK;
}

// FP64-pipe micro-benchmarks, 1024 resident threads/SM.  Variant 0: eight independent
// DFMA chains per thread.  Variant 1: four interleaved LV RK4 steps per thread (the hot
// loop's own instruction mix: 30 FP64-pipe instructions per step, DFMA/DMUL/DADD).  Both
// count 2 flop per FP64-pipe instruction, i.e. they measure the DFMA-equivalent peak.
__global__ void __launch_bounds__(256, 4) dfma_peak_kernel(double *sink, int iters, double a, double b)
{
    double v0 = threadIdx.x * 1e-3, v1 = v0 + 1.0, v2 = v0 + 2.0, v3 = v0 + 3.0;
    double v4 = v0 + 4.0, v5 = v0 + 5.0, v6 = v0 + 6.0, v7 = v0 + 7.0;
#pragma unroll 1
    for (int i = 0; i < iters; i++) {
#pragma unroll
        for (int k = 0; k < 8; k++) {
            v0 = fma(v0, a, b); v1 = fma(v1, a, b); v2 = fma(v2, a, b); v3 = fma(v3, a, b);
            v4 = fma(v4, a, b); v5 = fma(v5, a, b); v6 = fma(v6, a, b); v7 = fma(v7, a, b);
        }
    }
    const double s = ((v0 + v1) + (v2 + v3)) + ((v4 + v5) + (v6 + v7));
    if (s == 123.456) sink[0] = s;                      // keeps the chains live
}

// FP64-pipe peak probe, second instruction mix: 30 DFMA/DMUL/DADD per iteration and lane, every one
// with at most two vector-register sources (the third is a constant-bank operand), two independent
// dependency chains -- the mix of the k-form RK4 step.  Measures the pipe, not a model.
__global__ void __launch_bounds__(256, 4) mix_peak_kernel(double *sink, int iters, double b0, double d0, double ha,
                                                          double hg)
{
    double hb[4], hd[4], x[4], y[4];
#pragma unroll
    for (int i = 0; i < 4; i++) {
        hb[i] = b0 + 1e-6 * (threadIdx.x + i);
        hd[i] = d0 + 1e-6 * i;
        x[i] = 1.0 + 1e-3 * threadIdx.x;
        y[i] = 0.8 + 1e-3 * i;
    }
#pragma unroll 1
    for (int s = 0; s < iters; s++) {
#pragma unroll
        for (int i = 0; i < 4; i++) {
            double kx = x[i] * fma(-hb[i], y[i], ha), ky = y[i] * fma(hd[i], x[i], -hg);
            double xs = fma(0.5, kx, x[i]), ys = fma(0.5, ky, y[i]);
            double ax = fma(0.125, kx, x[i]), ay = fma(0.125, ky, y[i]);
            kx = xs * fma(-hb[i], ys, ha); ky = ys * fma(hd[i], xs, -hg);
            xs = fma(0.5, kx, x[i]); ys = fma(0.5, ky, y[i]);
            ax = fma(0.25, kx, ax); ay = fma(0.25, ky, ay);
            kx = xs * fma(-hb[i], ys, ha); ky = ys * fma(hd[i], xs, -hg);
            xs = x[i] + kx; ys = y[i] + ky;
            ax = fma(0.25, kx, ax); ay = fma(0.25, ky, ay);
            kx = xs * fma(-hb[i], ys, ha); ky = ys * fma(hd[i], xs, -hg);
            x[i] = fma(0.125, kx, ax);
            y[i] = fma(0.125, ky, ay);
        }
    }
    const double s = (x[0] + y[0]) + (x[1] + y[1]) + (x[2] + y[2]) + (x[3] + y[3]);
    if (s == 1.2345) sink[0] = s;
}

// The bare RK4 integrator of lv_model.cuh (20 FP64 instructions per step), one integration per thread,
// 1024 threads per SM like lv_mh_kernel: the ceiling of RK4 steps/s for the LV step kernel.
__global__ void __launch_bounds__(1024, 1) rk4_loop_kernel(double *sink, int n_steps, double h, LvStepConsts kc)
{
    const LvRates r = lv_rates(h, 0.4 * (1.0 + 1e-3 * (threadIdx.x & 63)), 0.6 * (1.0 + 2e-3 * (threadIdx.x & 31)));
    double x = 0.5 + (threadIdx.x & 15) / 16.0, y = 1.5 - (threadIdx.x & 7) / 8.0;
    lv_integrate(kc, r, n_steps, x, y);
    if (x + y == 1.2345) sink[0] = x;
}

}  // namespace

extern "C" int yg_iat_ess(const double *samples_dev, int64_t n_samples, int32_t d, int64_t n_chains,
                          int32_t method, double sokal_const, int64_t *iat_dev, int64_t *ess_dev, void *stream)
{
    if (!samples_dev || n_samples < 2 || d < 1 || n_chains < 1 || (method != 0 && method != 1)) {
        yg_set_error("yg_iat_ess: invalid arguments");
        return YG_ERR_INVALID;
    }
    size_t smem = sizeof(double) * (size_t)n_samples;
    const bool long_series = smem > 200 * 1024;
    if (long_series) smem = 0;
    else YG_CUDA_CHECK(cudaFuncSetAttribute(iat_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    const int per_sm = long_series ? 2 : (int)std::max<size_t>(1, std::min<size_t>(8, (220 * 1024) / (smem + 1024)));
    const int grid = (int)std::min<int64_t>(n_chains, (int64_t)sms * per_sm);
    cudaStream_t st = (cudaStream_t)stream;
    double *scratch = nullptr;
    if (long_series)     // stream-ordered scratch (one contiguous copy of the series per CTA): no host synchronisation
        YG_CUDA_CHECK(cudaMallocAsync((void **)&scratch, sizeof(double) * (size_t)grid * (size_t)n_samples, st));
    iat_kernel<<<grid, IAT_THREADS, smem, st>>>(samples_dev, n_samples, d, n_chains, method, sokal_const,
                                                (int64_t *)iat_dev, (int64_t *)ess_dev, scratch);
    YG_CUDA_CHECK(cudaGetLastError());
    if (long_series) YG_CUDA_CHECK(cudaFreeAsync(scratch, st));
    return YG_OK;
}

extern "C" int yg_split_moments(const double *samples_dev, int64_t n_samples, int32_t d, int64_t n_chains,
                                double *half_mean_dev, double *half_var_dev, void *stream)
{
    if (!samples_dev || !half_mean_dev || !half_var_dev || n_samples < 4 || d < 1 || n_chains < 1) {
        yg_set_error("yg_split_moments: invalid arguments");
        return YG_ERR_INVALID;
    }
    const int64_t total = (int64_t)d * n_chains;
    const int grid = (int)std::min<int64_t>((total + 127) / 128, 148 * 16);
    split_moments_kernel<<<grid, 128, 0, (cudaStream_t)stream>>>(samples_dev, n_samples, d, n_chains, half_mean_dev,
                                                                 half_var_dev);
    YG_CUDA_CHECK(cudaGetLastError());
    return YG_OK;
}

extern "C" int64_t yg_pooled_len(int32_t d) { return 3 + (int64_t)d + 2 * (int64_t)d * d + d; }

int yg_pooled_impl(const double *w_mean, const double *w_m2, const unsigned long long *n_accept, int d, int64_t nc,
                   int64_t welford_n, double *partials, int n_part, double *out_dev, cudaStream_t st)
{
    const int len = (int)yg_pooled_len(d);
    const size_t smem = sizeof(double) * (POOL_THREADS / 32) * len;
    pooled_stage1<<<n_part, POOL_THREADS, smem, st>>>(w_mean, w_m2, n_accept, d, nc, (double)welford_n, partials, len);
    YG_CUDA_CHECK(cudaGetLastError());
    pooled_stage2<<<1, 128, 0, st>>>(partials, n_part, len, out_dev);
    YG_CUDA_CHECK(cudaGetLastError());
    return YG_OK;
}

extern "C" int64_t yg_pooled_samples_workspace_len(int32_t d, int64_t n_chains)
{
    if (d < 1 || n_chains < 1) return 0;
    return ps_parts_max(n_chains) * yg_pooled_len(d) + (int64_t)d * n_chains;
}

extern "C" int yg_pooled_samples(const double *samples_dev, int64_t n_samples, int32_t d, int64_t n_chains,
                                 double *workspace_dev, int64_t workspace_len, double *out_dev, void *stream)
{
    if (!samples_dev || !workspace_dev || !out_dev || n_samples < 1 || n_chains < 1 || d < 1) {
        yg_set_error("yg_pooled_samples: invalid arguments");
        return YG_ERR_INVALID;
    }
    if (d > YG_BIG_MAX_DIM) {
        yg_set_error("yg_pooled_samples: dim %d exceeds %d", d, YG_BIG_MAX_DIM);
        return YG_ERR_UNSUPPORTED;
    }
    if (workspace_len < yg_pooled_samples_workspace_len(d, n_chains)) {
        yg_set_error("yg_pooled_samples: workspace of %lld doubles, %lld needed", (long long)workspace_len,
                     (long long)yg_pooled_samples_workspace_len(d, n_chains));
        return YG_ERR_INVALID;
    }
    cudaStream_t st = (cudaStream_t)stream;
    switch ((d + 7) / 8) {
    case 1: return launch_pooled_samples<1>(samples_dev, n_samples, d, n_chains, workspace_dev, out_dev, st);
    case 2: return launch_pooled_samples<2>(samples_dev, n_samples, d, n_chains, workspace_dev, out_dev, st);
    case 3: return launch_pooled_samples<3>(samples_dev, n_samples, d, n_chains, workspace_dev, out_dev, st);
    case 4: return launch_pooled_samples<4>(samples_dev, n_samples, d, n_chains, workspace_dev, out_dev, st);
    case 5: return launch_pooled_samples<5>(samples_dev, n_samples, d, n_chains, workspace_dev, out_dev, st);
    case 6: return launch_pooled_samples<6>(samples_dev, n_samples, d, n_chains, workspace_dev, out_dev, st);
    case 7: return launch_pooled_samples<7>(samples_dev, n_samples, d, n_chains, workspace_dev, out_dev, st);
    default: return launch_pooled_samples<8>(samples_dev, n_samples, d, n_chains, workspace_dev, out_dev, st);
    }
}

extern "C" int yg_fp64_peak(int32_t device, double ms, double *tflops_out)
{
    if (!tflops_out) return YG_ERR_INVALID;
    YG_CUDA_CHECK(cudaSetDevice(device));
    int sms = 0;
    YG_CUDA_CHECK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device));
    double *sink = nullptr;
    YG_CUDA_CHECK(cudaMalloc(&sink, 8));
    cudaEvent_t e0, e1;
    YG_CUDA_CHECK(cudaEventCreate(&e0));
    YG_CUDA_CHECK(cudaEventCreate(&e1));
    const int grid = sms * 4, threads = 256;
    double best = 0.0;
    for (int variant = 0; variant < 2; variant++) {
        // FP64-pipe instructions per thread per iteration: 64 DFMA, or 4 x 30 of the two-source mix
        const double per_iter = variant == 0 ? 64.0 : 120.0;
        int iters = 2048;
        float t = 0.f;
        // calibrate the iteration count to about `ms` per launch, then take the best of 5
        for (int rep = 0; rep < 7; rep++) {
            YG_CUDA_CHECK(cudaEventRecord(e0));
            if (variant == 0) dfma_peak_kernel<<<grid, threads>>>(sink, iters, 0.999999, 1e-9);
            else mix_peak_kernel<<<grid, threads>>>(sink, iters, 0.4 * 10 / 512, 0.6 * 10 / 512, 0.8 * 10 / 512, 0.4 * 10 / 512);
            YG_CUDA_CHECK(cudaEventRecord(e1));
            YG_CUDA_CHECK(cudaEventSynchronize(e1));
            YG_CUDA_CHECK(cudaEventElapsedTime(&t, e0, e1));
            const double flops = 2.0 * per_iter * (double)iters * (double)grid * threads;
            if (rep >= 2) best = std::max(best, flops / (t * 1e-3) / 1e12);
            if (rep < 2 && t > 0.f) iters = (int)std::max(256.0, std::min(4.0e6, iters * (ms > 0 ? ms : 20.0) / t));
        }
    }
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    cudaFree(sink);
    *tflops_out = best;
    return YG_OK;
}

extern "C" int yg_rk4_loop_rate(int32_t device, double ms, double *steps_per_s_out)
{
    if (!steps_per_s_out) return YG_ERR_INVALID;
    YG_CUDA_CHECK(cudaSetDevice(device));
    int sms = 0;
    YG_CUDA_CHECK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device));
    double *sink = nullptr;
    YG_CUDA_CHECK(cudaMalloc(&sink, 8));
    cudaEvent_t e0, e1;
    YG_CUDA_CHECK(cudaEventCreate(&e0));
    YG_CUDA_CHECK(cudaEventCreate(&e1));
    const double h = 10.0 / 512;
    const LvStepConsts kc = lv_step_consts(0.8, 0.4, h);
    int n_steps = 4096;
    double best = 0.0;
    float t = 0.f;
    for (int rep = 0; rep < 7; rep++) {
        YG_CUDA_CHECK(cudaEventRecord(e0));
        rk4_loop_kernel<<<sms, 1024>>>(sink, n_steps, h, kc);
        YG_CUDA_CHECK(cudaEventRecord(e1));
        YG_CUDA_CHECK(cudaEventSynchronize(e1));
        YG_CUDA_CHECK(cudaEventElapsedTime(&t, e0, e1));
        if (rep >= 2) best = std::max(best, (double)n_steps * sms * 1024.0 / (t * 1e-3));
        if (rep < 2 && t > 0.f)
            n_steps = 8 * (int)std::max(64.0, std::min(4.0e6, n_steps / 8 * (ms > 0 ? ms : 20.0) / t));
    }
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    cudaFree(sink);
    *steps_per_s_out = best;
    return YG_OK;
}
