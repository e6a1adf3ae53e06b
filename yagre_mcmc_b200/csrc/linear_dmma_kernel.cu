// linear_dmma_kernel.cu -- Metropolis-Hastings over an ensemble of chains on the LINEAR model
// F = G theta + b when the parameter / data dimensions are too large for one chain per thread
// (d up to 64, data_dim up to 256): the forward model of a tile of chains is a dense FP64 GEMM
// [data_dim x d] . [d x chains], issued on the FP64 tensor path (DMMA, mma.sync m16n8k4.f64),
// with the Gaussian-misfit log-likelihood fused into the accumulator epilogue.
//
// Reference semantics restated (rkutri/yagre-mcmc):
//   linear forward       exampleSetup.py:42-52 (A @ theta + b, broadcast against the data rows)
//   likelihood / prior   statistics/likelihood.py:33-39,74-84, statistics/gaussian.py:19-24,
//                        statistics/covariance.py:19-22,54-55 (diagonal precisions)
//   proposal             statistics/gaussian.py:61-66 with a diagonal factor (covariance.py:51-52);
//                        pCN: chain/method/pcn.py:23-35
//   MRW / MLDA ratios    chain/method/mrw.py:51-57, chain/method/mlda.py:100-110,146-154
//   step loop            chain/metropolisHastings.py:55-120
//   Welford diagnostics  chain/diagnostics.py:91-94, statistics/estimation.py:36-53 (diagonal M2)
//
// B200 mapping (measured facts: tools/probe_dmma.cu, profiles/r02_linear_dmma.md)
//   * On B200 DMMA executes on the FP64 units themselves: DMMA.8x8x4 occupies a sub-partition's FP64 pipe for 16
//     cycles, FP64 vector instructions queue behind it (a DFMA + DMMA mix takes the SUM of the two times), and a
//     DMMA that depends on the previous one issues only every 26 cycles.  The roofline of this kernel is therefore
//     the FP64 pipe shared by the GEMM and every DADD / DMUL / DFMA around it, and one warp alone must be able to
//     keep the pipe full.
//   * "swap-AB" GEMM on m16n8k4: G is the A operand (16 data rows x 4 parameters per instruction, two 8-byte
//     shared-memory loads), the 8 chains of the warp are the N extent.  ptxas schedules the accumulator chains of a
//     pass one after the other whatever the source order; an m16n8k4 is two DMMA.8x8x4 on separate accumulator
//     halves, so even a single dependent chain issues at the full rate (32.5 cycles per m16n8k4, measured), where
//     the m8n8k4 formulation of round 1 ran at 16 / 26 of it unless two warps happened to overlap.
//   * a warp owns a tile of 8 chains; proposals live in registers in the B-fragment layout -- lane (g = lane / 4,
//     t = lane % 4) holds p[chain g][k = 4 i + t] -- so a proposal IS the GEMM operand; the current state of the
//     tile sits in a per-warp shared-memory tile in the same lane-private pattern;
//   * G of every level is staged once per CTA into shared memory (row stride = 4 mod 16 doubles: the A-fragment
//     loads of a warp are bank-conflict free), pre-multiplied by sqrt(n_data x noise precision) on the host, as is
//     b - mean(data): the epilogue per accumulator element is one DADD and one DFMA (every FP64 vector instruction
//     costs GEMM time);
//   * the accumulators hold F[row][chain]: a lane sums the squares of its rows for chains 2t and 2t + 1, a
//     butterfly over the row lanes finishes the sums and one shuffle hands every lane the value of ITS chain, so
//     the four lanes of a chain hold bit-identical log-posteriors and take the same accept decision;
//   * balanced schedule: the (tile, step) pairs of a launch are cut into equal contiguous ranges, one per warp of
//     the persistent grid.  A warp first runs the HEAD of the tile its range ends in, then its whole tiles, then
//     the TAIL of the tile its range starts in -- whose head the previous warp ran first -- with the chain state
//     handed over through global memory and a per-tile progress counter.  No warp idles while another still has
//     tiles (with whole tiles per warp 65,536 chains on 148 x 16 warps wasted 13.5 % of the launch);
//   * Philox noise is keyed like the one-chain-per-thread kernels (seed, global chain id, step, sub-step, pair); the
//     Box-Muller transform of this kernel runs in FP32 (see philox_normal_pair_f32): d normals per chain-step on
//     the FP64 pipe would cost as much as a fifth of the GEMM.
#include "ensemble.h"
#include "big_linear.h"
#include "smem_plan.h"
#include <math_constants.h>

namespace {

YG_DEVFN void dmma_m16n8k4(double &c0, double &c1, double &c2, double &c3, double a0, double a1, double b0)
{
    asm volatile(
        "mma.sync.aligned.m16n8k4.row.col.f64.f64.f64.f64 {%0,%1,%2,%3}, {%4,%5}, {%6}, {%0,%1,%2,%3};"
        : "+d"(c0), "+d"(c1), "+d"(c2), "+d"(c3)
        : "d"(a0), "d"(a1), "d"(b0));
}

// Box-Muller on one Philox block with the TRANSFORM in FP32 (the FP32 / SFU pipes are idle next to the GEMM, the
// FP64 pipe is not).  Same uniforms as the oracle's yo_philox_normals: u1 = m1 2^-53 in (0, 1] and u2 = k2 2^-53 in
// [0, 1) from the 53 high bits of the two word pairs; z = sqrt(-2 ln u1) (cos, sin)(2 pi u2).
//   * BRANCH-FREE on purpose (no logf / sqrtf / sincospif: their slow paths are branches): the transform is inlined
//     into the GEMM loop of the preceding evaluation and must share a basic block with the DMMAs for the scheduler
//     to interleave the two instruction streams;
//   * -ln u1 keeps its RELATIVE accuracy over the whole range: u1 = m 2^e with m in [0.75, 1.5), ln m = 2 atanh(s),
//     s = (m - 1) / (m + 1), and for u1 >= 0.75 the numerator m - 1 = -(1 - u1) is formed exactly in integers,
//     (2^53 - m1) 2^-53 (a float of u1 itself would round to 1 for u1 > 1 - 2^-25 and give a zero radius, i.e. a
//     spurious "proposal == state"); the radius is zero only for u1 = 1, probability 2^-53, like the FP64 transform;
//   * the top bit of k2 is the SIGN of (cos, sin) -- (cos, sin)(x + pi) = -(cos, sin)(x) -- and the other 52 bits the
//     angle in [0, pi): P(z) = P(-z) holds exactly, not up to the float grid of the angle.
// The normals equal the oracle's FP64 ones to |dz| <= 6e-6 (1 + |z|) (tests/test_round2_gpu.py: MUFU sine / cosine
// have an absolute error of 2^-21.4); a recorded stream replays bit-exactly.
YG_DEVFN float neg_log_u53(const uint64_t m1)        // -ln(m1 2^-53), m1 in [1, 2^53]
{
    const float t = (float)((1ull << 53) - m1) * 0x1.0p-53f;                   // 1 - u1, relative accuracy 2^-24
    const float x = (float)m1 * 0x1.0p-53f;                                    // u1 in [2^-53, 1]: a normal float
    const int bits = __float_as_int(x);
    int e = ((bits >> 23) & 0xff) - 127;
    float m = __int_as_float((bits & 0x007fffff) | 0x3f800000);                // [1, 2)
    const bool up = m >= 1.5f;
    m = up ? 0.5f * m : m;                                                     // [0.75, 1.5)
    e += up ? 1 : 0;
    const float dm = (e == 0) ? -t : m - 1.0f;                                 // m - 1 (exact for the float m)
    const float s = __fdividef(dm, 2.0f + dm), s2 = s * s;                     // |s| <= 1/5
    float P = fmaf(s2, 1.0f / 11.0f, 1.0f / 9.0f);
    P = fmaf(s2, P, 1.0f / 7.0f);
    P = fmaf(s2, P, 0.2f);
    P = fmaf(s2, P, 1.0f / 3.0f);
    P = fmaf(s2, P, 1.0f);
    return -fmaf((float)e, 0.693147180559945309f, 2.0f * s * P);
}

// The same transform cut into 13 micro-steps (10 Philox rounds, radius, angle, store) that logpost_tile spreads over
// the k-steps of one pass of its GEMM loop: ptxas keeps the order of the PTX it is given, so the interleaving has to
// be written out -- a block of noise code placed before the DMMAs of a pass is executed before them, not under them.
struct NoiseSlice {
    uint4 c;
    uint2 k;
    float R;
    float2 z;
    float2 *dst;
    bool on;
    YG_DEVFN void begin(uint64_t seed, uint64_t chain, uint64_t step, uint32_t sub, uint32_t b, float2 *dst_, bool on_)
    {
        k = make_uint2((uint32_t)seed, (uint32_t)(seed >> 32));
        c = make_uint4((uint32_t)chain, (uint32_t)step, (uint32_t)(step >> 32),
                       (uint32_t)(((chain >> 32) & 0xFFu) << 24) | (sub << 8) | b);       // philox_block's counter
        dst = dst_;
        on = on_;
    }
    YG_DEVFN void micro(const int u)
    {
        if (u < 10) {                                            // one Philox4x32 round (common.cuh:philox4x32_10)
            const uint32_t hi0 = __umulhi(0xD2511F53u, c.x), lo0 = 0xD2511F53u * c.x;
            const uint32_t hi1 = __umulhi(0xCD9E8D57u, c.z), lo1 = 0xCD9E8D57u * c.z;
            c = make_uint4(hi1 ^ c.y ^ k.x, lo1, hi0 ^ c.w ^ k.y, lo0);
            k.x += 0x9E3779B9u;
            k.y += 0xBB67AE85u;
        } else if (u == 10) {
            const uint64_t m1 = ((((uint64_t)c.x << 32) | c.y) >> 11) + 1ull;
            asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(R) : "f"(2.0f * neg_log_u53(m1)));
        } else if (u == 11) {
            const uint64_t k2 = (((uint64_t)c.z << 32) | c.w) >> 11;
            float sn, cs;
            __sincosf(3.14159265358979324f * ((float)(k2 & ((1ull << 52) - 1ull)) * 0x1.0p-52f), &sn, &cs);
            const float sg = (k2 >> 52) ? -R : R;
            z = make_float2(sg * cs, sg * sn);
        } else if (u == 12) {
            if (on) *dst = z;
        }
    }
    // k-step i of KQ: its share of the 13 micro-steps
    template <int KQ>
    YG_DEVFN void stage(const int i)
    {
#pragma unroll
        for (int u = 0; u < 13; u++)
            if (u >= (13 * i) / KQ && u < (13 * (i + 1)) / KQ) micro(u);
    }
    YG_DEVFN void all()
    {
#pragma unroll
        for (int u = 0; u < 13; u++) micro(u);
    }
};

// Shared-memory load of a GEMM operand that ptxas may not move across its neighbours.  Left to itself ptxas gathers the
// DMMAs of one accumulator into one dependent chain (whatever the order of the PTX), and a DMMA that waits for its
// predecessor issues every 26 cycles instead of every 16.  Volatile loads keep their program order, so the operands of
// k-step i + 1 of ALL accumulator chains are fetched before the DMMAs of k-step i: gathering a chain would mean
// keeping every other chain's operands alive in registers, and the scheduler keeps the interleaved order instead
// (SASS: DMMA R28 / R32 / R36 / R24 round robin; profiles/r02_linear_dmma.md).
YG_DEVFN double lds_ordered(const double *p)
{
    double v;
    asm volatile("ld.volatile.shared.f64 %0, [%1];" : "=d"(v) : "r"((uint32_t)__cvta_generic_to_shared(p)));
    return v;
}

YG_DEVFN double quad_sum(double v)
{
    v += __shfl_xor_sync(0xffffffffu, v, 1);
    v += __shfl_xor_sync(0xffffffffu, v, 2);
    return v;
}

struct SmemLevel {
    const double *G;        // [np][ks]  sqrt(w_row) G_row, w = n_data * noise precision
    const double *bd;       // [np]      sqrt(w_row) (b - mean over the data rows)   (likelihood.py:74-75 broadcasts F against the rows)
    const double *pmean;    // [kp]
    const double *pprec;    // [kp]   (zero beyond dim)
    double q_const;         // sum_col prec_col * sum_rows (d_row,col - mean_col)^2
    int np;                 // data_dim rounded up to a multiple of 16
};

// log-posterior of the chain (column g of the warp's d x 8 tile) whose parameters are spread over the quad:
// a[i] = theta[4 i + t].  Every lane of a quad returns the same value.
// side.begin(pass) is called at the start of every pass over 32 (or the last 16) data rows and side.stage(i) after
// k-step i of the pass: independent work written out between the DMMAs (the noise of the NEXT proposal; SideNone
// for the evaluations that have none to draw).
struct SideNone {
    YG_DEVFN void begin(int) {}
    YG_DEVFN void stage(int) {}
};

template <int KQ, typename SIDE>
YG_DEVFN double logpost_tile(const SmemLevel &L, const int ks, const double (&a)[KQ], const int g, const int t, SIDE &&side)
{
    // sum_rows ||F - d_row||^2_P = sum_col w_col (F_col - mean_col)^2 + q_const  (exact identity; no cancellation:
    // the row scatter is a precomputed constant).  Accumulator layout of m16n8k4 with G as the A operand:
    // c0, c1 = F[row nb + g][chains 2t, 2t + 1], c2, c3 = F[row nb + 8 + g][the same chains].
    double qa = 0.0, qb = 0.0;                 // partial sums of chains 2t and 2t + 1 over this lane's rows
    auto epilogue = [&](const int nb, const double c0, const double c1, const double c2, const double c3) {
        const double b0 = L.bd[nb + g], b1 = L.bd[nb + 8 + g];
        const double e0 = c0 + b0, e1 = c1 + b0, e2 = c2 + b1, e3 = c3 + b1;     // sqrt(w) (A @ theta + b - mean(data))
        qa = fma(e2, e2, fma(e0, e0, qa));
        qb = fma(e3, e3, fma(e1, e1, qb));
    };
    int nb = 0, pass = 0;
    for (; nb + 32 <= L.np; nb += 32) {        // two 16-row blocks per pass = four interleaved DMMA.8x8x4 chains
        double c[2][4] = {{0.0, 0.0, 0.0, 0.0}, {0.0, 0.0, 0.0, 0.0}};
        const double *Gb = L.G + (size_t)(nb + g) * ks + t;
        side.begin(pass++);
        double A[2][2], An[2][2];
#pragma unroll
        for (int m = 0; m < 2; m++) {
            A[m][0] = lds_ordered(Gb + (size_t)(16 * m) * ks);
            A[m][1] = lds_ordered(Gb + (size_t)(16 * m + 8) * ks);
        }
#pragma unroll
        for (int i = 0; i < KQ; i++) {
            if (i + 1 < KQ) {
#pragma unroll
                for (int m = 0; m < 2; m++) {
                    An[m][0] = lds_ordered(Gb + (size_t)(16 * m) * ks + 4 * (i + 1));
                    An[m][1] = lds_ordered(Gb + (size_t)(16 * m + 8) * ks + 4 * (i + 1));
                }
            }
#pragma unroll
            for (int m = 0; m < 2; m++) dmma_m16n8k4(c[m][0], c[m][1], c[m][2], c[m][3], A[m][0], A[m][1], a[i]);
#pragma unroll
            for (int m = 0; m < 2; m++) { A[m][0] = An[m][0]; A[m][1] = An[m][1]; }
            side.stage(i);
        }
#pragma unroll
        for (int m = 0; m < 2; m++) epilogue(nb + 16 * m, c[m][0], c[m][1], c[m][2], c[m][3]);
    }
    for (; nb < L.np; nb += 16) {              // last 16 rows: two chains
        double c0 = 0.0, c1 = 0.0, c2 = 0.0, c3 = 0.0;
        const double *Gb = L.G + (size_t)(nb + g) * ks + t;
        side.begin(pass++);
        double A0 = lds_ordered(Gb), A1 = lds_ordered(Gb + (size_t)8 * ks), B0 = 0.0, B1 = 0.0;
#pragma unroll
        for (int i = 0; i < KQ; i++) {
            if (i + 1 < KQ) {
                B0 = lds_ordered(Gb + 4 * (i + 1));
                B1 = lds_ordered(Gb + (size_t)8 * ks + 4 * (i + 1));
            }
            dmma_m16n8k4(c0, c1, c2, c3, A0, A1, a[i]);
            A0 = B0; A1 = B1;
            side.stage(i);
        }
        epilogue(nb, c0, c1, c2, c3);
    }
    // rows are spread over the 8 lanes that share t: butterfly over g, then every lane fetches the sum of ITS chain
    // (chain g sits in element g & 1 of the lanes with t = g >> 1)
#pragma unroll
    for (int o = 4; o < 32; o <<= 1) {
        qa += __shfl_xor_sync(0xffffffffu, qa, o);
        qb += __shfl_xor_sync(0xffffffffu, qb, o);
    }
    const int src = (g << 2) | (g >> 1);
    const double va = __shfl_sync(0xffffffffu, qa, src), vb = __shfl_sync(0xffffffffu, qb, src);
    const double q = (g & 1) ? vb : va;
    double pr = 0.0;
#pragma unroll
    for (int i = 0; i < KQ; i++) {
        const double x = a[i] - L.pmean[4 * i + t];
        pr = fma(L.pprec[4 * i + t] * x, x, pr);
    }
    return -0.5 * (q + L.q_const) + (-0.5 * quad_sum(pr));
}

// ---- streamed operands: A fragments read from the global copy of the blob (smem_plan.h: big_tensor_plan) -----------
// The blob is constant during a launch, so the non-coherent read-only path is legal.  A lane reads 8 bytes and the four
// t lanes of a row 32 contiguous bytes: whole sectors (every streamed operand starts on a 32-byte boundary of the tail).
// Volatile for the reason lds_ordered is: the loads keep their place in the DMMA stream.
YG_DEVFN double ldg_ordered(const double *p)
{
    double v;
    asm volatile("ld.global.nc.f64 %0, [%1];" : "=d"(v) : "l"(p));
    return v;
}

// k-steps of A fragments in flight ahead of the DMMA that consumes them, chosen from the sweep over 2, 4, 6 and 8 in
// profiles/streamed_operand.md (B200, 1,000 W): two-level 64 x 256 at 65,536 chains ran at 2.00, 2.04, 2.01 and
// 1.99e8 chain-steps/s.  At 4 the streamed two-level instances spill what the resident ones spill (72 B; 88 B in the
// general instance) and the single-level one nothing; ptxas -v: at 6 the single-level instance spills 104 B, at 8 the
// two-level ones 168 / 176 B.  YG_STREAM_DEPTH overrides it in the dev builds of that sweep.
#ifndef YG_STREAM_DEPTH
#define YG_STREAM_DEPTH 4
#endif
constexpr int STREAM_DEPTH = YG_STREAM_DEPTH;

// Where a streamed operand lives, for the bounds-checked build: every index is checked against the tail.
struct StreamTail {
    const double *tail;
    int len;
    YG_DEVFN const double *at(const double *p) const
    {
        YG_CHK(p - tail, len);
        return p;
    }
};

// logpost_tile with G in global memory.  Same DMMAs in the same order on the same operands; the fragments of k-step
// i + STREAM_DEPTH are requested before the DMMAs of k-step i, across the boundary of 32-row passes too.  A row block
// that does not exist (after the last pass, or the second half of a trailing 16-row block) re-reads rows of the current
// pass instead (addresses stay inside G, no branch splits the DMMA stream).
template <int KQ, typename SIDE>
YG_DEVFN double logpost_tile_streamed(const SmemLevel &L, const int ks, const double (&a)[KQ], const int g, const int t,
                                      SIDE &&side, const StreamTail &st)
{
    constexpr int D = STREAM_DEPTH < KQ ? STREAM_DEPTH : KQ - 1;       // (KQ = 16, and 8 for three levels)
    double qa = 0.0, qb = 0.0;
    auto epilogue = [&](const int nb, const double c0, const double c1, const double c2, const double c3) {
        const double b0 = L.bd[nb + g], b1 = L.bd[nb + 8 + g];
        const double e0 = c0 + b0, e1 = c1 + b0, e2 = c2 + b1, e3 = c3 + b1;
        qa = fma(e2, e2, fma(e0, e0, qa));
        qb = fma(e3, e3, fma(e1, e1, qb));
    };
    // k-step i of the row block at nb: rows nb + g, nb + 8 + g, nb + h2 + g, nb + h2 + 8 + g (h2 = 16 for 32 rows)
    auto fetch = [&](const int nb, const int h2, const int i, double (&f)[4]) {
        const double *Gb = L.G + (size_t)(nb + g) * ks + t + 4 * i;
        f[0] = ldg_ordered(st.at(Gb));
        f[1] = ldg_ordered(st.at(Gb + (size_t)8 * ks));
        f[2] = ldg_ordered(st.at(Gb + (size_t)h2 * ks));
        f[3] = ldg_ordered(st.at(Gb + (size_t)(h2 + 8) * ks));
    };
    double F[D][4];                            // F[0]: the fragments of the k-step the DMMAs consume next
#pragma unroll
    for (int j = 0; j < D; j++) fetch(0, L.np >= 32 ? 16 : 0, j, F[j]);
    int nb = 0, pass = 0;
    for (; nb + 32 <= L.np; nb += 32) {
        double c[2][4] = {{0.0, 0.0, 0.0, 0.0}, {0.0, 0.0, 0.0, 0.0}};
        const int nn = nb + 32 < L.np ? nb + 32 : nb, hn = nn + 32 <= L.np ? 16 : 0;       // the next row block
        side.begin(pass++);
#pragma unroll
        for (int i = 0; i < KQ; i++) {
            double N[4];
            if (i + D < KQ) fetch(nb, 16, i + D, N);
            else fetch(nn, hn, i + D - KQ, N);
#pragma unroll
            for (int m = 0; m < 2; m++) dmma_m16n8k4(c[m][0], c[m][1], c[m][2], c[m][3], F[0][2 * m], F[0][2 * m + 1], a[i]);
#pragma unroll
            for (int j = 0; j < D; j++)
#pragma unroll
                for (int r = 0; r < 4; r++) F[j][r] = j + 1 < D ? F[j + 1][r] : N[r];
            side.stage(i);
        }
#pragma unroll
        for (int m = 0; m < 2; m++) epilogue(nb + 16 * m, c[m][0], c[m][1], c[m][2], c[m][3]);
    }
    for (; nb < L.np; nb += 16) {              // last 16 rows: its first D k-steps are already in F
        double c0 = 0.0, c1 = 0.0, c2 = 0.0, c3 = 0.0;
        side.begin(pass++);
#pragma unroll
        for (int i = 0; i < KQ; i++) {
            double N[4] = {0.0, 0.0, 0.0, 0.0};
            if (i + D < KQ) fetch(nb, 0, i + D, N);
            dmma_m16n8k4(c0, c1, c2, c3, F[0][0], F[0][1], a[i]);
#pragma unroll
            for (int j = 0; j < D; j++)
#pragma unroll
                for (int r = 0; r < 4; r++) F[j][r] = j + 1 < D ? F[j + 1][r] : N[r];
            side.stage(i);
        }
        epilogue(nb, c0, c1, c2, c3);
    }
#pragma unroll
    for (int o = 4; o < 32; o <<= 1) {
        qa += __shfl_xor_sync(0xffffffffu, qa, o);
        qb += __shfl_xor_sync(0xffffffffu, qb, o);
    }
    const int src = (g << 2) | (g >> 1);
    const double va = __shfl_sync(0xffffffffu, qa, src), vb = __shfl_sync(0xffffffffu, qb, src);
    const double q = (g & 1) ? vb : va;
    double pr = 0.0;
#pragma unroll
    for (int i = 0; i < KQ; i++) {
        const double x = a[i] - L.pmean[4 * i + t];
        pr = fma(L.pprec[4 * i + t] * x, x, pr);
    }
    return -0.5 * (q + L.q_const) + (-0.5 * quad_sum(pr));
}

// L z of the 8 chains with the dense factor in global memory: the DMMAs of propose's loop in its order, the fragments
// STREAM_DEPTH k-steps ahead over the whole triangle; the accumulators go to the transpose tile as there.
template <int KQ>
YG_DEVFN void lz_streamed(const double *Ld, const int ks, const double (&zv)[KQ], const int g, const int t, double *scr,
                          const StreamTail &st)
{
    constexpr int D = STREAM_DEPTH;
    static_assert(D <= 8, "the next block of the triangle has at least 8 k-steps");
    // fragments of k-step i of 16-row block b; block b has the 4 (b + 1) k-steps i with 4 i <= 16 b + 15
    auto fetch = [&](const int b, const int i, double (&n)[2]) {
        const double *p = Ld + (size_t)(16 * b + g) * ks + t + 4 * i;
        n[0] = ldg_ordered(st.at(p));
        n[1] = ldg_ordered(st.at(p + (size_t)8 * ks));
    };
    double F[D][2];
#pragma unroll
    for (int j = 0; j < D; j++) fetch(j < 4 ? 0 : 1, j < 4 ? j : j - 4, F[j]);
#pragma unroll
    for (int b = 0; b < KQ / 4; b++) {
        double c0 = 0.0, c1 = 0.0, c2 = 0.0, c3 = 0.0;
#pragma unroll
        for (int i = 0; i <= 4 * b + 3; i++) {
            double N[2] = {0.0, 0.0};
            if (i + D <= 4 * b + 3) fetch(b, i + D, N);                         // k-step D ahead: this block
            else if (b + 1 < KQ / 4) fetch(b + 1, i + D - 4 * (b + 1), N);       // or the next one
            dmma_m16n8k4(c0, c1, c2, c3, F[0][0], F[0][1], zv[i]);
#pragma unroll
            for (int j = 0; j < D; j++) {
                F[j][0] = j + 1 < D ? F[j + 1][0] : N[0];
                F[j][1] = j + 1 < D ? F[j + 1][1] : N[1];
            }
        }
        const int nb = 16 * b;
        YG_CHK((2 * t + 1) * ks + nb + 8 + g, 8 * ks);
        scr[(2 * t) * ks + nb + g] = c0;
        scr[(2 * t + 1) * ks + nb + g] = c1;
        scr[(2 * t) * ks + nb + 8 + g] = c2;
        scr[(2 * t + 1) * ks + nb + 8 + g] = c3;
    }
}

// FREE_NOISE = true: the production instance (Philox noise, diagonal proposal factor).  The injected / recorded noise
// paths of the parity tests and the DENSE proposal factor (p = s + L z with L z as a second small GEMM) live in the
// FREE_NOISE = false instance, which keeps the step loop of the production one small enough for the instruction cache
// (stall reason no_instruction in profiles/r01_linear_dmma.md).
// NL: levels -- 1 (MRW / pCN), 2 (two-level delayed acceptance) or 3 (MLDA with two surrogates: the sub-chain on level
// 0, the screen on level 1 in place of level 0, generic_kernel.cuh's three-level step).
// STREAMED = true: the operands of H.stream (smem_plan.h: big_tensor_plan: the G of levels 1 and 2, the dense factor)
// are read from the global blob, and only the prefix of sp.blob bytes is staged.  Level 0's G -- J evaluations per
// transition, under which the next proposal's noise is drawn -- always stays in shared memory.  Instantiated at KQ = 16,
// and for three levels at KQ = 8: the widths whose blobs can outgrow shared memory.
template <int KQ, int NL, bool FREE_NOISE, bool STREAMED = false>
__global__ void __launch_bounds__(big_max_warps(KQ) * 32, 1) linear_dmma_mh_kernel(const RunArgs a, const DevBigHeader *gh,
                                                                          long long *tile_done, const BigSmemPlan sp)
{
    const int noise_mode = FREE_NOISE ? (int)YG_NOISE_PHILOX : a.noise_mode;
    extern __shared__ __align__(16) double smem[];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, g = lane >> 2, t = lane & 3, odd = t & 1;
    // ---- stage the problem into shared memory -------------------------------------------------
    const DevBigHeader H = *gh;
    const double *gtail = reinterpret_cast<const double *>(gh + 1);
    const int staged = STREAMED ? (int)(sp.blob / sizeof(double)) : H.tail_len;
    for (int i = tid; i < staged; i += blockDim.x) smem[i] = gtail[i];
    __syncthreads();
    const StreamTail stail{gtail, H.tail_len};
    constexpr bool TWO_LEVEL = NL >= 2;             // a sub-chain on level 0 and a screen above it
    constexpr int NLV = NL < 2 ? 2 : NL;
    auto g_bit = [](const int l) { return l == 1 ? BIG_STREAM_G1 : (l == 2 ? BIG_STREAM_G2 : 0); };
    SmemLevel Lv[NLV];
#pragma unroll
    for (int l = 0; l < NLV; l++) {
        Lv[l].G = ((STREAMED && (H.stream & g_bit(l))) ? gtail : smem) + H.lvl[l].G_off;
        Lv[l].bd = smem + H.lvl[l].bd_off;
        Lv[l].pmean = smem + H.lvl[l].pmean_off;
        Lv[l].pprec = smem + H.lvl[l].pprec_off;
        Lv[l].q_const = H.lvl[l].q_const;
        Lv[l].np = H.lvl[l].np;
    }
    const double *propL = smem + H.propL_off;      // [kp] diagonal proposal factor (zero beyond dim)
    const bool pcn = H.proposal == YG_PROPOSAL_PCN;
    const double *pcn_mean = smem + H.pcn_mean_off;
    // current state of the warp's 8 chains: [8][ks] doubles after the problem blob; lane (g, t) only ever
    // touches its own slots (row g, columns 4 i + t), so no synchronisation is needed, and the row stride
    // (4 mod 16 doubles) makes the accesses bank-conflict free
    const int d = H.dim, ks = H.ks, J = TWO_LEVEL ? H.J : 1, n_lvl = NL;
    constexpr int ZS = big_zs(KQ);
    const int n_warps = blockDim.x >> 5;
    const bool dense_L = !FREE_NOISE && H.dense_L;
    const bool ld_streamed = STREAMED && (H.stream & BIG_STREAM_LD);
    const double *Ld = (ld_streamed ? gtail : smem) + H.Ld_off;      // [kp][ks] lower-triangular factor (dense_L only)
    // the warp's tiles (smem_plan.h): state, transpose buffer of L z (dense_L only), Welford moments (wsm only), noise
    const int wsm = sp.wsm;
    unsigned char *wreg = reinterpret_cast<unsigned char *>(smem) + sp.blob + (size_t)warp * sp.stride;
    double *ths = reinterpret_cast<double *>(wreg);
    double *scr = reinterpret_cast<double *>(wreg + sp.scr);
    double *wmt = reinterpret_cast<double *>(wreg + sp.wm), *wvt = reinterpret_cast<double *>(wreg + sp.wv);
    float *zb = reinterpret_cast<float *>(wreg + sp.zb);
#ifdef YG_BOUNDS_CHECK
    // every per-warp tile is [8][ks] doubles; the warp's region must end inside the dynamic shared memory of the launch
    YG_CHK(sp.blob + (size_t)(warp + 1) * sp.stride - 1, yg_dynamic_smem_bytes());
    auto tile_at = [&](double *tile, const int i) -> double & {
        YG_CHK(g * ks + 4 * i + t, 8 * ks);
        return tile[g * ks + 4 * i + t];
    };
#define WM(i) tile_at(wmt, (i))
#define WV(i) tile_at(wvt, (i))
#define TH(i) tile_at(ths, (i))
#else
#define WM(i) wmt[g * ks + 4 * (i) + t]
#define WV(i) wvt[g * ks + 4 * (i) + t]
#define TH(i) ths[g * ks + 4 * (i) + t]
#endif
    const int64_t N = a.n_chains;
    unsigned long long cnt_acc = 0ull, cnt_ev0 = 0ull, cnt_ev1 = 0ull, cnt_tr = 0ull, cnt_cacc = 0ull;

    // ---- one piece of work: transitions [s0, s1) of the 8 chains of `tile` -------------------------------------
    auto run_piece = [&](const int64_t tile, const int64_t s0, const int64_t s1) {
        // this lane's chain (a row beyond n_chains is computed but never stored)
        const int64_t gr = tile * 8 + g;
        const bool live = gr < N;
        const int64_t gg = live ? gr : 0;
        const uint64_t gid = (uint64_t)(a.chain_offset + gg);
        YG_CHK(tile, (N + 7) / 8); YG_CHK(gg, N); YG_CHK(s0, s1); YG_CHK(s1 - 1, a.n_steps);
        if (s0 > 0) {      // the transitions before s0 belong to the warp that owns the preceding range: wait for its hand-over
            if (lane == 0) {
                while (*reinterpret_cast<volatile long long *>(tile_done + tile) != s0) __nanosleep(200);
            }
            __syncwarp();
            __threadfence();
        }
#pragma unroll 1
        for (int i = 0; i < KQ; i++) {
            const int k = 4 * i + t;
            TH(i) = (k < d) ? __ldcg(a.theta + (int64_t)k * N + gg) : 0.0;
        }
        double lp0 = __ldcg(a.logpost + gg), lp1 = TWO_LEVEL ? __ldcg(a.logpost + N + gg) : 0.0;
        double lp2 = NL == 3 ? __ldcg(a.logpost + 2 * N + gg) : 0.0;
        unsigned long long nacc = __ldcg(a.n_accept + gg);

        // Welford (estimation.py:36-53, diagonal M2) in run-length form: a chain that stays at x for m
        // consecutive steps contributes  n' = n + m, mean' = mean + (x - mean) m / n',
        // M2' = M2 + (x - mean)^2 n m / n'  -- algebraically the m sequential updates.  With the
        // accumulators in (L2-resident) global memory this touches them once per accepted move
        // instead of once per step; the registers stay with the GEMM operands.  Loads of a batch of
        // columns are issued before any store (a store may alias the next load for the compiler).
        // wsm: the moments of the tile are staged in shared memory for the piece (whenever the problem blob leaves room:
        // not at d = 64 with 256 data rows) -- the L2 round trip of the flush was 15 % of the warp time.
        double run = 0.0, wn = (double)(a.welford_n0 + s0);
        if (wsm && a.welford) {
#pragma unroll 1
            for (int i = 0; i < KQ; i++) {
                const int k = 4 * i + t;
                WM(i) = (live && k < d) ? __ldcg(a.w_mean + (int64_t)k * N + gr) : 0.0;
                WV(i) = (live && k < d) ? __ldcg(a.w_m2 + (int64_t)big_w2_index(k, d) * N + gr) : 0.0;
            }
        }
        auto welford_flush = [&](const bool f) {
            const bool fl = f && live && run != 0.0 && a.welford;
            if (!__any_sync(0xffffffffu, fl)) return;
            const double n1 = wn + run, c1 = run / n1, c2 = wn * c1;
            if (wsm) {
                if (fl) {
#pragma unroll 1
                    for (int i = 0; i < KQ; i++) {
                        const double m0 = WM(i), dl = TH(i) - m0;
                        WM(i) = fma(dl, c1, m0);
                        WV(i) = fma(dl * dl, c2, WV(i));
                    }
                    wn += run; run = 0.0;
                }
                return;
            }
            constexpr int B = KQ < 8 ? KQ : 8;
#pragma unroll 1
            for (int i0 = 0; i0 < KQ; i0 += B) {
                double m0[B], v0[B];
#pragma unroll
                for (int i = 0; i < B; i++) {
                    const int k = 4 * (i0 + i) + t;
                    const bool on = fl && k < d;
                    m0[i] = on ? __ldcg(a.w_mean + (int64_t)k * N + gr) : 0.0;
                    v0[i] = on ? __ldcg(a.w_m2 + (int64_t)big_w2_index(k, d) * N + gr) : 0.0;
                }
#pragma unroll
                for (int i = 0; i < B; i++) {
                    const int k = 4 * (i0 + i) + t;
                    if (fl && k < d) {
                        const double dl = TH(i0 + i) - m0[i];
                        a.w_mean[(int64_t)k * N + gr] = fma(dl, c1, m0[i]);
                        a.w_m2[(int64_t)big_w2_index(k, d) * N + gr] = fma(dl * dl, c2, v0[i]);
                    }
                }
            }
            if (fl) { wn += run; run = 0.0; }
        };

        // Noise of proposal (n, j): pair b of the sub-step gives z[2b], z[2b+1], keyed like the per-thread kernels.
        // Columns 4i+t and 4i+(t^1) of a lane pair are the two halves of pair b = (4i + (t & ~1)) / 2: the even lane
        // draws the pairs of even i, the odd lane those of odd i -- one Philox block + one Box-Muller per lane and 4
        // parameters -- and both halves go to the warp's noise tile, from where every lane later picks its columns.
        // Slice `it` (of KQ / 2) is one pair per lane; the slices are drawn INSIDE the GEMM loop of the evaluation that
        // precedes the proposal (the noise does not depend on the chain state: counter-based Philox).
        NoiseSlice ns;
        auto slice_begin = [&](const int64_t n, const int j, const int it, const bool on) {
            // a slice index beyond KQ / 2 (more passes than slices) redraws an earlier slice: same values, same place
            const int i_mine = 2 * (it & (KQ / 2 - 1)) + odd;
            YG_CHK(g * ZS + 4 * i_mine + (t & ~1) + 1, 8 * ZS);
            ns.begin(a.seed, gid, (uint64_t)(a.step0 + n), (uint32_t)j, (uint32_t)((4 * i_mine + (t & ~1)) >> 1),
                     reinterpret_cast<float2 *>(zb + g * ZS + 4 * i_mine + (t & ~1)), on && noise_mode != YG_NOISE_INJECT);
        };
        auto gen_noise = [&](const int64_t n, const int j, const int it) {       // one slice, not interleaved with anything
            slice_begin(n, j, it, true);
            ns.all();
        };
        struct SideNoise {
            decltype(slice_begin) &sb;
            NoiseSlice &ns;
            int64_t n;
            int j;
            bool on;
            YG_DEVFN void begin(const int pass) { sb(n, j, pass, on); }
            YG_DEVFN void stage(const int i) { ns.template stage<KQ>(i); }
        };
        // the proposal after (n, j) in the order the chain consumes them; n == s1 means "none in this piece"
        auto next_of = [&](int64_t &n, int &j) {
            if (++j == J) { j = 0; n++; }
        };
        // p = s + L z with a diagonal L, unfused like numpy.  pCN (pcn.py:30-35): p = sqrt(1 - 2h) s + sqrt(2h) (m + L z).
        auto propose = [&](auto &&src, int64_t n, int j, double (&p)[KQ]) {
            bool same = true;
            __syncwarp();                                  // the noise tile was written by other lanes
            double zv[KQ];
#pragma unroll
            for (int i = 0; i < KQ; i++) {
                const int k = 4 * i + t;
                zv[i] = 0.0;
                if (noise_mode != YG_NOISE_PHILOX && k < d) YG_CHK(((n * J + j) * d + k) * N + gg, a.n_steps * J * d * N);
                if (noise_mode == YG_NOISE_INJECT) {
                    if (k < d) zv[i] = a.z[((n * J + j) * d + k) * N + gg];
                } else if (k < d) {
                    YG_CHK(g * ZS + k, 8 * ZS);
                    zv[i] = (double)zb[g * ZS + k];
                    if (noise_mode == YG_NOISE_RECORD && live) a.z[((n * J + j) * d + k) * N + gr] = zv[i];
                }
            }
            if (dense_L && ld_streamed) {
                lz_streamed<KQ>(Ld, ks, zv, g, t, scr, stail);
                __syncwarp();
            } else if (dense_L) {
                // L z of the 8 chains as a GEMM: L is the A operand (16 rows x 4 columns per mma), z -- already in the
                // B-fragment layout -- the other one; only the k-steps of the lower triangle are issued.  The accumulators
                // hold (L z)[row][chain]; the scratch tile transposes them back to "lane (g, t) holds chain g, row 4i + t".
                for (int nb = 0; nb < H.kp; nb += 16) {
                    double c0 = 0.0, c1 = 0.0, c2 = 0.0, c3 = 0.0;
                    const double *Lb = Ld + (size_t)(nb + g) * ks + t;
#pragma unroll
                    for (int i = 0; i < KQ; i++)
                        if (4 * i <= nb + 15) dmma_m16n8k4(c0, c1, c2, c3, Lb[4 * i], Lb[(size_t)8 * ks + 4 * i], zv[i]);
                    YG_CHK((2 * t + 1) * ks + nb + 8 + g, 8 * ks);
                    scr[(2 * t) * ks + nb + g] = c0;
                    scr[(2 * t + 1) * ks + nb + g] = c1;
                    scr[(2 * t) * ks + nb + 8 + g] = c2;
                    scr[(2 * t + 1) * ks + nb + 8 + g] = c3;
                }
                __syncwarp();
            }
#pragma unroll
            for (int i = 0; i < KQ; i++) {
                const int k = 4 * i + t;
                const double sv = src(i);
                const double lz = dense_L ? scr[g * ks + k] : __dmul_rn(propL[k], zv[i]);
                p[i] = pcn ? __dadd_rn(__dmul_rn(H.pcn_a, sv), __dmul_rn(H.pcn_b, __dadd_rn(pcn_mean[k], lz))) : __dadd_rn(sv, lz);
                same = same && (p[i] == sv);
            }
            __syncwarp();                                  // every lane has read its columns: the tiles may be refilled
            // parameter/vector.py:37-45: equal iff every coordinate is equal (all four lanes agree)
            const unsigned m = __ballot_sync(0xffffffffu, same);
            return ((m >> (4 * g)) & 0xFu) == 0xFu;
        };
        // log-posterior of proposal (n, j) on level 0 while the noise of the following proposal is drawn
        auto eval_and_draw = [&](const double (&p)[KQ], int64_t n, int j) {
            next_of(n, j);
            const bool more = n < s1;
            if (!more) n = s1 - 1;                                                 // a valid counter; nothing is stored
            const double lp = logpost_tile<KQ>(Lv[0], ks, p, g, t, SideNoise{slice_begin, ns, n, j, more});
            const int passes = (Lv[0].np + 31) >> 5;
            if (more)
                for (int it = passes; it < KQ / 2; it++) gen_noise(n, j, it);       // few data rows: the rest of the slices
            return lp;
        };
        for (int it = 0; it < KQ / 2; it++) gen_noise(s0, 0, it);                 // the first proposal of the piece

        int64_t thin_left = a.thin - (s0 % a.thin), thin_out = s0 / a.thin - 1;      // once per piece, not per step
        for (int64_t n = s0; n < s1; n++) {
            const uint64_t step = (uint64_t)(a.step0 + n);
            const bool store_now = (--thin_left == 0);     // (n + 1) % thin == 0 without a 64-bit division per step
            if (store_now) { thin_left = a.thin; thin_out++; }
            // FullDiagnostics: Welford of the pre-transition state (diagnostics.py:91-94): the state of
            // this step is seen once more; the accumulators are touched when the state changes.
            run += 1.0;
            bool accepted = false;
            if (!TWO_LEVEL) {
                double p[KQ];
                const bool eq = propose([&](int i) { return TH(i); }, n, 0, p);
                const double lpp = eval_and_draw(p, n, 0);
                if (!eq) {                                              // metropolisHastings.py:60-61
                    if (t == 0 && live) cnt_ev0++;
                    double u;
                    if (noise_mode == YG_NOISE_INJECT) u = a.u_f[n * N + gg];
                    else {
                        u = philox_uniform(a.seed, gid, step, YG_SUB_FINE);
                        if (noise_mode == YG_NOISE_RECORD && live && t == 0) a.u_f[n * N + gg] = u;
                    }
                    accepted = accept_rule(lpp - lp0, u);
                }
                welford_flush(accepted);
                if (accepted) {
#pragma unroll
                    for (int i = 0; i < KQ; i++) TH(i) = p[i];
                    lp0 = lpp;
                }
            } else {
                double s[KQ], p[KQ], lps = lp0;
#pragma unroll
                for (int i = 0; i < KQ; i++) s[i] = TH(i);
                for (int j = 0; j < J; j++) {                           // coarse sub-chain, mlda.py:100-110
                    const bool eq = propose([&](int i) { return s[i]; }, n, j, p);
                    const double lpp = eval_and_draw(p, n, j);
                    if (eq) continue;
                    if (t == 0 && live) cnt_ev0++;
                    const int64_t ui = (n * J + j) * N + gg;
                    double u;
                    if (noise_mode == YG_NOISE_INJECT) u = a.u_c[ui];
                    else {
                        u = philox_uniform(a.seed, gid, step, (uint32_t)j);
                        if (noise_mode == YG_NOISE_RECORD && live && t == 0) a.u_c[ui] = u;
                    }
                    if (accept_rule(lpp - lps, u)) {
#pragma unroll
                        for (int i = 0; i < KQ; i++) s[i] = p[i];
                        lps = lpp;
                        if (t == 0 && live) cnt_cacc++;
                    }
                }
                // the sub-chain's end point is the proposal; no fine evaluation for a chain that did
                // not move (metropolisHastings.py:60-61).  The GEMM is warp wide: it runs when ANY of
                // the 8 chains moved, and only the chains that moved use (and count) its result.
                bool same = true;
#pragma unroll
                for (int i = 0; i < KQ; i++) same = same && (s[i] == TH(i));
                const unsigned m = __ballot_sync(0xffffffffu, same);
                const bool moved = (((m >> (4 * g)) & 0xFu) != 0xFu) && live;
                double lpf = 0.0, lpm = 0.0;
                if (__any_sync(0xffffffffu, moved)) {
                    if constexpr (NL == 3) {
                        // the finest surrogate, then the target, from ONE call site (two inlined evaluations spill)
#pragma unroll 1
                        for (int l = 1; l < 3; l++) {
                            const SmemLevel &L = l == 1 ? Lv[1] : Lv[2];
                            const double v = (STREAMED && (H.stream & g_bit(l)))
                                                 ? logpost_tile_streamed<KQ>(L, ks, s, g, t, SideNone{}, stail)
                                                 : logpost_tile<KQ>(L, ks, s, g, t, SideNone{});
                            if (l == 1) lpm = v; else lpf = v;
                        }
                    } else {
                        lpf = (STREAMED && (H.stream & BIG_STREAM_G1)) ? logpost_tile_streamed<KQ>(Lv[1], ks, s, g, t, SideNone{}, stail)
                                                                        : logpost_tile<KQ>(Lv[1], ks, s, g, t, SideNone{});
                    }
                    if (moved) {
                        if (t == 0) cnt_ev1++;
                        double u;
                        if (noise_mode == YG_NOISE_INJECT) u = a.u_f[n * N + gg];
                        else {
                            u = philox_uniform(a.seed, gid, step, YG_SUB_FINE);
                            if (noise_mode == YG_NOISE_RECORD && t == 0) a.u_f[n * N + gg] = u;
                        }
                        // mlda.py:148-152, this order; with two surrogates the screen's coarse density is the FINEST
                        // surrogate although the sub-chain ran on level 0 (mlda.py:130,146-154)
                        const double delta = NL == 3 ? lpf + lp1 - lpm - lp2 : lpf + lp0 - lps - lp1;
                        accepted = accept_rule(delta, u);
                    }
                }
                welford_flush(accepted);
                if (accepted) {
#pragma unroll
                    for (int i = 0; i < KQ; i++) TH(i) = s[i];
                    lp0 = lps;
                    if (NL == 3) { lp1 = lpm; lp2 = lpf; } else lp1 = lpf;
                }
            }
            if (live) {
                if (accepted) { nacc++; if (t == 0) cnt_acc++; }
                if (t == 0) {
                    cnt_tr++;
                    if (a.accepted) a.accepted[n * N + gr] = accepted ? 1 : 0;
                }
                if (store_now) {
                    const int64_t o = thin_out;
                    YG_CHK(o, a.n_steps / a.thin);
                    if (a.samples) {
#pragma unroll 1
                        for (int i = 0; i < KQ; i++)
                            if (4 * i + t < d) a.samples[(o * d + 4 * i + t) * N + gr] = TH(i);
                    }
                    if (a.lp_out && t == 0) {
                        a.lp_out[(o * n_lvl) * N + gr] = lp0;
                        if (TWO_LEVEL) a.lp_out[(o * n_lvl + 1) * N + gr] = lp1;
                        if (NL == 3) a.lp_out[(o * n_lvl + 2) * N + gr] = lp2;
                    }
                }
            }
        }
        // ---- store chain state ------------------------------------------------------------------
        welford_flush(true);
        if (live) {
#pragma unroll 1
            for (int i = 0; i < KQ; i++) {
                const int k = 4 * i + t;
                if (k < d) a.theta[(int64_t)k * N + gr] = TH(i);
                if (wsm && a.welford && k < d) {
                    a.w_mean[(int64_t)k * N + gr] = WM(i);
                    a.w_m2[(int64_t)big_w2_index(k, d) * N + gr] = WV(i);
                }
            }
            if (t == 0) {
                a.logpost[gr] = lp0;
                if (TWO_LEVEL) a.logpost[N + gr] = lp1;
                if (NL == 3) a.logpost[2 * N + gr] = lp2;
                a.n_accept[gr] = nacc;
            }
        }
        if (s1 < a.n_steps) {       // hand the tile over to the warp that owns the following range
            __threadfence();
            __syncwarp();
            if (lane == 0) *reinterpret_cast<volatile long long *>(tile_done + tile) = s1;
        }
    };

    // ---- balanced schedule: this warp's contiguous range of the (tile-major, step-minor) work list ------------------
    // A warp only ever waits for the warp with the next lower global index (same CTA or the CTA with the next lower
    // blockIdx), which never waits for a higher one: with CTAs dispatched in index order nothing can wait for a CTA that
    // is not resident yet, even if the grid shares the GPU with other work.
    const int64_t n_tiles = (N + 7) / 8, S = a.n_steps;
    const int64_t gw = (int64_t)blockIdx.x * n_warps + warp, GW = (int64_t)gridDim.x * n_warps;
    // ranges in units of transitions: [lo, hi); n_tiles * S < 2^63 / GW for every admissible size
    const int64_t U = n_tiles * S;
    const int64_t lo = (U / GW) * gw + ((U % GW) * gw) / GW, hi = (U / GW) * (gw + 1) + ((U % GW) * (gw + 1)) / GW;
    if (lo < hi) {
        const int64_t t_first = lo / S, s_first = lo - t_first * S;
        const int64_t t_last = (hi - 1) / S, s_end = hi - t_last * S;          // transitions [.., s_end) of the last tile
        // Pieces in the order they are run (ONE call site: the step loop must not be inlined several times, it would
        // no longer fit the instruction cache): the head of the last tile (it has no predecessor, so it can always
        // run), the whole tiles, and last the tail of the first tile -- it waits for the previous warp's head, which
        // that warp ran FIRST.  A range inside one tile is a single piece.
        const bool single = t_first == t_last;
        const int64_t has_head = (!single && s_end < S) ? 1 : 0, has_tail = (!single && s_first > 0) ? 1 : 0;
        const int64_t w_lo = t_first + has_tail, n_whole = single ? 0 : (t_last + (s_end == S ? 1 : 0)) - w_lo;
        const int64_t n_pieces = single ? 1 : has_head + n_whole + has_tail;
#pragma unroll 1
        for (int64_t q = 0; q < n_pieces; q++) {
            int64_t tile = w_lo + (q - has_head), s0 = 0, s1 = S;
            if (single) { tile = t_first; s0 = s_first; s1 = s_end; }
            else if (has_head && q == 0) { tile = t_last; s1 = s_end; }
            else if (q - has_head >= n_whole) { tile = t_first; s0 = s_first; }
            run_piece(tile, s0, s1);
        }
    }
#undef TH
#undef WM
#undef WV
    // ---- counters: warp-shuffle reduction, one atomic per warp ----------------------------------
    // slots (yg_get_counters): transitions, accepted, level-0 evaluations, target evaluations, level-1 evaluations of
    // three levels (the same chains evaluate both upper levels), coarse accepts
    unsigned long long v[6] = {cnt_tr, cnt_acc, cnt_ev0, cnt_ev1, cnt_ev1, cnt_cacc};
#pragma unroll
    for (int k = 0; k < 6; k++) {
        if (NL < 3 && k == 4) continue;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v[k] += __shfl_xor_sync(0xffffffffu, v[k], o);
        if (lane == 0 && v[k]) atomicAdd(&a.counters[k], v[k]);
    }
}

// log-posterior of arbitrary points, one chain per thread, plain loops over global memory
// (yg_set_state / yg_logpost: outside the step loop).
__global__ void big_logpost_kernel(const DevBigHeader *gh, int lvl, const double *theta, int64_t n, double *out)
{
    const DevBigHeader &H = *gh;
    const double *tail = reinterpret_cast<const double *>(gh + 1);
    const BigLevel &L = H.lvl[lvl];
    const double *G = tail + L.G_off, *bd = tail + L.bd_off;             // both carry sqrt(n_data * noise precision)
    const double *pm = tail + L.pmean_off, *pw = tail + L.pprec_off;
    for (int64_t c = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; c < n; c += (int64_t)gridDim.x * blockDim.x) {
        double s = 0.0;
        for (int col = 0; col < L.n_rows; col++) {
            double f = 0.0;
            for (int k = 0; k < H.dim; k++) f = fma(G[(size_t)col * H.ks + k], theta[(int64_t)k * n + c], f);
            const double e = f + bd[col];
            s = fma(e, e, s);
        }
        s += L.q_const;
        double p = 0.0;
        for (int k = 0; k < H.dim; k++) {
            const double x = theta[(int64_t)k * n + c] - pm[k];
            p = fma(pw[k] * x, x, p);
        }
        out[c] = -0.5 * s + (-0.5 * p);
    }
}

// FP64 tensor-path micro-benchmark: independent m16n8k4 accumulator chains, 8 warps per SM.
__global__ void __launch_bounds__(256, 1) dmma_peak_kernel(double *sink, int iters, double x)
{
    double c[8][4];
#pragma unroll
    for (int k = 0; k < 8; k++) c[k][0] = c[k][1] = c[k][2] = c[k][3] = 0.0;
    const double a0 = x + threadIdx.x * 1e-9, a1 = x - threadIdx.x * 1e-9, b0 = 1.0 + 1e-9 * threadIdx.x;
#pragma unroll 1
    for (int i = 0; i < iters; i++) {
#pragma unroll
        for (int k = 0; k < 8; k++) dmma_m16n8k4(c[k][0], c[k][1], c[k][2], c[k][3], a0, a1, b0);
    }
    double s = 0.0;
#pragma unroll
    for (int k = 0; k < 8; k++) s += c[k][0] + c[k][1] + c[k][2] + c[k][3];
    if (s == 123.456) sink[0] = s;
}

template <int KQ>
int launch_t(yg_ensemble *e, const RunArgs &a, cudaStream_t st)
{
    const DevBigHeader *hh = reinterpret_cast<const DevBigHeader *>(e->h_problem.data());
    // warps per CTA: as many as the shared memory left by the staged part of the problem blob holds (at most 12 for
    // d > 32, else 16; yg_set_problem streamed operands until BIG_MIN_WARPS fit); Welford moments of the tiles in shared
    // memory when that costs no warp (and FullDiagnostics asked for them at all)
    const int nl = e->cfg.n_levels;
    const BigTensorPlan tp = big_tensor_plan(hh->lvl[0].np, nl >= 2 ? hh->lvl[1].np : 0, KQ, hh->dense_L != 0,
                                             a.welford != 0, nl == 3 ? hh->lvl[2].np : 0);
    const BigSmemPlan sp = tp.smem;
    const bool free_noise = a.noise_mode == YG_NOISE_PHILOX && !hh->dense_L;      // the general instance also knows dense factors
    decltype(&linear_dmma_mh_kernel<KQ, 2, true>) kern;
    if (tp.stream) {
        // streamed instances: KQ = 16, and KQ = 8 for three levels; one level streams only the dense factor (general
        // instance)
        if constexpr (KQ == 16) {
            kern = nl == 3 ? (free_noise ? linear_dmma_mh_kernel<KQ, 3, true, true> : linear_dmma_mh_kernel<KQ, 3, false, true>)
                 : nl == 2 ? (free_noise ? linear_dmma_mh_kernel<KQ, 2, true, true> : linear_dmma_mh_kernel<KQ, 2, false, true>)
                           : linear_dmma_mh_kernel<KQ, 1, false, true>;
        } else if constexpr (KQ == 8) {
            if (nl != 3) {
                yg_set_error("large linear model: streamed operands of fewer than three levels need d > 32");
                return YG_ERR_STATE;
            }
            kern = free_noise ? linear_dmma_mh_kernel<KQ, 3, true, true> : linear_dmma_mh_kernel<KQ, 3, false, true>;
        } else {
            yg_set_error("large linear model: streamed operands need d > 16");
            return YG_ERR_STATE;
        }
    } else {
        kern = nl == 3 ? (free_noise ? linear_dmma_mh_kernel<KQ, 3, true> : linear_dmma_mh_kernel<KQ, 3, false>)
             : nl == 2 ? (free_noise ? linear_dmma_mh_kernel<KQ, 2, true> : linear_dmma_mh_kernel<KQ, 2, false>)
                       : (free_noise ? linear_dmma_mh_kernel<KQ, 1, true> : linear_dmma_mh_kernel<KQ, 1, false>);
    }
    YG_CUDA_CHECK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sp.total));
    const int64_t tiles = (a.n_chains + 7) / 8;
    // persistent grid, every CTA resident (one per SM): the balanced schedule lets warps wait on one another
    const int grid = (int)std::max<int64_t>(1, std::min<int64_t>((tiles + sp.warps - 1) / sp.warps, e->sm_count));
    YG_CUDA_CHECK(cudaMemsetAsync(e->big_done, 0, sizeof(long long) * (size_t)tiles, st));
    kern<<<grid, sp.warps * 32, sp.total, st>>>(a, reinterpret_cast<const DevBigHeader *>(e->d_problem), e->big_done, sp);
    YG_CUDA_CHECK(cudaGetLastError());
    e->last_grid = grid;
    e->last_block = sp.warps * 32;
    e->last_smem = (int)sp.total;
    e->launches += 1;
    return YG_OK;
}

}  // namespace

int yg_launch_linear_big(yg_ensemble *e, const RunArgs &a, cudaStream_t st)
{
    const DevBigHeader *hh = reinterpret_cast<const DevBigHeader *>(e->h_problem.data());
    switch (hh->kp) {       // 16, 32 or 64 (build_big_blob)
    case 16: return launch_t<4>(e, a, st);
    case 32: return launch_t<8>(e, a, st);
    default: return launch_t<16>(e, a, st);
    }
}

int yg_launch_logpost_big(yg_ensemble *e, int level, const double *theta, int64_t n, double *out, cudaStream_t st)
{
    const int grid = (int)std::max<int64_t>(1, std::min<int64_t>((n + 127) / 128, (int64_t)e->sm_count * 16));
    big_logpost_kernel<<<grid, 128, 0, st>>>(reinterpret_cast<const DevBigHeader *>(e->d_problem), level, theta, n, out);
    YG_CUDA_CHECK(cudaGetLastError());
    e->launches += 1;
    return YG_OK;
}

int yg_dmma_peak(int device, double ms, double *tflops_out)
{
    YG_CUDA_CHECK(cudaSetDevice(device));
    int sms = 148;
    YG_CUDA_CHECK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device));
    double *sink = nullptr;
    YG_CUDA_CHECK(cudaMalloc((void **)&sink, 8));
    cudaEvent_t e0, e1;
    cudaEventCreate(&e0);
    cudaEventCreate(&e1);
    int iters = 2000;
    double best = 0.0;
    for (int rep = 0; rep < 6; rep++) {
        cudaEventRecord(e0);
        dmma_peak_kernel<<<sms, 256>>>(sink, iters, 1.0);
        cudaEventRecord(e1);
        cudaEventSynchronize(e1);
        float t = 0.f;
        cudaEventElapsedTime(&t, e0, e1);
        const double flop = 2.0 * 16 * 8 * 4 * 8.0 * iters * 8.0 * sms;       // per mma x 8 chains x 8 warps x SMs
        if (rep > 0) best = std::max(best, flop / (t * 1e-3) / 1e12);
        if (t < ms / 6.0) iters *= 2;
    }
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    cudaFree(sink);
    YG_CUDA_CHECK(cudaGetLastError());
    *tflops_out = best;
    return YG_OK;
}
