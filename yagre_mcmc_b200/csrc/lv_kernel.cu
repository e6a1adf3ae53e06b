// lv_kernel.cu -- the headline hot path: Metropolis-Hastings over an ensemble of
// independent chains on the Lotka-Volterra (RK4) posterior, single level (MRW)
// or two-level delayed acceptance (MLDA with one surrogate).
//
// Reference semantics restated (rkutri/yagre-mcmc):
//   step loop            chain/metropolisHastings.py:103-120
//   proposal             chain/method/mrw.py:27-38 -> statistics/gaussian.py:61-66; pCN: chain/method/pcn.py:23-35
//   equality skip        chain/metropolisHastings.py:60-61, parameter/vector.py:37-45
//   likelihood           statistics/likelihood.py:33-39,74-84, statistics/covariance.py:19-22
//   prior / posterior    statistics/gaussian.py:19-24, chain/target.py:19-22
//   coarse sub-chain     chain/method/mlda.py:100-110
//   fine screen          chain/method/mlda.py:146-154 (this summation order)
//   Welford diagnostics  chain/diagnostics.py:91-94, statistics/estimation.py:36-53
//
// B200 mapping (DESIGN.md "LV kernel"):
//   * persistent CTAs, grid = SMs x blocks_per_sm, every CTA resident; a CTA owns
//     a contiguous range of chains and walks it in chunks of <= CMAX chains, each
//     chunk running all n_steps with no inter-CTA communication;
//   * the unit of FP64 work is one ODE integration = (chain, design point): after
//     the owners' phase has proposed, the CTA spreads `active chains x n_data`
//     integrations over ALL its threads, so a chain whose coarse sub-chain did not
//     move (no fine evaluation, mlda.py / metropolisHastings.py:60-61) costs
//     nothing in the fine phase -- block-level compaction instead of lane masks;
//   * ODE state and the chain's six scaled rate constants live in registers, chain
//     state lives in shared memory between phases so the integration loop stays
//     small; one CTA of 768 threads per SM (80 registers per thread) by default;
//   * the problem blob (design points, observations, precisions) is staged once
//     per CTA into shared memory by one TMA bulk copy (cp.async.bulk + mbarrier);
//   * proposal noise does not depend on the chain state (counter-based Philox), so
//     it is produced INSIDE the evaluation phases, one sub-step ahead of its use:
//     the integer Philox rounds of the warps that draw noise overlap the FP64-pipe
//     work of the warps that are already integrating.
#include "ensemble.h"
#include "lv_model.cuh"
#include "smem_plan.h"
#include <math_constants.h>

namespace {

constexpr int LV_D = 2;

#ifdef YG_TIMERS
YG_DEVFN long long yg_clk()
{
    long long t;
    asm volatile("mov.u64 %0, %%clock64;" : "=l"(t)::"memory");
    return t;
}
#endif

YG_DEVFN uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

// One TMA bulk copy global -> shared, completion on an mbarrier (UBLKCP in SASS).
YG_DEVFN void tma_stage_blob(void *dst, const void *src, uint32_t bytes, uint64_t *mbar)
{
    if (threadIdx.x == 0) {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(smem_u32(mbar)));
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(mbar)), "r"(bytes)
                     : "memory");
        asm volatile(
            "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                smem_u32(dst)),
            "l"(src), "r"(bytes), "r"(smem_u32(mbar))
            : "memory");
    }
    uint32_t done = 0;
    while (!done) {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], 0;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(done)
            : "r"(smem_u32(mbar))
            : "memory");
    }
}

// u / d for 0 <= u < 2^24 via a float reciprocal and one correction step: two integer
// divisions per work unit were a measurable share of the non-FP64 issue slots.
// Appends to a shared-memory list with ONE atomic per converged group of lanes.
YG_DEVFN void list_append(int *list, int *count, int value, int limit)
{
    const unsigned m = __activemask();
    const int leader = __ffs(m) - 1, lane = threadIdx.x & 31;
    int base = 0;
    if (lane == leader) base = atomicAdd(count, __popc(m));
    base = __shfl_sync(m, base, leader);
    YG_CHK(base + __popc(m & ((1u << lane) - 1u)), limit);
    list[base + __popc(m & ((1u << lane) - 1u))] = value;
}

YG_DEVFN int fast_div(int u, int d, float inv)
{
    int q = __float2int_rz(__int2float_rz(u) * inv);
    const int r = u - q * d;
    q += (r >= d) ? 1 : 0;
    q -= (r < 0) ? 1 : 0;
    return q;
}

// Lane of the k-th (0-based) set bit of m; requires k < popc(m).
YG_DEVFN int nth_set_bit(unsigned m, int k)
{
    int pos = 0;
#pragma unroll
    for (int w = 16; w > 0; w >>= 1) {
        const int lo = __popc(m & ((1u << w) - 1u));
        if (k >= lo) { k -= lo; pos += w; m >>= w; }
    }
    return pos;
}

template <bool TWO_LEVEL, int MAXT>
__global__ void __launch_bounds__(MAXT, 1) lv_mh_kernel(const RunArgs a, const LvSmemPlan sp, const int seg_len,
                                                          const bool early_reject)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int tid = threadIdx.x, nthr = blockDim.x;

    // ---- shared memory carve-up (smem_plan.h) ------------------------------------
    const int cmax = sp.cmax, nd_max = sp.nd_max;
    DevProblemHeader *pb = reinterpret_cast<DevProblemHeader *>(smem_raw);
    double *chain = reinterpret_cast<double *>(smem_raw + sp.off[LV_CHAIN]);
    double *q = reinterpret_cast<double *>(smem_raw + sp.off[LV_Q]);
    double *sx = reinterpret_cast<double *>(smem_raw + sp.off[LV_SX]);
    double *sy = reinterpret_cast<double *>(smem_raw + sp.off[LV_SY]);
    double *nz = reinterpret_cast<double *>(smem_raw + sp.off[LV_NZ]);
    double *qmax = reinterpret_cast<double *>(smem_raw + sp.off[LV_QMAX]);
    double *qpart = reinterpret_cast<double *>(smem_raw + sp.off[LV_QPART]);
    double *qsum = reinterpret_cast<double *>(smem_raw + sp.off[LV_QSUM]);
    unsigned long long *nacc = reinterpret_cast<unsigned long long *>(smem_raw + sp.off[LV_NACC]);
    int *list0 = reinterpret_cast<int *>(smem_raw + sp.off[LV_LIST0]);
    int *segdone = reinterpret_cast<int *>(smem_raw + sp.off[LV_SEGDONE]);
    int *perm = reinterpret_cast<int *>(smem_raw + sp.off[LV_PERM]);
    unsigned char *evald = smem_raw + sp.off[LV_EVALD];
    uint64_t *mbar = reinterpret_cast<uint64_t *>(smem_raw + sp.mbar);
    int *nact = reinterpret_cast<int *>(smem_raw + sp.nact);
    unsigned long long *blk_cnt = reinterpret_cast<unsigned long long *>(smem_raw + sp.blk_cnt);
    int *qhead = reinterpret_cast<int *>(smem_raw + sp.qhead);        // work-queue head of the current phase
    YG_CHK(sp.total - 1, yg_dynamic_smem_bytes());                     // the plan fits the launch

    tma_stage_blob(pb, a.problem, (uint32_t)((a.problem_bytes + 15u) & ~15u), mbar);
    if (tid < 6) blk_cnt[tid] = 0ull;
    if (tid < 2) nact[tid] = 0;
    for (int i = tid; i < nd_max; i += nthr) perm[i] = i;

    const double *tail = dev_tail(pb);
    const int J = TWO_LEVEL ? pb->J : 1;
    const int n_lvl = TWO_LEVEL ? 2 : 1;
    const double L00 = pb->prop_L[0], L10 = pb->prop_L[LV_D], L11 = pb->prop_L[LV_D + 1];
    const bool pcn = pb->proposal == YG_PROPOSAL_PCN;
    const int n_phases = TWO_LEVEL ? J + 1 : 1;

    // Early rejection at level 0 (the coarse level, or the only one): a proposal whose partial misfit sum
    // passed its budget is rejected whatever the remaining design points give, so their integrations are
    // skipped.  Exact only when every q_n >= 0 and never NaN: diagonal noise precision with positive finite
    // entries and finite data (a non-finite forward output then gives q = +inf).  Only for levels of one
    // segment per item, where a skipped unit has no successor waiting on it.
    bool skip_lvl0 = false;
    {
        const DevLevel &L0 = pb->lvl[0];
        const double *P = L0.noise_prec;
        bool ok = early_reject && L0.data_dim == 2 && L0.rk4_steps <= seg_len && P[1] == 0.0 && P[2] == 0.0 &&
                  P[0] > 0.0 && P[3] > 0.0 && isfinite(P[0]) && isfinite(P[3]);
        for (int i = 0; ok && i < 2 * L0.n_data; i++) ok = isfinite(tail[L0.data_off + i]);
        skip_lvl0 = ok;
    }
    // design-point order of the level-0 queue: learned from the misfits of the launch's first level-0 phase
    bool perm_ready = false;

#ifdef YG_BOUNDS_CHECK
    auto ch_at = [&](const int field, const int c) -> double & {
        YG_CHK(c, cmax);
        return chain[field * cmax + c];
    };
#define CH(field, c) ch_at(LvSlot::field, (c))
#else
#define CH(field, c) chain[(LvSlot::field) * cmax + (c)]
#endif

    // chains of this CTA: even split of [0, n_chains) over the grid
    const int64_t cta_lo = (a.n_chains * (int64_t)blockIdx.x) / gridDim.x;
    const int64_t cta_hi = (a.n_chains * (int64_t)(blockIdx.x + 1)) / gridDim.x;
    const int64_t N = a.n_chains;

    // ---- one phase of forward evaluations over the compacted list ---------------
    // Work unit = (item, segment): item = (active chain, design point), segment = `seg_len`
    // consecutive RK4 steps.  Units are ordered segment-major and handed out 32 at a time from
    // a shared-memory queue: a warp that finishes grabs the next batch, so there is NO barrier
    // inside a phase (with barriers between rounds the warps of a sub-partition finished a
    // round one after another and the FP64 pipe ran dry at the end of every round: 5-8 % of
    // the phase, profiles/r01_summary.md).  A unit of segment s > 0 continues the state its
    // predecessor left in sx/sy; the predecessor has a smaller queue index, so it was grabbed
    // earlier and never waits on anything later: the spin on segdone[item] cannot deadlock.
    // A batch never holds two segments of one item (batch size <= nItems).
    //
    // With early rejection (skip_lvl0, level 0) a warp drops the units of proposals whose rejection is already
    // certain when it takes them, and keeps taking units until its 32 lanes hold live ones: FP64 instructions
    // issue per warp, so a skipped lane saves nothing unless its slot is refilled.  Design points are visited
    // in the order `perm`; q stays indexed by the design point, so results do not depend on the order.
    auto eval_phase = [&](const int lvl, const int cur, const double h, const LvStepConsts &kc,
                          unsigned long long &n_skip) {
        const DevLevel &Lv = pb->lvl[lvl];
        const int na = nact[cur];
        const int nD = Lv.n_data;
        const int nItems = na * nD;
        const int Nrk = Lv.rk4_steps;
        const int nSeg = (Nrk + seg_len - 1) / seg_len;
        const int nUnits = nItems * nSeg;
        const int batch = min(32, nItems);
        const int *lst = list0 + cur * cmax;
        const double *design = tail + Lv.design_off;
        const double *data = tail + Lv.data_off;
        const double P00 = Lv.noise_prec[0], P01 = Lv.noise_prec[1], P10 = Lv.noise_prec[2], P11 = Lv.noise_prec[3];
        const float inv_items = 1.0f / (float)nItems, inv_na = 1.0f / (float)na;
        const int lane = tid & 31;
        if (tid == 0) {
            nact[cur ^ 1] = 0;
            blk_cnt[2 + lvl] += (unsigned long long)na;
        }
        auto integrate = [&](const int steps, const LvRates &r, double &x, double &y) {
#ifdef YG_TIMERS
            lv_integrate(kc, r, a.thin == 7 ? 0 : steps, x, y);   // thin == 7: overhead-only run
#else
            lv_integrate(kc, r, steps, x, y);
#endif
        };
        // misfit of design point n from the forward output (x, y)
        auto misfit = [&](const int n, double x, double y) {
            // non-finite forward output -> +inf (policy of the oracle's RK4 plugin)
            x = isfinite(x) ? x : CUDART_INF;
            y = isfinite(y) ? y : CUDART_INF;
            const double r0 = x - data[2 * n], r1 = y - data[2 * n + 1];
            // r' P r with P applied first; exact zeros skipped (diagonal noise, inf-safe)
            double t0 = P00 * r0;
            if (P01 != 0.0) t0 = fma(P01, r1, t0);
            double t1 = (P10 != 0.0) ? P10 * r0 : 0.0;
            t1 = (P10 != 0.0) ? fma(P11, r1, t1) : P11 * r1;
            return fma(r1, t1, r0 * t0);
        };
        if (lvl == 0 && skip_lvl0) {      // one segment per item: unit == item, design-point major
            int mine = 0, pend = 0;        // this lane's unit; lanes [0, pend) hold one
            bool drained = false;
            for (;;) {
                while (pend < 32 && !drained) {
                    const int want = 32 - pend;
                    int u0 = 0;
                    if (lane == 0) u0 = atomicAdd(qhead, want);
                    u0 = __shfl_sync(0xffffffffu, u0, 0);
                    if (u0 >= nUnits) { drained = true; break; }
                    const int u = u0 + lane;
                    bool live = false;
                    if (lane < want && u < nUnits) {
                        const int nq = fast_div(u, na, inv_na), ai = u - nq * na;
                        YG_CHK(ai, cmax); YG_CHK(nq, nD);
                        const int c = lst[ai];
                        YG_CHK(c, cmax);
                        live = !(qpart[c] > qmax[c]);
                        if (!live) n_skip += 1ull;
                    }
                    const unsigned m = __ballot_sync(0xffffffffu, live);
                    const int k = lane - pend, nl = __popc(m);
                    const int v = __shfl_sync(0xffffffffu, u, (k >= 0 && k < nl) ? nth_set_bit(m, k) : lane);
                    if (k >= 0 && k < nl) mine = v;
                    pend += nl;
                }
                if (pend == 0) break;
                if (lane < pend) {
                    const int nq = fast_div(mine, na, inv_na), ai = mine - nq * na;
                    YG_CHK(ai, cmax); YG_CHK(nq, nD);
                    const int n = perm[nq], c = lst[ai];
                    YG_CHK(n, nD); YG_CHK(c, cmax);
                    const LvRates r = lv_rates(h, CH(BETA, c), CH(DELTA, c));
                    double x = design[2 * n], y = design[2 * n + 1];
                    integrate(Nrk, r, x, y);
                    const double qn = misfit(n, x, y);
                    q[n * cmax + c] = qn;
                    atomicAdd(&qpart[c], qn);
                }
                pend = 0;
                __syncwarp();
            }
            return;
        }
        for (;;) {
            int u = 0;
            if (lane == 0) u = atomicAdd(qhead, batch);
            u = __shfl_sync(0xffffffffu, u, 0);
            if (u >= nUnits) break;
            u += lane;
            if (lane < batch && u < nUnits) {
                const int seg = fast_div(u, nItems, inv_items), it = u - seg * nItems;
                const int n = fast_div(it, na, inv_na), ai = it - n * na;
                YG_CHK(ai, cmax); YG_CHK(n, nD); YG_CHK(it, nd_max * cmax);
                const int c = lst[ai];
                YG_CHK(c, cmax);
                const LvRates r = lv_rates(h, CH(BETA, c), CH(DELTA, c));
                double x, y;
                if (seg == 0) { x = design[2 * n]; y = design[2 * n + 1]; }
                else {
                    const volatile int *flag = segdone + it;
                    while (*flag < seg) __nanosleep(32);
                    __threadfence_block();
                    x = sx[it]; y = sy[it];
                }
                integrate(min(seg_len, Nrk - seg * seg_len), r, x, y);
                if (seg + 1 < nSeg) {
                    sx[it] = x; sy[it] = y;
                    __threadfence_block();
                    *(volatile int *)(segdone + it) = seg + 1;
                } else {
                    q[n * cmax + c] = misfit(n, x, y);
                }
            }
            __syncwarp();
        }
    };

    auto log_prior = [&](int lvl, double t0, double t1) {
        const DevLevel &Lv = pb->lvl[lvl];
        const double x[2] = {t0 - Lv.prior_mean[0], t1 - Lv.prior_mean[1]};
        return -0.5 * quad_form<2>(Lv.prior_prec, LV_D, x, 2);
    };
    auto log_post_from_q = [&](int lvl, int c, double t0, double t1) {
        const int nD = pb->lvl[lvl].n_data;
        const double logL = -0.5 * (nD <= 128 ? np_sum_le128(q + c, nD, cmax) : np_pairwise_sum(q + c, nD, cmax));
        // tempering = 1 (exact identity) unless the level is a TemperedUnnormalisedPosterior (target.py:40-43)
        return __dmul_rn(pb->lvl[lvl].tempering, logL) + log_prior(lvl, t0, t1);
    };

    // noise: injected arrays are indexed by (step, sub-step), never by call count.  draw_z /
    // draw_u fill the chain's slot of nz one phase ahead of its use, always from the thread
    // that owns the chain (producer == consumer, no barrier needed).  The uniform goes to slot 3:
    // the owners' phase moves it to slot 2 after slot 2 decided the previous sub-step, so the
    // budget of the proposals about to be evaluated is known before the barrier.
    auto draw_z = [&](int c, int64_t g, int64_t n, int j) {
        const uint64_t gid = (uint64_t)(a.chain_offset + g);
        const int64_t zi = ((n * J + j) * LV_D) * N + g;
        YG_CHK(c, cmax); YG_CHK(g, N);
        if (a.noise_mode != YG_NOISE_PHILOX) YG_CHK(zi + N, a.n_steps * J * LV_D * N);
        double z0, z1;
        if (a.noise_mode == YG_NOISE_INJECT) {
            z0 = a.z[zi]; z1 = a.z[zi + N];
        } else {
            philox_normal_pair(a.seed, gid, (uint64_t)(a.step0 + n), (uint32_t)j, 0u, z0, z1);
            if (a.noise_mode == YG_NOISE_RECORD) { a.z[zi] = z0; a.z[zi + N] = z1; }
        }
        nz[c] = z0; nz[cmax + c] = z1;
    };
    auto draw_u = [&](int c, int64_t g, int64_t n, int j, bool fine) {
        const uint64_t gid = (uint64_t)(a.chain_offset + g);
        double *arr = fine ? a.u_f : a.u_c;
        const int64_t i = fine ? n * N + g : (n * J + j) * N + g;
        YG_CHK(c, cmax); YG_CHK(g, N);
        if (a.noise_mode != YG_NOISE_PHILOX) YG_CHK(i, fine ? a.n_steps * N : a.n_steps * J * N);
        double u;
        if (a.noise_mode == YG_NOISE_INJECT) u = arr[i];
        else {
            u = philox_uniform(a.seed, gid, (uint64_t)(a.step0 + n), fine ? YG_SUB_FINE : (uint32_t)j);
            if (a.noise_mode == YG_NOISE_RECORD) arr[i] = u;
        }
        nz[3 * cmax + c] = u;
    };

    // Adaptive Metropolis (chain/adaptive.py:55-60: update() before every proposal of the MRW chain it drives,
    // with that chain's current state = the sub-chain state s; t = number of earlier updates).  Per-chain
    // moments and proposal factor stay in (L2-resident) global memory: they are touched once per proposal by the
    // chain's owner only, and the shared-memory budget belongs to the evaluation phases.  Recurrence of
    // DESIGN.md section 5 in the unfused numpy order of oracle/ref_harness.py HaarioAdaptiveCovariance; the
    // 2 x 2 Cholesky in LAPACK dpotf2's order (reciprocal scaling), like the reference's DenseCovarianceMatrix.
    auto am_update = [&](const int64_t g, const int64_t t, const double x0, const double x1, double &l00, double &l10,
                         double &l11) {
        l00 = a.prop_L[g]; l10 = a.prop_L[2 * N + g]; l11 = a.prop_L[3 * N + g];
        if (t < a.am_idle) return;
        const int64_t n_am = t - a.am_idle + 1;
        double m0 = a.am_mean[g], m1 = a.am_mean[N + g];
        double v00 = a.am_m2[g], v01 = a.am_m2[N + g], v10 = a.am_m2[2 * N + g], v11 = a.am_m2[3 * N + g];
        const double dn = (double)n_am;
        const double d0 = __dsub_rn(x0, m0), d1 = __dsub_rn(x1, m1);
        m0 = __dadd_rn(m0, d0 / dn); m1 = __dadd_rn(m1, d1 / dn);
        const double e0 = __dsub_rn(x0, m0), e1 = __dsub_rn(x1, m1);
        v00 = __dadd_rn(v00, __dmul_rn(d0, e0)); v01 = __dadd_rn(v01, __dmul_rn(d0, e1));
        v10 = __dadd_rn(v10, __dmul_rn(d1, e0)); v11 = __dadd_rn(v11, __dmul_rn(d1, e1));
        a.am_mean[g] = m0; a.am_mean[N + g] = m1;
        a.am_m2[g] = v00; a.am_m2[N + g] = v01; a.am_m2[2 * N + g] = v10; a.am_m2[3 * N + g] = v11;
        if (n_am >= a.am_collect && n_am >= 2 && (a.am_refresh == 1 || ((n_am - a.am_collect) % a.am_refresh) == 0)) {
            const double dm = (double)(n_am - 1);
            const double c00 = __dmul_rn(a.am_scale, __dadd_rn(__dmul_rn(0.5, __dadd_rn(v00, v00)) / dm, a.am_eps));
            const double c10 = __dmul_rn(a.am_scale, __dmul_rn(0.5, __dadd_rn(v10, v01)) / dm);
            const double c11 = __dmul_rn(a.am_scale, __dadd_rn(__dmul_rn(0.5, __dadd_rn(v11, v11)) / dm, a.am_eps));
            if (c00 > 0.0) {
                const double n00 = sqrt(c00), n10 = __dmul_rn(c10, 1.0 / n00);
                const double s11 = __dsub_rn(c11, __dmul_rn(n10, n10));
                if (s11 > 0.0) {
                    l00 = n00; l10 = n10; l11 = sqrt(s11);
                    a.prop_L[g] = l00; a.prop_L[2 * N + g] = l10; a.prop_L[3 * N + g] = l11;
                }
            }
        }
    };

#ifdef YG_TIMERS
    // per-warp phase timers (dev build only): [0] owners' work [1] wait at the barrier after it
    // [2] noise draws [3] evaluation loop [4] wait at the trailing barrier [5] commit
    // [6] coarse items (tid 0) [7] fine items (tid 0)
    long long dbg_t[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    long long dbg_last = yg_clk();
    const long long dbg_start = dbg_last;
#endif
    int cur = 0;
    unsigned long long my_skip = 0ull;      // level-0 integrations skipped by early rejection
    for (int64_t cb = cta_lo; cb < cta_hi; cb += cmax) {
        const int C = (int)min((int64_t)cmax, cta_hi - cb);
        __syncthreads();
        // ---- load chunk state ---------------------------------------------------
        for (int c = tid; c < C; c += nthr) {
            const int64_t g = cb + c;
            YG_CHK(g, N);
            CH(TH0, c) = a.theta[g];
            CH(TH1, c) = a.theta[N + g];
            CH(LP0, c) = a.logpost[g];
            CH(LP1, c) = TWO_LEVEL ? a.logpost[N + g] : 0.0;
            CH(WM0, c) = a.w_mean[g];
            CH(WM1, c) = a.w_mean[N + g];
            CH(W00, c) = a.w_m2[g];
            CH(W01, c) = a.w_m2[N + g];
            CH(W10, c) = a.w_m2[2 * N + g];
            CH(W11, c) = a.w_m2[3 * N + g];
            nacc[c] = a.n_accept[g];
            if (a.n_steps > 0) {
                draw_u(c, g, 0, 0, n_phases == 1);
                draw_z(c, g, 0, 0);
            }
        }
        unsigned long long my_acc = 0ull, my_cacc = 0ull;      // accepted transitions / accepted coarse sub-steps

        int64_t thin_left = a.thin, thin_out = -1;
        for (int64_t n = 0; n < a.n_steps; n++) {
            const double wn = (double)(a.welford_n0 + n + 1);
            // (n + 1) % thin == 0 without a 64-bit division per transition
            const bool store_now = (--thin_left == 0);
            if (store_now) { thin_left = a.thin; thin_out++; }
            // Phases j = 0..J-1: decide sub-step j-1, propose sub-step j, evaluate level 0.
            // Two level only, phase j = J: decide sub-step J-1, evaluate level 1 where the
            // sub-chain moved.  Then the commit below decides the transition.
            for (int j = 0; j < n_phases; j++) {
                // =============== owners' phase ===================================
                if (tid == 0) *qhead = 0;
                if (pb->lvl[(TWO_LEVEL && j == J) ? 1 : 0].rk4_steps > seg_len)
                    for (int i = tid; i < C * nd_max; i += nthr) segdone[i] = 0;
                for (int c = tid; c < C; c += nthr) {
                    double s0, s1, lps;
                    if (j == 0) {
                        // FullDiagnostics: Welford of the pre-transition state
                        // (diagnostics.py:91-94, estimation.py:36-53)
                        const double t0 = CH(TH0, c), t1 = CH(TH1, c);
                        const double d0 = t0 - CH(WM0, c), d1 = t1 - CH(WM1, c);
                        const double m0 = CH(WM0, c) + d0 / wn, m1 = CH(WM1, c) + d1 / wn;
                        const double e0 = t0 - m0, e1 = t1 - m1;
                        CH(WM0, c) = m0; CH(WM1, c) = m1;
                        CH(W00, c) += d0 * e0; CH(W01, c) += d0 * e1;
                        CH(W10, c) += d1 * e0; CH(W11, c) += d1 * e1;
                        s0 = t0; s1 = t1; lps = CH(LP0, c);
                    } else {
                        // coarse decision of sub-step j-1 (mrw.py:51-57)
                        s0 = CH(S0, c); s1 = CH(S1, c); lps = CH(LPS, c);
                        if (evald[c]) {
                                const double p0 = CH(P0, c), p1 = CH(P1, c);
                            YG_CHK(c, cmax);
                            if (!(skip_lvl0 && qpart[c] > qmax[c])) {           // else rejection certified
                                const double lpp = log_post_from_q(0, c, p0, p1);
                                if (accept_rule(lpp - lps, nz[2 * cmax + c])) {      // u_c(n, j-1)
                                    s0 = p0; s1 = p1; lps = lpp;
                                    my_cacc += 1ull;
                                }
                            }
                        }
                    }
                    CH(S0, c) = s0; CH(S1, c) = s1; CH(LPS, c) = lps;
                    nz[2 * cmax + c] = nz[3 * cmax + c];      // the uniform that decides this phase's proposals
                    if (j < J) {
                        double l00 = L00, l10 = L10, l11 = L11;
                        if (a.adaptive) am_update(cb + c, (a.am_t0 + n) * J + j, s0, s1, l00, l10, l11);
                        // propose sub-step j: p = s + L z  (gaussian.py:61-66), unfused like numpy
                        const double z0 = nz[c], z1 = nz[cmax + c];          // z(n, j)
                        const double lz0 = __dmul_rn(l00, z0);
                        const double lz1 = (l10 != 0.0) ? __dadd_rn(__dmul_rn(l10, z0), __dmul_rn(l11, z1))
                                                        : __dmul_rn(l11, z1);
                        double p0, p1;
                        if (pcn) {    // pcn.py:30-35: sqrt(1-t) * state + sqrt(t) * (mean + L z)
                            p0 = __dadd_rn(__dmul_rn(pb->pcn_a, s0), __dmul_rn(pb->pcn_b, __dadd_rn(pb->pcn_mean[0], lz0)));
                            p1 = __dadd_rn(__dmul_rn(pb->pcn_a, s1), __dmul_rn(pb->pcn_b, __dadd_rn(pb->pcn_mean[1], lz1)));
                        } else {
                            p0 = __dadd_rn(s0, lz0);
                            p1 = __dadd_rn(s1, lz1);
                        }
                        const bool eq = (p0 == s0) && (p1 == s1);   // vector.py:37-45
                        evald[c] = !eq;
                        CH(P0, c) = p0; CH(P1, c) = p1;
                        if (!eq) {
                            CH(BETA, c) = exp(p0);     // LotkaVolterraParameter.evaluate, testSetup.py:57-58
                            CH(DELTA, c) = exp(p1);
                            if (skip_lvl0) {
                                qpart[c] = 0.0;
                                qmax[c] = perm_ready ? reject_budget(log_prior(0, p0, p1), lps, nz[2 * cmax + c],
                                                                     pb->lvl[0].tempering)
                                                     : CUDART_INF;
                            }
                            list_append(list0 + cur * cmax, &nact[cur], c, cmax);
                        }
                    } else {
                        // sub-chain finished: s is the MLDA proposal (mlda.py:106-110); a chain whose
                        // sub-chain did not move is rejected without a fine evaluation and without
                        // consuming a uniform (metropolisHastings.py:60-61)
                        const bool moved = !((s0 == CH(TH0, c)) && (s1 == CH(TH1, c)));
                        evald[c] = moved;
                        if (moved) {
                            CH(BETA, c) = exp(s0);
                            CH(DELTA, c) = exp(s1);
                            list_append(list0 + cur * cmax, &nact[cur], c, cmax);
                        }
                    }
                }
#ifdef YG_TIMERS
                const long long dbg_own = yg_clk();
                dbg_t[0] += dbg_own - dbg_last;
#endif
                __syncthreads();
                // =============== forward evaluations =============================
#ifdef YG_TIMERS
                const long long tA = yg_clk();
                dbg_t[1] += tA - dbg_own;
                if (tid == 0) dbg_t[6 + ((TWO_LEVEL && j == J) ? 1 : 0)] += nact[cur] * pb->lvl[(TWO_LEVEL && j == J) ? 1 : 0].n_data;
#endif
                // noise one phase ahead: the uniform that decides the proposals of the next phase,
                // and the normals of the next proposal
                {
                    const bool last = (j == n_phases - 1);
                    for (int c = tid; c < C; c += nthr) {
                        const int64_t g = cb + c;
                        if (!last) {
                            draw_u(c, g, n, j + 1, j + 1 == n_phases - 1);
                            if (j + 1 < J) draw_z(c, g, n, j + 1);
                        } else if (n + 1 < a.n_steps) {
                            draw_u(c, g, n + 1, 0, n_phases == 1);
                            draw_z(c, g, n + 1, 0);
                        }
                    }
                }
#ifdef YG_TIMERS
                const long long dbg_nz = yg_clk();
                dbg_t[2] += dbg_nz - tA;
#endif
                // two inlined copies so that h and the chain-independent rates are constant-bank operands
                if (TWO_LEVEL && j == J) eval_phase(1, cur, a.lv_h[1], a.lv_k[1], my_skip);
                else eval_phase(0, cur, a.lv_h[0], a.lv_k[0], my_skip);
#ifdef YG_TIMERS
                const long long dbg_ev = yg_clk();
                dbg_t[3] += dbg_ev - dbg_nz;
#endif
                __syncthreads();
#ifdef YG_TIMERS
                dbg_last = yg_clk();
                dbg_t[4] += dbg_last - dbg_ev;
#endif
                if (skip_lvl0 && !perm_ready) {
                    // first level-0 phase of the launch, evaluated in full: design points by total misfit,
                    // largest first (ties by index), so that rejections are certified after fewer of them
                    const int nD = pb->lvl[0].n_data, na = nact[cur];
                    const int *lst = list0 + cur * cmax;
                    for (int i = tid; i < nD; i += nthr) {
                        double sum = 0.0;
                        for (int k = 0; k < na; k++) {
                            YG_CHK(lst[k], cmax);
                            sum += q[i * cmax + lst[k]];
                        }
                        YG_CHK(i, nd_max);
                        qsum[i] = sum;
                    }
                    __syncthreads();
                    for (int i = tid; i < nD; i += nthr) {
                        int rank = 0;
                        for (int k = 0; k < nD; k++) rank += (qsum[k] > qsum[i] || (qsum[k] == qsum[i] && k < i)) ? 1 : 0;
                        YG_CHK(rank, nd_max);
                        perm[rank] = i;
                    }
                    __syncthreads();
                    perm_ready = true;
                }
                cur ^= 1;
            }
            // =============== commit the transition ===============================
            for (int c = tid; c < C; c += nthr) {
                const int64_t g = cb + c;
                bool accepted = false;
                if (evald[c]) {
                    if (TWO_LEVEL) {
                        const double s0 = CH(S0, c), s1 = CH(S1, c);
                        const double lpf_s = log_post_from_q(1, c, s0, s1);
                        // mlda.py:148-152: pi_f(p) + pi_c(s) - pi_c(p) - pi_f(s), left to right
                        const double delta = lpf_s + CH(LP0, c) - CH(LPS, c) - CH(LP1, c);
                        if (accept_rule(delta, nz[2 * cmax + c])) {                  // u_f(n)
                            CH(TH0, c) = s0; CH(TH1, c) = s1;
                            CH(LP0, c) = CH(LPS, c); CH(LP1, c) = lpf_s;
                            accepted = true;
                        }
                    } else if (!(skip_lvl0 && qpart[c] > qmax[c])) {               // else rejection certified
                        const double p0 = CH(P0, c), p1 = CH(P1, c);
                        const double lpp = log_post_from_q(0, c, p0, p1);
                        if (accept_rule(lpp - CH(LP0, c), nz[2 * cmax + c])) {       // u_f(n)
                            CH(TH0, c) = p0; CH(TH1, c) = p1; CH(LP0, c) = lpp;
                            accepted = true;
                        }
                    }
                }
                if (accepted) { nacc[c] += 1ull; my_acc += 1ull; }
                if (a.accepted) a.accepted[n * N + g] = accepted ? 1 : 0;
                YG_CHK(c, cmax); YG_CHK(g, N);
                if (store_now) {
                    const int64_t o = thin_out;
                    YG_CHK(o, a.n_steps / a.thin);
                    if (a.samples) {
                        a.samples[(o * LV_D) * N + g] = CH(TH0, c);
                        a.samples[(o * LV_D + 1) * N + g] = CH(TH1, c);
                    }
                    if (a.lp_out) {
                        a.lp_out[(o * n_lvl) * N + g] = CH(LP0, c);
                        if (TWO_LEVEL) a.lp_out[(o * n_lvl + 1) * N + g] = CH(LP1, c);
                    }
                }
            }
#ifdef YG_TIMERS
            { const long long t = yg_clk(); dbg_t[5] += t - dbg_last; dbg_last = t; }
#endif
            // the next owners' phase touches only the owner's own slots and list `cur`,
            // whose counter was zeroed during the last evaluation phase: no barrier needed
        }

        // ---- store chunk state --------------------------------------------------
        for (int c = tid; c < C; c += nthr) {
            const int64_t g = cb + c;
            a.theta[g] = CH(TH0, c);
            a.theta[N + g] = CH(TH1, c);
            a.logpost[g] = CH(LP0, c);
            if (TWO_LEVEL) a.logpost[N + g] = CH(LP1, c);
            a.w_mean[g] = CH(WM0, c);
            a.w_mean[N + g] = CH(WM1, c);
            a.w_m2[g] = CH(W00, c);
            a.w_m2[N + g] = CH(W01, c);
            a.w_m2[2 * N + g] = CH(W10, c);
            a.w_m2[3 * N + g] = CH(W11, c);
            a.n_accept[g] = nacc[c];
        }
        if (my_acc) atomicAdd(&blk_cnt[1], my_acc);
        if (my_cacc) atomicAdd(&blk_cnt[4], my_cacc);
        if (my_skip) atomicAdd(&blk_cnt[5], my_skip);
        my_skip = 0ull;
        if (tid == 0) blk_cnt[0] += (unsigned long long)C * (unsigned long long)a.n_steps;
    }
    __syncthreads();
#ifdef YG_TIMERS
    if ((tid & 31) == 0 && a.lp_out == nullptr && a.samples != nullptr) {   // debug: timers into the samples buffer
        long long *o = reinterpret_cast<long long *>(a.samples) + 10 * (32 * blockIdx.x + (tid >> 5));
        for (int k = 0; k < 8; k++) o[k] = dbg_t[k];
        o[8] = yg_clk() - dbg_start;
        o[9] = 0;
    }
#endif
    if (tid < 4 && blk_cnt[tid]) atomicAdd(&a.counters[tid], blk_cnt[tid]);
    if (tid == 4 && blk_cnt[4]) atomicAdd(&a.counters[5], blk_cnt[4]);       // [4] is the middle level of three-level problems
    if (tid == 5 && blk_cnt[5]) atomicAdd(&a.counters[6], blk_cnt[5]);       // skipped level-0 integrations
#undef CH
}

}  // namespace

int yg_launch_lv(yg_ensemble *e, const RunArgs &a, cudaStream_t st)
{
    const DevProblemHeader *hp = reinterpret_cast<const DevProblemHeader *>(e->h_problem.data());
    const bool two = e->cfg.n_levels == 2;
    const int nd_max = std::max(hp->lvl[0].n_data, two ? hp->lvl[1].n_data : 0);
    const LvGeometry g = lv_geometry(a.problem_bytes, nd_max, a.n_chains, e->sm_count, e->cfg.blocks_per_sm,
                                     e->cfg.threads_per_block);
    const int threads = g.threads;
    if (threads % 32 || threads > 1024) {
        yg_set_error("threads_per_block must be a multiple of 32 and <= 1024 (got %d)", threads);
        return YG_ERR_INVALID;
    }
    if (g.cmax < 1) {
        yg_set_error("problem blob too large for shared memory (%u bytes)", g.plan.total);
        return YG_ERR_UNSUPPORTED;
    }
    RunArgs args = a;
    for (int l = 0; l < e->cfg.n_levels; l++) {
        args.lv_h[l] = hp->lvl[l].T / (double)hp->lvl[l].rk4_steps;
        args.lv_k[l] = lv_step_consts(hp->lvl[l].alpha, hp->lvl[l].gamma, args.lv_h[l]);
    }
    // register budget follows the thread count: 128 (<= 512 threads), 80 (<= 768), 64 (<= 1024)
    auto kern = threads <= 512 ? (two ? lv_mh_kernel<true, 512> : lv_mh_kernel<false, 512>)
                : threads <= 768 ? (two ? lv_mh_kernel<true, 768> : lv_mh_kernel<false, 768>)
                                 : (two ? lv_mh_kernel<true, 1024> : lv_mh_kernel<false, 1024>);
    YG_CUDA_CHECK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)g.plan.total));
    const int seg_len = e->cfg.rk4_segment > 0 ? e->cfg.rk4_segment : 128;
    kern<<<g.grid, threads, g.plan.total, st>>>(args, g.plan, seg_len, e->cfg.early_reject_off == 0);
    YG_CUDA_CHECK(cudaGetLastError());
    e->last_grid = g.grid;
    e->last_block = threads;
    e->last_smem = (int)g.plan.total;
    e->launches += 1;
    return YG_OK;
}
