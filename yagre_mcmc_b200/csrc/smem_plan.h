// smem_plan.h -- the dynamic shared-memory layout of each step kernel, defined once for the kernel that carves it up
// and the launcher that sizes the launch: the LV kernel (lv_kernel.cu), the FP64 tensor path (linear_dmma_kernel.cu,
// and abi.cu's refusal of problems that do not fit) and the ring of the warp-specialised generic kernel
// (generic_kernel.cuh).  Host and device code.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <algorithm>

__host__ __device__ constexpr uint32_t smem_align16(uint32_t x) { return (x + 15u) & ~15u; }

// ---------------------------------------------------------------------------------------------------------------------
// LV kernel.  After the problem blob (rounded up to 16 bytes), with C = cmax chains per CTA and N = nd_max design points:
// ---------------------------------------------------------------------------------------------------------------------
// doubles per chain slot of the LV_CHAIN region
struct LvSlot {
    enum { TH0, TH1, LP0, LP1, S0, S1, LPS, P0, P1, BETA, DELTA, WM0, WM1, W00, W01, W10, W11, NDBL };
};

enum LvRegion {
    LV_CHAIN,       // double [NDBL][C]  chain slots (LvSlot)
    LV_Q,           // double [N][C]     misfit per design point
    LV_SX, LV_SY,   // double [N * C]    ODE state between segments, indexed by item
    LV_NZ,          // double [4][C]     z0, z1, uniform, next uniform
    LV_QMAX,        // double [C]        misfit budget (reject_budget)
    LV_QPART,       // double [C]        misfit summed so far
    LV_QSUM,        // double [N]        misfit per design point over the active chains
    LV_NACC,        // uint64 [C]        accept counts
    LV_LIST0,       // int [2][C]        active-chain lists
    LV_SEGDONE,     // int [N * C]       segments done per item
    LV_PERM,        // int [N]           level-0 design points, heaviest first
    LV_EVALD,       // uint8 [C]         padded to a multiple of 16 bytes
    LV_NREG
};

// Bytes of region r per chain, per (chain x design point) and per design point.
struct LvRegionSize {
    uint32_t chain, item, point;
};
__host__ __device__ constexpr LvRegionSize lv_region_size(int r)
{
    constexpr LvRegionSize size[LV_NREG] = {
        {8 * LvSlot::NDBL, 0, 0}, {0, 8, 0}, {0, 8, 0}, {0, 8, 0}, {8 * 4, 0, 0}, {8, 0, 0}, {8, 0, 0},
        {0, 0, 8},                {8, 0, 0}, {4 * 2, 0, 0}, {0, 4, 0}, {0, 0, 4}, {1, 0, 0}};
    return size[r];
}

struct LvSmemPlan {
    int cmax, nd_max;
    uint32_t off[LV_NREG];       // byte offset of each region
    // then, 16-byte aligned: the blob's mbarrier (uint64), nact (int [2]), blk_cnt (uint64 [6]), qhead (int)
    uint32_t mbar, nact, blk_cnt, qhead;
    uint32_t total;              // bytes of the launch
};

__host__ __device__ inline LvSmemPlan lv_smem_plan(uint32_t problem_bytes, int cmax, int nd_max)
{
    LvSmemPlan p{cmax, nd_max};
    uint32_t off = smem_align16(problem_bytes);
    for (int r = 0; r < LV_NREG; r++) {
        const LvRegionSize s = lv_region_size(r);
        p.off[r] = off;
        off += s.chain * cmax + s.item * cmax * nd_max + s.point * nd_max;
    }
    off = smem_align16(p.off[LV_EVALD] + smem_align16(cmax));     // the int arrays leave 4-byte alignment when N * C is odd
    p.mbar = off;
    p.nact = p.mbar + 8;
    p.blk_cnt = p.nact + 8;
    p.qhead = p.blk_cnt + 48;
    p.total = smem_align16(p.qhead + 4);
    return p;
}

// Bytes that one more chain adds to the regions, without the padding of LV_EVALD and of the mbarrier block.
__host__ __device__ inline uint32_t lv_bytes_per_chain(int nd_max)
{
    uint32_t b = 0;
    for (int r = 0; r < LV_NREG; r++) b += lv_region_size(r).chain + lv_region_size(r).item * nd_max;
    return b;
}

constexpr uint32_t LV_SMEM_BUDGET = 220 * 1024;    // per SM, shared by blocks_per_sm CTAs
constexpr int LV_MAX_CMAX = 1024;

struct LvGeometry {
    int grid, threads, cmax;     // cmax == 0: the blob leaves no room for one chain (plan is then the one of no chains)
    LvSmemPlan plan;
};

// Launch geometry of the LV kernel.  blocks_per_sm, threads_per_block <= 0: the defaults.  The caller checks threads.
inline LvGeometry lv_geometry(uint32_t problem_bytes, int nd_max, int64_t n_chains, int sm_count, int blocks_per_sm,
                              int threads_per_block)
{
    // Default geometry (profiles/r01_lv_tuning.md): ONE persistent CTA per SM with up to 768 threads
    // (6 warps per sub-partition saturate the FP64 pipe, and 768 threads leave 80 registers per thread:
    // fewer spills in the owners' phases than the 64 of 1024 threads, +2 %).  Several smaller CTAs per SM
    // finish at very different times because the FP64 issue arbiter is not fair between CTAs, which
    // leaves SMs half empty towards the end.
    const int bps = blocks_per_sm > 0 ? blocks_per_sm : 1;
    const int64_t ctas = std::min<int64_t>((int64_t)sm_count * bps, n_chains);
    LvGeometry g;
    g.threads = threads_per_block;
    if (g.threads <= 0) {
        const int64_t items = ((n_chains + ctas - 1) / ctas) * nd_max;
        g.threads = (int)std::min<int64_t>((bps == 1 ? 768 : 1024) / bps, std::max<int64_t>(128, (items + 31) / 32 * 32));
    }
    g.grid = (int)std::max<int64_t>(ctas, 1);
    // chains per chunk: the CTA's share, capped so that shared memory fits bps CTAs per SM
    const int64_t share = (n_chains + g.grid - 1) / g.grid;
    const uint32_t budget = LV_SMEM_BUDGET / bps;
    const LvSmemPlan none = lv_smem_plan(problem_bytes, 0, nd_max);
    const int64_t cap = none.total < budget ? (budget - none.total) / lv_bytes_per_chain(nd_max) : 0;
    g.cmax = cap < 1 ? 0 : (int)std::max<int64_t>(1, std::min<int64_t>(share, std::min<int64_t>(cap, LV_MAX_CMAX)));
    g.plan = cap < 1 ? none : lv_smem_plan(problem_bytes, g.cmax, nd_max);
    return g;
}

// ---------------------------------------------------------------------------------------------------------------------
// FP64 tensor path.  After the problem blob, one region per warp: the state tile [8][ks] doubles at 0; for a dense
// proposal factor the transpose buffer of L z [8][ks]; when shared memory allows, the Welford mean and second moment
// of the tile, 2 x [8][ks] doubles; the noise tile of the next proposal [8][big_zs(kq)] floats.
// ---------------------------------------------------------------------------------------------------------------------
constexpr uint32_t BIG_SMEM_BUDGET = 227 * 1024;   // the opt-in maximum of dynamic shared memory per block
constexpr int BIG_MIN_WARPS = 4;                    // a problem that leaves fewer is refused by yg_set_problem

constexpr int BIG_WARPS = 16;      // most warps per CTA (8 chains each, <= 128 registers per thread); fewer when shared memory is short
// d > 32 (KQ = 16): G of a 256-row model leaves shared memory for 13 warps; 12 are used -- three per sub-partition may
// take 168 registers each (a fourth warp on one sub-partition caps everybody at 128: the register file is per
// sub-partition), which the 64-parameter operand tiles need: no spills, 25.2 against 20.7 TFLOP/s with 13 x 128.
#ifndef YG_BIG_WARPS_KQ16
#define YG_BIG_WARPS_KQ16 12
#endif
__host__ __device__ constexpr int big_max_warps(int kq) { return kq == 16 ? YG_BIG_WARPS_KQ16 : BIG_WARPS; }
// floats per chain of the noise tile
__host__ __device__ constexpr int big_zs(int kq) { return 4 * kq + 4; }

struct BigSmemPlan {
    int warps;                  // warps per CTA: as many as fit, at most big_max_warps
    int wsm;                    // 1: the Welford tiles are in the warp regions (they cost no warp)
    uint32_t blob;              // bytes of the problem blob = offset of warp 0's region
    uint32_t stride;            // bytes per warp region
    uint32_t scr, wm, wv, zb;   // offsets in a warp region: transpose buffer, Welford mean, second moment, noise
    uint32_t total;             // bytes of the launch
};

// tail_len, ks, kq: DevBigHeader's (kq = kp / 4); welford: FullDiagnostics asked for the moments.
__host__ __device__ inline BigSmemPlan big_smem_plan(int tail_len, int ks, int kq, bool dense_L, bool welford)
{
    const uint32_t tile = sizeof(double) * 8 * ks, noise = sizeof(float) * 8 * big_zs(kq);
    BigSmemPlan p;
    p.blob = sizeof(double) * ((tail_len + 1) & ~1);
    p.scr = tile;
    p.wm = tile * (dense_L ? 2 : 1);
    p.wv = p.wm + tile;
    const uint32_t plain = p.wm + noise;
    const uint32_t fit = p.blob < BIG_SMEM_BUDGET ? (BIG_SMEM_BUDGET - p.blob) / plain : 0;
    p.warps = fit < (uint32_t)big_max_warps(kq) ? (int)fit : big_max_warps(kq);
    p.wsm = welford && p.warps >= BIG_MIN_WARPS && p.blob + p.warps * (plain + 2 * tile) <= BIG_SMEM_BUDGET;
    p.zb = p.wm + (p.wsm ? 2 * tile : 0);
    p.stride = p.zb + noise;
    p.total = p.blob + p.warps * p.stride;
    return p;
}

// Operands that the tensor path may leave in the global copy of the blob (read through L2 with ld.global.nc) when the
// whole blob leaves room for fewer than BIG_MIN_WARPS warps, in the order they are moved out: level 1's G, then level
// 2's G of three levels (each evaluated at most once per transition, only when the sub-chain moved; level 0 is evaluated
// J times), then the dense proposal factor (J times per transition, but only kp x ks).  With all of them out, every
// problem of the envelope (d <= 64, data_dim <= 256 per level, dense prior and factor, up to three levels) fits with
// BIG_MIN_WARPS warps or more (tests/test_tensor_path_streamed_cpu.py, tests/test_tensor_path_three_level_cpu.py), so
// level 0's G always stays in shared memory.  bd, pmean, pprec, propL and pcn_mean always stay there too.  Two levels
// stream only at d > 32; three levels of 256 data rows outgrow shared memory from d = 32 on, so three levels also
// stream at 16 < d <= 32.
enum BigStream { BIG_STREAM_G1 = 1, BIG_STREAM_LD = 2, BIG_STREAM_G2 = 4 };

struct BigTensorPlan {
    BigSmemPlan smem;   // the plan of the staged (resident) part of the blob
    int stream;         // BigStream bits of the operands read from global memory
    int resident;       // doubles of the tail staged into shared memory: a prefix of the tail
    int tail;           // doubles of the whole tail; the streamed operands follow the prefix, G1 before G2 before Ld
};

// Doubles of the tail of one level (G, b - mean, prior mean and precision) and of the shared part (diagonal factor,
// pCN mean, dense factor): abi.cu's build_big_blob.
__host__ __device__ constexpr int big_level_doubles(int np, int kp) { return np * (kp + 4) + np + 2 * kp; }
__host__ __device__ constexpr int big_shared_doubles(int kp, bool dense_L) { return 2 * kp + (dense_L ? kp * (kp + 4) : 0); }

// The plan of the tensor path.  np0, np1, np2: operand rows of levels 0, 1 and 2 (multiples of 16; np1 = 0 for one
// level, np2 = 0 for fewer than three).  Nothing is streamed while the whole blob leaves BIG_MIN_WARPS warps: the plan is
// then big_smem_plan of the whole blob.  Otherwise operands move out in BigStream's order until it does; the staged
// prefix is rounded up to 32 bytes, so every streamed operand starts on a whole sector (G rows and Ld rows are
// ks = 4 mod 16 doubles: 32-byte multiples).  With np2 = 0 the plan is the two-level one, field for field.
__host__ __device__ inline BigTensorPlan big_tensor_plan(int np0, int np1, int kq, bool dense_L, bool welford, int np2 = 0)
{
    const int kp = 4 * kq, ks = kp + 4;
    const int raw = big_level_doubles(np0, kp) + (np1 ? big_level_doubles(np1, kp) : 0) +
                    (np2 ? big_level_doubles(np2, kp) : 0) + big_shared_doubles(kp, dense_L);
    BigTensorPlan p;
    p.stream = 0;
    p.resident = p.tail = (raw + 1) & ~1;
    p.smem = big_smem_plan(p.resident, ks, kq, dense_L, welford);
    const int order[3] = {BIG_STREAM_G1, BIG_STREAM_G2, BIG_STREAM_LD};
    const int size[3] = {np1 * ks, np2 * ks, dense_L ? kp * ks : 0};
    int staged = raw;
#ifdef YG_STREAM_ALWAYS
    const int need = big_max_warps(kq) + 1;     // dev builds (measurement): stream every operand that can be streamed
#else
    const int need = BIG_MIN_WARPS;
#endif
    for (int i = 0; i < 3 && p.smem.warps < need; i++) {
        if (size[i] == 0) continue;
        p.stream |= order[i];
        staged -= size[i];
        p.resident = (staged + 3) & ~3;
        p.smem = big_smem_plan(p.resident, ks, kq, dense_L, welford);
    }
    if (p.stream) p.tail = p.resident + raw - staged;
    return p;
}

// ---------------------------------------------------------------------------------------------------------------------
// Warp-specialised generic kernel.  After the problem blob (rounded up to 16 bytes): the ring [WS_RING][3][32] doubles,
// WS_RING ready flags and the consumed counter (uint64).
// ---------------------------------------------------------------------------------------------------------------------
constexpr int WS_RING = 16;                // ring entries; one entry = (z0, z1, u) of one sub-step for 32 chains
constexpr uint32_t WS_RING_BYTES = sizeof(double) * WS_RING * 96 + sizeof(unsigned long long) * (WS_RING + 1);
