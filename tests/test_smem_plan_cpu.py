"""CPU: the shared-memory plans of smem_plan.h (host build of the header), swept over the shapes the kernels accept.

LV kernel: one and two levels, n_data 1 .. 300, blocks_per_sm 1 .. 4, 1 .. 524,288 chains.  Tensor path: d 1 .. 64,
up to 320 operand rows per level on one or two levels, dense or diagonal proposal factor, Welford tiles asked for or not.
Every region is aligned for its element type (the blob end at 16 bytes), lies inside the launch's bytes and overlaps no
other; the launch stays within 227 KiB, the LV kernel within its 220 KiB / blocks_per_sm budget up to the rounding that
its cap formula ignores; the tensor path refuses a problem exactly when four warps do not fit."""
from support import host_program

# The LV cap divides the budget by the unpadded bytes per chain.  Rounding the end of the int arrays up to 16 bytes
# adds at most 12 bytes (every region before it is a multiple of 4 bytes), padding evald to 16 bytes at most 15.
LV_ROUNDING_SLACK = 12 + 15

_PROGRAM = r"""
#include "yagre_mcmc_b200/csrc/common.cuh"
#include "yagre_mcmc_b200/csrc/smem_plan.h"
#include <algorithm>
#include <cstdio>
#include <cstring>
#include <vector>

struct Region { long long off, bytes, align; };
static long long overlap = 0, misaligned = 0, outside = 0, over = 0, wrong = 0;

static void check(std::vector<Region> r, long long total)
{
    std::sort(r.begin(), r.end(), [](const Region &a, const Region &b) { return a.off < b.off; });
    for (size_t i = 0; i < r.size(); i++) {
        misaligned += r[i].off % r[i].align != 0;
        outside += r[i].off < 0 || r[i].off + r[i].bytes > total;
        if (i) overlap += r[i - 1].off + r[i - 1].bytes > r[i].off;
    }
}

int main()
{
    const long long KiB = 1024, slack = SLACK;
    // ---- LV kernel: the problem blob holds data [n][2] and design [n][2] per level after the header ----
    const long long chains[] = {1, 2, 3, 31, 147, 148, 149, 443, 1000, 4095, 16384, 65535, 65536, 65537, 100003,
                                151552, 151553, 262144, 524287, 524288};
    long long lv_cases = 0;
    for (int levels = 1; levels <= 2; levels++)
    for (int N = 1; N <= 300; N++)
    for (int bps = 1; bps <= 4; bps++)
    for (long long n : chains) {
        const uint32_t pb = sizeof(DevProblemHeader) + 8u * levels * 4 * N;
        const LvGeometry g = lv_geometry(pb, N, n, 148, bps, 0);
        lv_cases++;
        if (g.cmax == 0) { wrong++; continue; }         // every blob of the sweep leaves room for chains
        const LvSmemPlan p = g.plan, q = lv_smem_plan(pb, g.cmax, N);
        wrong += memcmp(&p, &q, sizeof p) != 0 || p.cmax != g.cmax || p.nd_max != N || g.cmax > 1024 ||
                 g.cmax > (n + g.grid - 1) / g.grid || g.grid < 1 || g.grid > 148 * bps;
        const long long C = g.cmax;
        check({{0, pb, 16}, {p.off[LV_CHAIN], 8 * LvSlot::NDBL * C, 16}, {p.off[LV_Q], 8 * N * C, 8},
               {p.off[LV_SX], 8 * N * C, 8}, {p.off[LV_SY], 8 * N * C, 8}, {p.off[LV_NZ], 8 * 4 * C, 8},
               {p.off[LV_QMAX], 8 * C, 8}, {p.off[LV_QPART], 8 * C, 8}, {p.off[LV_QSUM], 8 * N, 8},
               {p.off[LV_NACC], 8 * C, 8}, {p.off[LV_LIST0], 4 * 2 * C, 4}, {p.off[LV_SEGDONE], 4 * N * C, 4},
               {p.off[LV_PERM], 4 * N, 4}, {p.off[LV_EVALD], C, 1}, {p.mbar, 8, 8}, {p.nact, 4 * 2, 4},
               {p.blk_cnt, 8 * 6, 8}, {p.qhead, 4, 4}}, p.total);
        over += p.total > 227 * KiB || p.total > 220 * KiB / bps + slack;
    }
    // the geometry of three benchmark configurations: LV two-level with 10 design points at 65,536 and 524,288 chains,
    // and with 256 design points at 16,384 chains
    const LvGeometry h = lv_geometry(sizeof(DevProblemHeader) + 8 * 80, 10, 65536, 148, 0, 0);
    const LvGeometry c5 = lv_geometry(sizeof(DevProblemHeader) + 8 * 80, 10, 524288, 148, 0, 0);
    const LvGeometry l = lv_geometry(sizeof(DevProblemHeader) + 8 * 2048, 256, 16384, 148, 0, 0);

    // ---- tensor path: abi.cu's tail per level (G, b - mean, prior mean and precision), proposal factor, pCN mean ----
    long long t_cases = 0, t_refused = 0, refusal = 0;
    for (int d = 1; d <= 64; d++)
    for (int dense = 0; dense <= 1; dense++)
    for (int welford = 0; welford <= 1; welford++)
    for (int r0 = 1; r0 <= 320; r0++)
    for (int r1 = 0; r1 <= 320; r1 += (r1 == 0 ? 1 : 7)) {
        if (r1 > 0 && r0 % 7 != 3) continue;        // two levels on a coarser grid
        const int kp = d <= 16 ? 16 : (d <= 32 ? 32 : 64), ks = kp + 4, kq = kp / 4;
        long long tail = 2 * kp + (dense ? kp * ks : 0);
        for (int r : {r0, r1})
            if (r > 0) tail += ((r + 15) & ~15) * (long long)(ks + 1) + 2 * kp;
        tail = (tail + 1) & ~1ll;
        const BigSmemPlan p = big_smem_plan((int)tail, ks, kq, dense, welford);
        const long long tile = 8 * 8 * ks, noise = 4 * 8 * (4 * kq + 4), blob = 8 * tail;
        const bool fits = blob + 4 * (tile * (1 + dense) + noise) <= 227 * KiB;
        t_cases++;
        refusal += (p.warps < 4) != !fits;
        if (p.warps < 4) { t_refused++; continue; }
        wrong += p.blob != blob || p.warps > (kq == 16 ? 12 : 16) || (p.wsm && !welford) ||
                 p.total != p.blob + (long long)p.warps * p.stride;
        std::vector<Region> r = {{0, blob, 16}};
        for (int w = 0; w < p.warps; w++) {
            const long long base = p.blob + (long long)w * p.stride;
            r.push_back({base, tile, 8});
            if (dense) r.push_back({base + p.scr, tile, 8});
            if (p.wsm) { r.push_back({base + p.wm, tile, 8}); r.push_back({base + p.wv, tile, 8}); }
            r.push_back({base + p.zb, noise, 8});          // float2 stores
        }
        check(r, p.total);
        over += p.total > 227 * KiB;
    }
    // blob + 4 warps between 226 and 227 KiB: d = 64, two levels of 176 and 192 rows
    const BigSmemPlan w = big_smem_plan(25776, 68, 16, false, true);

    printf("%lld %lld %lld %lld %lld %lld %lld %lld %lld\n", lv_cases, t_cases, t_refused,
           overlap, misaligned, outside, over, wrong, refusal);
    printf("%d %u %d %u %d %u\n", h.cmax, h.plan.total, c5.cmax, c5.plan.total, l.cmax, l.plan.total);
    printf("%u %d %u\n", w.blob, w.warps, w.total);
    return 0;
}
"""


def test_shared_memory_plans(tmp_path):
    lines = host_program(tmp_path, "smem_plan", _PROGRAM.replace("SLACK", str(LV_ROUNDING_SLACK))).splitlines()
    lv_cases, t_cases, t_refused, overlap, misaligned, outside, over, wrong, refusal = map(int, lines[0].split())
    assert lv_cases == 2 * 300 * 4 * 20
    assert t_cases > 100000 and 0 < t_refused < t_cases
    assert (overlap, misaligned, outside, over, wrong, refusal) == (0, 0, 0, 0, 0, 0)
    # headline: limited by the chains per CTA; C5 at 524,288 chains and 256 design points: limited by the budget
    assert list(map(int, lines[1].split())) == [443, 221520, 450, 224896, 26, 218720]
    assert list(map(int, lines[2].split())) == [206208, 4, 232320]
