"""CPU: the tensor path's plan with streamed operands (smem_plan.h: big_tensor_plan), host build of the header.

Swept over d 1 .. 64, one and two levels with up to 256 + d operand rows each (data_dim + d for a dense prior), dense or
diagonal proposal factor, Welford tiles asked for or not:
  (a) wherever the whole blob leaves BIG_MIN_WARPS (4) warps, the plan IS big_smem_plan of the whole blob, field for
      field, and streams nothing;
  (b) elsewhere it streams level 1's G first, then the dense factor, only as far as needed; the staged prefix and the
      streamed operands tile the tail without overlap, on 32-byte boundaries; the warp regions are aligned and inside
      227 KiB; it has at least 4 warps;
  (c) no shape of the envelope is refused.
And the plans of the shapes profiles/streamed_operand.md measures."""
from support import host_program

_PROGRAM = r"""
#include "yagre_mcmc_b200/csrc/common.cuh"
#include "yagre_mcmc_b200/csrc/smem_plan.h"
#include <algorithm>
#include <cstdio>
#include <cstring>
#include <vector>

struct Region { long long off, bytes, align; };
static long long overlap = 0, misaligned = 0, outside = 0, over = 0, wrong = 0, order = 0, refused = 0;
static long long cases = 0, streamed = 0, s_g1 = 0, s_ld = 0, s_both = 0;

static void check(std::vector<Region> r, long long total)
{
    std::sort(r.begin(), r.end(), [](const Region &a, const Region &b) { return a.off < b.off; });
    for (size_t i = 0; i < r.size(); i++) {
        misaligned += r[i].off % r[i].align != 0;
        outside += r[i].off < 0 || r[i].off + r[i].bytes > total;
        if (i) overlap += r[i - 1].off + r[i - 1].bytes > r[i].off;
    }
}

static void one(int d, int r0, int r1, bool dense, bool welford)
{
    const int kp = d <= 16 ? 16 : (d <= 32 ? 32 : 64), ks = kp + 4, kq = kp / 4;
    const int np0 = (r0 + 15) & ~15, np1 = r1 ? (r1 + 15) & ~15 : 0;
    long long raw = 2 * kp + (dense ? kp * ks : 0);
    for (int np : {np0, np1})
        if (np) raw += (long long)np * (ks + 1) + 2 * kp;
    const long long tail = (raw + 1) & ~1ll;
    const BigSmemPlan whole = big_smem_plan((int)tail, ks, kq, dense, welford);
    const BigTensorPlan p = big_tensor_plan(np0, np1, kq, dense, welford);
    cases++;
    if (whole.warps >= BIG_MIN_WARPS) {                                   // (a)
        wrong += memcmp(&whole, &p.smem, sizeof whole) != 0 || p.stream != 0 || p.resident != tail || p.tail != tail;
        return;
    }
    streamed++;
    if (p.smem.warps < BIG_MIN_WARPS) { refused++; return; }             // (c)
    // (b) the order: level 1's G first (two levels), then the dense factor, and only as far as needed
    const long long g1 = (long long)np1 * ks, ld = dense ? (long long)kp * ks : 0;
    const int first = np1 ? BIG_STREAM_G1 : BIG_STREAM_LD;
    order += !(p.stream & first) || (p.stream & ~(BIG_STREAM_G1 | BIG_STREAM_LD)) || (!dense && (p.stream & BIG_STREAM_LD)) ||
             (!np1 && (p.stream & BIG_STREAM_G1));
    if (p.stream == (BIG_STREAM_G1 | BIG_STREAM_LD)) {                   // the factor went only because G1 was not enough
        const long long res = ((raw - g1) + 3) & ~3ll;
        order += big_smem_plan((int)res, ks, kq, dense, false).warps >= BIG_MIN_WARPS;
        s_both++;
    } else if (p.stream == BIG_STREAM_G1) s_g1++;
    else s_ld++;
    // the tail: staged prefix, then G1, then Ld, each streamed one on a 32-byte boundary
    long long staged = raw, at = p.resident;
    std::vector<Region> t = {};
    if (p.stream & BIG_STREAM_G1) { staged -= g1; t.push_back({8 * at, 8 * g1, 32}); at += g1; }
    if (p.stream & BIG_STREAM_LD) { staged -= ld; t.push_back({8 * at, 8 * ld, 32}); at += ld; }
    wrong += p.resident % 4 != 0 || p.resident < staged || p.resident - staged > 3 || at != p.tail;
    t.push_back({0, 8 * staged, 32});
    check(t, 8LL * p.tail);
    // shared memory: the staged prefix, then the warp regions
    const BigSmemPlan &s = p.smem;
    const long long tile = 8 * 8 * ks, noise = 4 * 8 * (4 * kq + 4);
    wrong += s.blob != 8ull * p.resident || s.warps > big_max_warps(kq) || (s.wsm && !welford) ||
             s.total != s.blob + (long long)s.warps * s.stride;
    std::vector<Region> r = {{0, (long long)s.blob, 16}};
    for (int w = 0; w < s.warps; w++) {
        const long long base = s.blob + (long long)w * s.stride;
        r.push_back({base, tile, 8});
        if (dense) r.push_back({base + s.scr, tile, 8});
        if (s.wsm) { r.push_back({base + s.wm, tile, 8}); r.push_back({base + s.wv, tile, 8}); }
        r.push_back({base + s.zb, noise, 8});
    }
    check(r, s.total);
    over += s.total > 227 * 1024;
}

static void show(const char *name, int np0, int np1, bool dense)
{
    const BigTensorPlan p = big_tensor_plan(np0, np1, 16, dense, true);
    printf("%s %d %d %d %d %d %u\n", name, p.stream, p.resident, p.tail, p.smem.warps, p.smem.wsm, p.smem.total);
}

int main()
{
    for (int d = 1; d <= 64; d++)
    for (int dense = 0; dense <= 1; dense++)
    for (int welford = 0; welford <= 1; welford++) {
        for (int r0 = 1; r0 <= 256 + d; r0++) one(d, r0, 0, dense, welford);
        for (int r0 = 1; r0 <= 256 + d; r0 += (r0 % 16 == 0 ? 1 : 15))         // 1, 16, 17, 32, 33, ...: every np
            for (int r1 = 1; r1 <= 256 + d; r1 += (r1 % 16 == 0 ? 1 : 15)) one(d, r0, r1, dense, welford);
        for (int r = 241; r <= 256 + d; r++) one(d, r, r, dense, welford);       // the largest two-level shapes densely
    }
    printf("%lld %lld %lld %lld %lld\n", cases, streamed, s_g1, s_ld, s_both);
    printf("%lld %lld %lld %lld %lld %lld %lld\n", overlap, misaligned, outside, over, wrong, order, refused);
    // the measured shapes (d = 64: np = rows rounded up to 16)
    show("two_64x256", 256, 256, false);
    show("two_64x256_dense_factor", 256, 256, true);
    show("two_64x176", 176, 176, false);
    show("two_64x192", 192, 192, false);
    show("single_64x256_dense_prior_dense_factor", 320, 0, true);
    show("two_64x160_dense_factor", 160, 160, true);
    return 0;
}
"""


def test_streamed_operand_plans(tmp_path):
    lines = host_program(tmp_path, "streamed_plan", _PROGRAM).splitlines()
    cases, streamed, s_g1, s_ld, s_both = map(int, lines[0].split())
    assert cases > 400000 and streamed > 1000
    assert s_g1 > 0 and s_ld > 0 and s_both > 0 and s_g1 + s_ld + s_both == streamed
    assert list(map(int, lines[1].split())) == [0] * 7
    plans = {f[0]: list(map(int, f[1:])) for f in (ln.split() for ln in lines[2:])}
    # name: stream bits (1 = level 1's G, 2 = dense factor), staged doubles, tail doubles, warps, wsm, launch bytes
    assert plans == {
        "two_64x256": [1, 18304, 35712, 12, 0, 224768],
        "two_64x256_dense_factor": [1, 22656, 40064, 4, 0, 224768],
        "two_64x176": [0, 24672, 24672, 5, 0, 230016],               # today's largest resident two-level shape
        "two_64x192": [1, 13824, 26880, 12, 0, 188928],
        "single_64x256_dense_prior_dense_factor": [2, 22336, 26688, 4, 0, 222208],
        "two_64x160_dense_factor": [1, 15936, 26816, 9, 0, 225408],
    }
