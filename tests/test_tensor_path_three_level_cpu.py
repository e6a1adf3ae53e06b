"""CPU: MLDA with two surrogates and tempered levels on the tensor path.

  1. The plan with a third level (smem_plan.h: big_tensor_plan, np2 > 0), swept over d 1 .. 64 and every operand-row
     count of each level up to 256 + d (data_dim + d for a dense prior; the levels may differ), dense or diagonal
     factor, Welford tiles asked for or not: no refusal, at least 4 warps, the staged prefix and the streamed operands
     tile the tail without overlap on 32-byte boundaries, the warp regions are aligned and inside 227 KiB, operands
     leave in the order level 1's G, level 2's G, dense factor and only as far as needed.  With np2 = 0 the plan is the
     two-level call's, field for field.
  2. The law the two-surrogate recursion leaves invariant, mu ~ pi_2 pi_0 / pi_1 (three_level_reference.mlda_invariant_gaussian):
     on the 2-D Gaussian hierarchy whose covariance the unmodified reference pins, and at a tensor-sized linear
     hierarchy with a tempered level, through the C oracle.
  3. The tempered tensor-path bound (three_level_reference.tensor_logpost_and_bound) holds for a double-precision
     emulation of the folded evaluation and is broken by three wrong foldings; at t = 1 it is logpost_reference's."""
import numpy as np
import pytest

import bench_problems as bp
import logpost_reference as R
from support import check_closed_form, host_program, three_level_gauss
from three_level_reference import mlda_invariant_gaussian, tensor_logpost_bound

_PROGRAM = r"""
#include "yagre_mcmc_b200/csrc/common.cuh"
#include "yagre_mcmc_b200/csrc/smem_plan.h"
#include <algorithm>
#include <cstdio>
#include <cstring>
#include <vector>

struct Region { long long off, bytes, align; };
static long long overlap = 0, misaligned = 0, outside = 0, over = 0, wrong = 0, order = 0, refused = 0, two = 0;
static long long cases = 0, streamed = 0, kq8 = 0;
static long long by_bits[8] = {0};

static void check(std::vector<Region> r, long long total)
{
    std::sort(r.begin(), r.end(), [](const Region &a, const Region &b) { return a.off < b.off; });
    for (size_t i = 0; i < r.size(); i++) {
        misaligned += r[i].off % r[i].align != 0;
        outside += r[i].off < 0 || r[i].off + r[i].bytes > total;
        if (i) overlap += r[i - 1].off + r[i - 1].bytes > r[i].off;
    }
}

static void one(int d, int np0, int np1, int np2, bool dense, bool welford)
{
    const int kp = d <= 16 ? 16 : (d <= 32 ? 32 : 64), ks = kp + 4, kq = kp / 4;
    long long raw = 2 * kp + (dense ? kp * ks : 0);
    for (int np : {np0, np1, np2}) raw += (long long)np * (ks + 1) + 2 * kp;
    const long long tail = (raw + 1) & ~1ll;
    const BigSmemPlan whole = big_smem_plan((int)tail, ks, kq, dense, welford);
    const BigTensorPlan p = big_tensor_plan(np0, np1, kq, dense, welford, np2);
    cases++;
    if (whole.warps >= BIG_MIN_WARPS) {
        wrong += memcmp(&whole, &p.smem, sizeof whole) != 0 || p.stream != 0 || p.resident != tail || p.tail != tail;
        return;
    }
    streamed++;
    kq8 += kq == 8;
    if (p.smem.warps < BIG_MIN_WARPS) { refused++; return; }
    by_bits[p.stream & 7]++;
    // the order: G1, G2, Ld, each only when what went before was not enough
    const long long size[3] = {(long long)np1 * ks, (long long)np2 * ks, dense ? (long long)kp * ks : 0};
    const int bit[3] = {BIG_STREAM_G1, BIG_STREAM_G2, BIG_STREAM_LD};
    long long staged = raw;
    int last = -1;
    for (int i = 0; i < 3; i++)
        if (p.stream & bit[i]) { staged -= size[i]; last = i; }
    for (int i = 0; i < last; i++) order += !(p.stream & bit[i]) && size[i] != 0;     // an earlier one skipped
    if (last > 0) {        // without the last one moved, fewer than BIG_MIN_WARPS warps
        const long long res = ((staged + size[last]) + 3) & ~3ll;
        order += big_smem_plan((int)res, ks, kq, dense, false).warps >= BIG_MIN_WARPS;
    }
    order += (p.stream & ~(BIG_STREAM_G1 | BIG_STREAM_G2 | BIG_STREAM_LD)) != 0 || (!dense && (p.stream & BIG_STREAM_LD));
    long long at = p.resident;
    std::vector<Region> t = {{0, 8 * staged, 32}};
    for (int i = 0; i < 3; i++)
        if (p.stream & bit[i]) { t.push_back({8 * at, 8 * size[i], 32}); at += size[i]; }
    wrong += p.resident % 4 != 0 || p.resident < staged || p.resident - staged > 3 || at != p.tail;
    check(t, 8LL * p.tail);
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

static void two_level(int d, int np0, int np1, bool dense, bool welford)
{
    const int kq = (d <= 16 ? 16 : (d <= 32 ? 32 : 64)) / 4;
    const BigTensorPlan a = big_tensor_plan(np0, np1, kq, dense, welford);
    const BigTensorPlan b = big_tensor_plan(np0, np1, kq, dense, welford, 0);
    two += memcmp(&a.smem, &b.smem, sizeof a.smem) != 0 || a.stream != b.stream || a.resident != b.resident ||
           a.tail != b.tail;
}

static void show(const char *name, int d, int np0, int np1, int np2, bool dense)
{
    const int kq = (d <= 16 ? 16 : (d <= 32 ? 32 : 64)) / 4;
    const BigTensorPlan p = big_tensor_plan(np0, np1, kq, dense, true, np2);
    printf("%s %d %d %d %d %d %u\n", name, p.stream, p.resident, p.tail, p.smem.warps, p.smem.wsm, p.smem.total);
}

int main()
{
    for (int d = 1; d <= 64; d++)
    for (int dense = 0; dense <= 1; dense++)
    for (int welford = 0; welford <= 1; welford++) {
        const int top = (256 + d + 15) & ~15;          // the plan sees rows rounded up to 16 only
        for (int n0 = 16; n0 <= top; n0 += 16)
        for (int n1 = 16; n1 <= top; n1 += 16) {
            two_level(d, n0, n1, dense, welford);
            for (int n2 = 16; n2 <= top; n2 += 16) one(d, n0, n1, n2, dense, welford);
        }
    }
    printf("%lld %lld %lld %lld %lld %lld %lld %lld %lld %lld\n", cases, streamed, kq8, by_bits[1], by_bits[3],
           by_bits[5], by_bits[7], by_bits[4], by_bits[6], by_bits[2]);
    printf("%lld %lld %lld %lld %lld %lld %lld %lld\n", overlap, misaligned, outside, over, wrong, order, refused, two);
    show("three_64x256", 64, 256, 256, 256, false);
    show("three_64x256_dense_prior_dense_factor", 64, 320, 320, 320, true);
    show("three_32x96_dense_prior", 32, 128, 128, 128, false);
    show("three_32x256", 32, 256, 256, 256, false);
    show("three_48_40_97_256", 48, 48, 112, 256, false);
    return 0;
}
"""


def test_three_level_plans(tmp_path):
    lines = host_program(tmp_path, "three_level_plan", _PROGRAM).splitlines()
    cases, streamed, kq8, g1, g1_ld, g1_g2, all3, g2, g2_ld, ld = map(int, lines[0].split())
    assert cases > 1000000 and streamed > 100000 and kq8 > 0
    # every streamed shape moves G1 first; G2 and the factor follow only when needed; some need all three out
    assert g1 > 0 and g1_g2 > 0 and all3 > 0 and g2 == g2_ld == ld == 0
    assert g1 + g1_ld + g1_g2 + all3 == streamed
    # overlap, misaligned, outside, over budget, wrong, order, refused, two-level call != np2 = 0
    assert list(map(int, lines[1].split())) == [0] * 8
    plans = {f[0]: list(map(int, f[1:])) for f in (ln.split() for ln in lines[2:])}
    # name: stream bits (1 = level 1's G, 4 = level 2's G, 2 = dense factor), staged doubles, tail doubles, warps, wsm,
    # launch bytes
    assert plans == {
        "three_64x256": [5, 18688, 53504, 12, 0, 227840],
        "three_64x256_dense_prior_dense_factor": [7, 23232, 71104, 4, 0, 229376],     # the worst case: all three out
        "three_32x96_dense_prior": [0, 14464, 14464, 16, 0, 171008],
        "three_32x256": [1, 19456, 28672, 16, 0, 210944],
        "three_48_40_97_256": [1, 21600, 29216, 9, 0, 231552],
    }


# ------------------------------------------------------------------------------------------------------------------
# the invariant law of MLDA with two surrogates
# ------------------------------------------------------------------------------------------------------------------
def test_invariant_law_of_the_gaussian_hierarchy():
    """support.three_level_gauss: the formula gives what the unmodified reference's long runs give (the covariance
    test_round2_gpu pins, [[3.86, -0.86], [-0.86, 1.00]])."""
    meta, arrays = three_level_gauss()
    _, cov, _ = mlda_invariant_gaussian(arrays, 3)
    np.testing.assert_allclose(cov, [[3.859, -0.861], [-0.861, 0.994]], atol=1e-3)
    np.testing.assert_allclose(cov, [[3.86, -0.86], [-0.86, 1.00]], atol=0.01)


def test_invariant_law_through_the_oracle():
    """d = 12, data_dims 20 / 24 / 30, level 0 tempered at 0.6: the C oracle on numpy noise, chains started from exact
    draws of mu, keeps mu's mean and covariance -- and not the target's."""
    from oracle import cport
    meta, arrays = bp.big_linear_three_level_problem(12, (20, 24, 30), 2, J=3, tempering={0: 0.6}, seed=31)
    mean, cov, A = mlda_invariant_gaussian(arrays, 3)
    assert np.linalg.eigvalsh(A).min() > 0.0
    C, ns = 2048, 60
    rng = np.random.default_rng(5)
    th0 = rng.multivariate_normal(mean, cov, size=C)
    z = rng.standard_normal((C, ns, 3, 12))
    u_c, u_f = rng.random((C, ns, 3)), rng.random((C, ns))
    ref = cport.run_injected(cport.Problem(meta, arrays), th0, z, u_c, u_f)
    x = ref["traj"][:, 1:].reshape(-1, 12)
    check_closed_form(dict(mean=x.mean(0), covariance=np.cov(x.T)), mean, cov, C, "oracle mu")
    assert 0.2 < ref["accepted"].mean() < 0.95
    tmean, tcov = bp.linear_gaussian_posterior(arrays, 2)
    sm = np.sqrt(np.diag(tcov) / C)
    assert np.abs(x.mean(0) - tmean).max() > 10 * sm.max() or np.abs(cov - tcov).max() > 0.2 * np.abs(tcov).max()


def test_invariant_law_generator_shapes_are_positive_definite():
    """Every three-level shape of the GPU tests has a proper mu."""
    for d, dims, kw in ((9, (20, 20, 20), dict(tempering={0: 0.5})), (23, (45, 45, 45), {}),
                        (32, (96, 96, 96), dict(dense_prior=True)), (48, (40, 97, 256), {}), (64, (256, 256, 256), {}),
                        (64, (256, 256, 256), dict(dense_prior=True)), (32, (256, 256, 256), {})):
        _, arrays = bp.big_linear_three_level_problem(d, dims, 1, **kw)
        assert np.linalg.eigvalsh(mlda_invariant_gaussian(arrays, 3)[2]).min() > 0.0, (d, dims)


# ------------------------------------------------------------------------------------------------------------------
# the tempered tensor-path bound
# ------------------------------------------------------------------------------------------------------------------
def _folded(arrays, level, theta, fold="right"):
    """The tensor path's evaluation in double (abi.cu's host fold, then the kernel's sum).  fold: "right", or a wrong
    one: "untempered" (t not applied), "prior" (t applied to the dense prior's rows as well), "twice" (sqrt(t)
    folded twice)."""
    pre = f"L{level}_"
    t = float(np.asarray(arrays.get(pre + "tempering", 1.0)))
    G, b, data = arrays[pre + "G"], arrays[pre + "b"], arrays[pre + "data"]
    prec = np.diag(arrays[pre + "noise_prec"])
    n = data.shape[0]
    st = {"right": np.sqrt(t), "untempered": 1.0, "prior": np.sqrt(t), "twice": np.sqrt(t) * np.sqrt(t)}[fold]
    tq = 1.0 if fold == "untempered" else t
    mean = data.sum(axis=0) / n
    sw = st * np.sqrt(n * prec)
    rows = sw[:, None] * G
    bd = sw * (b - mean)
    q_const = tq * float((prec * ((data - mean) ** 2).sum(axis=0)).sum())
    P0, m0 = arrays[pre + "prior_prec"], arrays[pre + "prior_mean"]
    R_ = np.linalg.cholesky(0.5 * (P0 + P0.T)).T
    sp = np.sqrt(t) if fold == "prior" else 1.0
    rows = np.vstack([rows, sp * R_])
    bd = np.concatenate([bd, -(sp * R_) @ m0])
    e = theta @ rows.T + bd
    return -0.5 * ((e * e).sum(axis=1) + q_const)


@pytest.mark.parametrize("t", [0.5, 0.0, 0.93])
def test_tempered_tensor_bound(t):
    meta, arrays = bp.big_linear_three_level_problem(24, (40, 48, 56), 3, tempering={1: t}, dense_prior=True, seed=9)
    mean, cov, _ = mlda_invariant_gaussian(dict(arrays, L1_tempering=np.array(1.0)), 3)
    theta = np.random.default_rng(2).multivariate_normal(mean, 4.0 * cov, size=200)
    lp, bound = tensor_logpost_bound(meta, arrays, 1, theta)
    err = np.abs(_folded(arrays, 1, theta).astype(np.longdouble) - lp).astype(np.float64)
    assert np.all(err <= bound), float((err / bound).max())
    assert np.all(bound < 1e-9 * np.abs(np.asarray(lp, dtype=np.float64)) + 1e-9)
    wrong = ("untempered", "twice", "prior") if 0.0 < t < 1.0 else ("untempered", "prior")
    for fold in wrong:
        err = np.abs(_folded(arrays, 1, theta, fold).astype(np.longdouble) - lp).astype(np.float64)
        assert np.mean(err > bound) > 0.9, fold


def test_untempered_tensor_bound_unchanged():
    """A level with tempering 1 gets the untempered bound, term for term."""
    meta, arrays = bp.big_linear_three_level_problem(24, (40, 48, 56), 3, dense_prior=True, seed=9)
    theta = np.random.default_rng(2).standard_normal((50, 24))
    lp, b = R.logpost_bound(meta, arrays, 2, theta, path="tensor")
    lp1, b1 = tensor_logpost_bound(meta, dict(arrays, L2_tempering=np.array(1.0)), 2, theta)
    assert np.array_equal(lp, lp1) and np.array_equal(b, b1)
    err = np.abs(_folded(arrays, 2, theta).astype(np.longdouble) - lp).astype(np.float64)
    assert np.all(err <= b)
