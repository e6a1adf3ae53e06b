"""Early rejection in the LV kernel: at level 0 the remaining integrations of a proposal are skipped once its partial
misfit sum passes the budget from reject_budget (common.cuh).  Skipping must change nothing but the work done.

CPU: the budget against accept_rule on near-ties (host build of common.cuh).
GPU: with skipping on and off, samples, accept flags, log-posteriors, chain state and counters are bit-identical."""
import numpy as np
import pytest
import torch

import bench_problems as bp
from golden_io import load
from support import ensemble, host_program

_NEAR_TIE_PROGRAM = r"""
#include "yagre_mcmc_b200/csrc/common.cuh"
#include <cstdio>

static uint64_t s = 0x9E3779B97F4A7C15ull;
static uint64_t next() { s += 0x9E3779B97F4A7C15ull; uint64_t z = s; z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
                         z = (z ^ (z >> 27)) * 0x94D049BB133111EBull; return z ^ (z >> 31); }
static double unif() { return (double)(next() >> 11) * 0x1.0p-53; }

int main()
{
    // edge cases: never skip
    const double inf = (double)INFINITY, nan = (double)NAN;
    const double edge[][4] = {{-1.0, -2.0, 0.0, 1.0}, {-1.0, -2.0, 0.5, 0.0}, {-1.0, -inf, 0.5, 1.0},
                              {-1.0, nan, 0.5, 1.0}, {-inf, -2.0, 0.5, 1.0}, {-1.0, -2.0, 0.5, -1.0},
                              {-1.0, -2.0, 0.5, inf}, {-1.0, inf, 0.5, 1.0}, {nan, -2.0, 0.5, 1.0}};
    int edge_bad = 0;
    for (const auto &e : edge) edge_bad += !(reject_budget(e[0], e[1], e[2], e[3]) == inf);

    long cases = 0, violations = 0, certified = 0, missed = 0;
    const double ts[] = {1.0, 0.5, 1e-3, 7.25, 0.1};
    const double scales[] = {1.0, 30.0, 1e4, 1e8};
    double q[128];
    int order[128];
    for (int it = 0; it < 400000; it++) {
        const int n = 1 + (int)(next() % 128);
        const double t = (it % 7 == 6) ? 0.05 + 10.0 * unif() : ts[it % 5];
        const double sc = scales[(it / 5) % 4];
        const double lp = -sc * unif();
        const double lps = lp - sc * (unif() - 0.3);
        const double u = (it % 11 == 0) ? 1e-300 * (1.0 + unif()) : (it % 13 == 0 ? 1.0 - 0x1.0p-53 : unif());
        if (!(u > 0.0)) continue;
        const double b = reject_budget(lp, lps, u, t);
        if (!(b < inf)) continue;
        const double thr = 2.0 * (lp - lps - log(u)) / t;        // the tie in exact arithmetic
        if (!(thr > 0.0)) continue;
        const int k = (int)(next() % 40);
        const double e = (k < 20 ? -1.0 : 1.0) * pow(10.0, -16.0 + 0.5 * (k % 20)) * unif();
        const double S = thr * (1.0 + e);
        double w = 0.0;
        for (int i = 0; i < n; i++) { q[i] = (i % 5 == 0) ? unif() * unif() * 40.0 : unif(); w += q[i]; order[i] = i; }
        for (int i = 0; i < n; i++) q[i] *= S / w;
        for (int i = n - 1; i > 0; i--) { const int j = (int)(next() % (i + 1)); const int x = order[i]; order[i] = order[j]; order[j] = x; }
        const double lpp = t * (-0.5 * np_sum_le128(q, n, 1)) + lp;   // log_post_from_q, lv_kernel.cu
        const bool acc = accept_rule(lpp - lps, u);
        double part = 0.0;
        bool skip = false;
        for (int i = 0; i < n; i++) { part += q[order[i]]; skip = skip || part > b; }
        cases++;
        violations += (skip && acc);
        certified += skip;
        const double m = fabs(lp) + fabs(lps) + fabs(log(u)) + 1.0;     // the margin is relative to these terms
        missed += (!skip && S > thr + 1e-8 * (2.0 * m / t + thr));
    }
    printf("%d %ld %ld %ld %ld\n", edge_bad, cases, violations, certified, missed);
    return 0;
}
"""


def test_reject_budget_never_certifies_an_accept(tmp_path):
    """Near-ties: sums within 1e-16 .. 1e-7 relative of the exact accept / reject boundary, q split over up to 128
    design points and summed in a random order.  A partial sum above the budget must never belong to a proposal that
    accept_rule accepts; beyond a few times the margin the budget must certify.  u == 0, t <= 0, non-finite t, lp or lps:
    no budget."""
    edge_bad, cases, violations, certified, missed = map(int, host_program(tmp_path, "near_tie", _NEAR_TIE_PROGRAM).split())
    assert edge_bad == 0
    assert cases > 200000
    assert violations == 0
    assert missed == 0
    assert certified > 0.05 * cases


# ------------------------------------------------------------------------------------------------------------------
# GPU: skipping on == skipping off
# ------------------------------------------------------------------------------------------------------------------
def _run(meta, arrays, th0, early_reject, ns, inject=None, **kw):
    ens = ensemble(meta, arrays, th0.shape[0], seed=77, early_reject=early_reject, **kw)
    ens.set_state(th0)
    if inject is None:
        ens.run(ns, samples=False)                 # a second launch continues with a learned order
    out = ens.run(ns, samples=True, accepted=True, logpost=True, inject=inject)
    torch.cuda.synchronize()
    st = ens.state()
    got = dict(samples=out["samples"].clone(), accepted=out["accepted"].clone(), logpost=out["logpost"].clone())
    got.update({k: st[k].clone() for k in ("theta", "logpost", "n_accept", "w_mean", "w_m2")})
    res = (got, ens.counters(), ens.skipped_evals())
    ens.close()
    return res


def _same(meta, arrays, th0, ns, inject=None, **kw):
    on, c_on, skipped = _run(meta, arrays, th0, True, ns, inject, **kw)
    off, c_off, none = _run(meta, arrays, th0, False, ns, inject, **kw)
    for k in on:
        assert torch.equal(on[k], off[k]), k
    assert c_on == c_off
    assert none == 0
    return skipped, c_on


@pytest.mark.gpu
def test_headline_identical_with_and_without_early_rejection():
    meta, arrays = bp.lv_problem(True)
    nc, ns = 65536, 10             # the bench size: small CTAs take a whole phase's units in their first grab
    skipped, c = _same(meta, arrays, bp.lv_initial_states(nc), ns)
    assert 0 < skipped < c["coarse_evals"] * meta["n_data"]


@pytest.mark.gpu
def test_single_level_identical_with_and_without_early_rejection():
    """C4: the fine integration is one work unit when rk4_segment covers it, and the commit decides from the budget."""
    meta, arrays = bp.lv_problem(False)
    skipped, _ = _same(meta, arrays, bp.lv_initial_states(65536), 4, rk4_segment=512)
    assert skipped > 0


@pytest.mark.gpu
def test_dense_noise_disables_early_rejection():
    """A dense noise precision can round q below zero: no skipping, same results."""
    meta, arrays = bp.lv_problem(True)
    dense = np.array([[25.0, 4.0], [4.0, 25.0]])
    arrays = dict(arrays, L0_noise_prec=dense, L1_noise_prec=dense)
    skipped, _ = _same(meta, arrays, bp.lv_initial_states(2048), 6)
    assert skipped == 0


@pytest.mark.gpu
def test_nonfinite_fixture_identical_with_and_without_early_rejection():
    """Chain 0 starts where RK4 overflows (logpost -inf): its proposals must never be skipped into a rejection."""
    meta, a = load("mlda_lv_nonfinite")
    inject = dict(z=np.ascontiguousarray(np.transpose(a["z"], (1, 2, 3, 0))),
                  u_c=np.ascontiguousarray(np.transpose(a["u_c"], (1, 2, 0))),
                  u_f=np.ascontiguousarray(np.transpose(a["u_f"], (1, 0))))
    ns = a["u_f"].shape[1]
    _, c = _same(meta, a, a["theta0"], ns, inject=inject)
    on, _, _ = _run(meta, a, a["theta0"], True, ns, inject)
    assert np.array_equal(on["accepted"].cpu().numpy().T, a["accepted"])
