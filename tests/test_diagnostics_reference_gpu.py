"""GPU: every step kernel's chain diagnostics against a high-precision reference of the run that produced them.

Each case runs twice with the same seed: in record mode (the plain / recording kernel instances) and with Philox noise
only (the production instances: the warp-specialised kernel where eligible, FREE_NOISE on the tensor path).  The two
runs must agree bit for bit; the Welford moments (w_mean, w_m2, welford_n) must be those of the pre-transition states
within tests/diag_reference.py's bounds; n_accept, the ensemble counters and coarse_accepted must equal the oracle's
replay of the recorded noise exactly; and where yg_pooled_stats exists (d <= 8), its vector must be the long-double
sums of the state and moments_from_stats the long-double moments of all pre-states."""
import numpy as np
import pytest
import torch

import bench_problems as bp
from diag_reference import welford_reference, welford_tolerance
from golden_io import load
from support import check_case, lv_tempered, three_level_gauss

pytestmark = pytest.mark.gpu


# ------------------------------------------------------------------------------------------
# the LV kernel
# ------------------------------------------------------------------------------------------
LV_CASES = {
    # name: (problem, chains, plan, adaptive)
    "headline": (lambda: bp.lv_problem(True), 65536, [("run", 3)], None),
    "single_level": (lambda: bp.lv_problem(False), 3000, [("run", 6)], None),
    "adaptive_coarse": (lambda: bp.lv_problem(True), 700, [("run", 8)], dict(idle=1, collection=3, eps=1e-6, refresh=2)),
    "pcn": (lambda: bp.lv_pcn_problem(), 1000, [("run", 8)], None),
    "tempered_level0": (lv_tempered, 500, [("run", 6)], None),
    "300_design_points": (lambda: bp.lv_problem(True, n_data=300, Nc=4, Nf=12, prop_var=2e-4), 97, [("run", 6)], None),
    "one_chain": (lambda: bp.lv_problem(True, Nc=16, Nf=48), 1, [("run", 25)], None),
    "whole_c5_ensemble": (lambda: bp.lv_problem(True), 524288, [("run", 2)], None),
}


@pytest.mark.parametrize("name", sorted(LV_CASES))
def test_lv_kernel_diagnostics(name):
    """The LV kernel's Welford update (full 2 x 2 co-moment in the owners' phase) and its coarse-accept count.  The
    whole C5 ensemble makes every CTA walk several chunks and the pooled reduction's stage 1 stride over chains."""
    make, nc, plan, ad = LV_CASES[name]
    meta, arrays = make()
    check_case(meta, arrays, bp.lv_initial_states(nc), plan, seed=17, adaptive=ad, label=name)


def test_lv_headline_without_early_rejection():
    """The same counts and moments when every coarse integration runs (early rejection decides which path updates a
    rejected proposal's state and counters)."""
    meta, arrays = bp.lv_problem(True)
    c = check_case(meta, arrays, bp.lv_initial_states(65536), [("run", 3)], seed=17, early_reject=False,
                   label="headline, early rejection off")
    assert c["coarse_accepted"] > 0


# ------------------------------------------------------------------------------------------
# the one-chain-per-thread kernels
# ------------------------------------------------------------------------------------------
SMALL_SHAPES = [(d, dd) for d in (1, 2, 3, 5, 8) for dd in (2, 4, 8)]


@pytest.mark.parametrize("k", range(len(SMALL_SHAPES)))
def test_one_chain_per_thread_kernel_diagnostics_every_capacity(k):
    """d in {1, 2, 3, 5, 8} x data_dim in {2, 4, 8} (every capacity class of both), one and two levels in turn, 1, 33
    and 4,097 chains in turn: the full d x d co-moment of the per-thread Welford update."""
    d, dd = SMALL_SHAPES[k]
    two = k % 2 == 1
    nc = (1, 33, 4097)[k % 3]
    meta, arrays = bp.big_linear_problem(d, dd, 2, two_level=two, J=3, seed=40 + k)
    th0 = 0.1 * np.random.default_rng(k).standard_normal((nc, d))
    check_case(meta, arrays, th0, [("run", 12)], seed=5 + k, ws=d <= 2, label=f"d={d} data_dim={dd} two={two} nc={nc}")


def _fixture_problem(name):
    meta, a = load(name)
    return meta, {k: v for k, v in a.items() if k.startswith(("L0_", "L1_", "L2_")) or k == "prop_L"}


def _gauss2d_start(n):
    return np.tile([-8.0, -7.0], (n, 1))


GENERIC_CASES = {
    # name: (problem, initial states, chains, plan, adaptive, warp-specialised Philox run)
    "three_level": (three_level_gauss, _gauss2d_start, 33, [("run", 40)], None, True),
    "single_level_adaptive": (bp.gauss2d_problem, _gauss2d_start, 4097, [("run", 30)],
                              dict(idle=3, collection=8, refresh=2, eps=1e-4), True),
    "coarse_adaptive": (lambda: bp.linear_problem(True), lambda n: np.zeros((n, 2)), 1000, [("run", 20)],
                        dict(idle=2, collection=6, refresh=1, eps=1e-6), True),
    "pcn": (lambda: (dict(bp.linear_problem(False)[0], proposal="pcn", pcn_step=0.05),
                     dict(bp.linear_problem(False)[1], pcn_mean=np.array([0.3, -0.2]))),
            lambda n: np.zeros((n, 2)), 1000, [("run", 25)], None, True),
    "tempered_surrogate": (lambda: _fixture_problem("mlda_linear_tempered"), lambda n: np.zeros((n, 2)), 500,
                           [("run", 25)], None, True),
    "isclose_1d": (lambda: _fixture_problem("mrw_gauss1d"), lambda n: np.full((n, 1), -3.0), 33, [("run", 60)], None, True),
    "above_warp_specialised_limit": (lambda: bp.linear_problem(True), lambda n: np.zeros((n, 2)), 40001, [("run", 8)],
                                     None, False),
    "d5_two_level_40001": (lambda: bp.big_linear_problem(5, 4, 2, two_level=True, J=2, seed=9),
                           lambda n: 0.1 * np.random.default_rng(1).standard_normal((n, 5)), 40001, [("run", 5)], None, False),
}


@pytest.mark.parametrize("name", sorted(GENERIC_CASES))
def test_one_chain_per_thread_kernel_diagnostics(name):
    make, init, nc, plan, ad, ws = GENERIC_CASES[name]
    meta, arrays = make()
    check_case(meta, arrays, init(nc), plan, seed=23, adaptive=ad, ws=ws, label=name)


def test_adaptive_error_model_kernel_diagnostics():
    meta, _ = load("aem_linear")
    arrays = _fixture_problem("aem_linear")[1]
    nc = 600
    check_case(meta, arrays, np.zeros((nc, meta["dim"])), [("run", 40)], seed=29, aem=meta["aem"], ws=False,
               label="aem_linear")


# ------------------------------------------------------------------------------------------
# the FP64 tensor path (diagonal M2 in run-length form)
# ------------------------------------------------------------------------------------------
def _tensor_path_launch(d, rows, dense_L):
    """(wsm, dynamic shared memory) of linear_dmma_kernel.cu's launch_t for a model with d parameters and `rows` operand
    rows per level (data_dim, + d for a dense prior): the problem blob (abi.cu's tail), then as many warps as fit
    (12 at most for d > 32, else 16), each with its state and noise tiles (smem_plan.h), plus the two Welford tiles
    per warp when the blob leaves room for them at that warp count -- the shared-memory side of `wsm`; otherwise the
    moments are read and written in L2 at every flush."""
    kp = 16 if d <= 16 else (32 if d <= 32 else 64)
    ks, kq = kp + 4, kp // 4
    tail = sum(((r + 15) & ~15) * ks + ((r + 15) & ~15) + 2 * kp for r in rows) + 2 * kp + (kp * ks if dense_L else 0)
    blob = 8 * ((tail + 1) & ~1)

    def per_warp(wsm):
        return 8 * 8 * ks * (1 + (1 if dense_L else 0) + (2 if wsm else 0)) + 4 * 8 * (4 * kq + 4)
    budget = 227 * 1024
    warps = min(12 if kq == 16 else 16, (budget - blob) // per_warp(False))
    wsm = warps >= 4 and blob + warps * per_warp(True) <= budget
    return wsm, blob + warps * per_warp(wsm)


TENSOR_SHAPES = {
    # name: (d, data_dim, n_data, two level, J, side of wsm)
    "single_64x256": (64, 256, 1, False, 1, False),     # 140 KB of blob: the moments stay in L2
    "two_level_32x96": (32, 96, 2, True, 3, True),
    "ragged_23x45": (23, 45, 3, False, 1, True),
}


@pytest.mark.parametrize("nc", [5, 2500, 20011])
@pytest.mark.parametrize("shape", sorted(TENSOR_SHAPES))
def test_tensor_path_diagnostics(shape, nc):
    """Launches of 1 + 2 + 3 transitions: run-length flushes at accepted moves, at piece hand-overs inside a launch
    and at launch ends, in both storage forms of the moments (shared-memory tiles, L2)."""
    d, dd, nd, two, J, side = TENSOR_SHAPES[shape]
    meta, arrays = bp.big_linear_problem(d, dd, nd, two_level=two, J=J)
    wsm, smem = _tensor_path_launch(d, [dd] * meta["levels"], False)
    assert wsm == side, shape
    th0 = 0.01 * np.random.default_rng(nc).standard_normal((nc, d))
    check_case(meta, arrays, th0, [("run", 1), ("run", 2), ("run", 3)], seed=31, smem=smem, label=f"{shape} nc={nc}")


def test_tensor_path_dense_factor_dense_prior_and_pcn_diagnostics():
    rng = np.random.default_rng(11)
    d, dd, nc = 24, 40, 2500
    meta, arrays = bp.big_linear_problem(d, dd, 2)
    A = rng.standard_normal((d, d))
    prec = np.linalg.inv(1.5 * (A @ A.T / d + 0.5 * np.eye(d)))
    arrays = dict(arrays, L0_prior_prec=0.5 * (prec + prec.T), L0_prior_mean=0.1 * rng.standard_normal(d))
    mean, cov = bp.linear_gaussian_posterior(arrays, 0)
    arrays["prop_L"] = np.linalg.cholesky(2.4 ** 2 / d * cov)
    th0 = mean + 0.01 * rng.standard_normal((nc, d))
    wsm, smem = _tensor_path_launch(d, [dd + d], True)
    check_case(meta, arrays, th0, [("run", 1), ("run", 2), ("run", 3)], seed=37, smem=smem, label="dense")
    pmeta, parrays = bp.big_linear_problem(23, 45, 3)
    pmeta = dict(pmeta, proposal="pcn", pcn_step=0.05)
    parrays = dict(parrays, pcn_mean=0.1 * rng.standard_normal(23))
    wsm, smem = _tensor_path_launch(23, [45], False)
    check_case(pmeta, parrays, 0.01 * rng.standard_normal((nc, 23)), [("run", 4), ("run", 3)], seed=41, smem=smem,
               label="pcn")


# ------------------------------------------------------------------------------------------
# accumulation across runs, keep_diagnostics restarts and load_state
# ------------------------------------------------------------------------------------------
def _accumulation_plan(th0):
    return [("run", 3), ("run", 4), ("restart", th0[::-1].copy()), ("run", 2), ("reload",), ("run", 5)]


ACCUMULATION_CASES = {
    "lv": (lambda: bp.lv_problem(True, Nc=16, Nf=48), bp.lv_initial_states, 300),
    "one_chain_per_thread": (lambda: bp.linear_problem(True), lambda n: 0.2 * np.random.default_rng(2).standard_normal((n, 2)), 300),
    "warp_specialised": (bp.gauss2d_problem, _gauss2d_start, 77),
    "tensor_path": (lambda: bp.big_linear_problem(32, 96, 2, two_level=True, J=2),
                    lambda n: 0.01 * np.random.default_rng(3).standard_normal((n, 32)), 2500),
    "tensor_path_l2": (lambda: bp.big_linear_problem(64, 256, 1),
                       lambda n: 0.01 * np.random.default_rng(4).standard_normal((n, 64)), 300),
}


@pytest.mark.parametrize("name", sorted(ACCUMULATION_CASES))
def test_diagnostics_accumulate_across_runs_restarts_and_reloads(name):
    """run(3), run(4); set_state(other states, keep_diagnostics=True), run(2); state() -> load_state into a fresh
    handle, run(5): one reference over all the pre-states since the reset; counters of the last handle only."""
    make, init, nc = ACCUMULATION_CASES[name]
    meta, arrays = make()
    th0 = init(nc)
    check_case(meta, arrays, th0, _accumulation_plan(th0), seed=43, label=name)


# ------------------------------------------------------------------------------------------
# split moments at an odd length
# ------------------------------------------------------------------------------------------
def test_split_moments_odd_length_drops_the_last_sample():
    """split_moments_kernel's halves are [0, ns // 2) and [ns // 2, 2 (ns // 2)): at odd ns the last sample is in
    neither -- what split_rhat's half = ns // 2 assumes.  d = 8, 1,001 chains (not a multiple of 128)."""
    from yagre_mcmc_b200.ensemble import split_moments
    rng = np.random.default_rng(8)
    ns, d, nc = 301, 8, 1001
    x = rng.standard_normal((ns, d, nc)).cumsum(axis=0) * 0.1 + rng.normal(0.0, 3.0, (1, d, nc))
    x[-1] = 1e6                                    # would move both moments far if it were counted
    hm, hv = split_moments(torch.as_tensor(x, device="cuda"))
    half = ns // 2
    for h in range(2):
        pre = x[h * half:(h + 1) * half].transpose(2, 0, 1)           # [nc, half, d]
        mu, R = welford_reference(pre)
        tm, t2 = welford_tolerance(pre, (mu, R))
        assert np.all(np.abs(hm[h].cpu().numpy().T - mu.astype(np.float64)) <= tm), h
        m2 = hv[h].cpu().numpy().T * (half - 1)
        assert np.all(np.abs(m2 - np.einsum('cii->ci', R).astype(np.float64)) <= np.einsum('cii->ci', t2)), h
