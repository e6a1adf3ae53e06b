"""CPU: pins the C oracle (oracle/yagre_oracle.c) against the fixtures the
unmodified reference produced under injected noise (oracle/make_golden.py)."""
import numpy as np
import pytest

from oracle import cport
from golden_io import load, rel_err, CHAIN_CASES, MLDA3_CASES, AM_CASES, TEMPERED_CASES
from support import LOGPOST_RTOL


@pytest.mark.parametrize("name", CHAIN_CASES + MLDA3_CASES + TEMPERED_CASES)
def test_chain_trajectory_matches_reference(name):
    meta, a = load(name)
    pb = cport.Problem(meta, a)
    out = cport.run_injected(pb, a["theta0"], a["z"], a["u_c"], a["u_f"])
    # identical accept decisions
    assert np.array_equal(out["accepted"], a["accepted"]), name
    # trajectories: proposals are s + L z in both, so states agree to rounding
    assert rel_err(out["traj"], a["traj"]).max() <= 1e-13, name
    assert rel_err(out["logpost_L0"], a["logpost_L0"]).max() <= LOGPOST_RTOL, name
    if meta["levels"] >= 2:
        assert rel_err(out["logpost_L1"], a["logpost_L1"]).max() <= LOGPOST_RTOL, name
    if meta["levels"] == 3:
        assert rel_err(out["logpost_L2"], a["logpost_L2"]).max() <= LOGPOST_RTOL, name
    if "welford_mean" in a:     # FullDiagnostics: Welford of the pre-transition state
        np.testing.assert_allclose(out["welford_mean"], a["welford_mean"], rtol=1e-12)
        np.testing.assert_allclose(out["welford_var"], a["welford_var"], rtol=1e-12)


@pytest.mark.parametrize("name", AM_CASES)
def test_adaptive_metropolis_matches_reference_interface(name):
    """a14: the unmodified AdaptiveMRWProposal + MetropolisHastings.run (chain/adaptive.py:37-64,
    chain/metropolisHastings.py:103-120) drove our concrete AdaptiveCovarianceMatrix
    (oracle/ref_harness.py HaarioAdaptiveCovariance) under injected noise; update() call order, the
    covariance swap and the Cholesky (scipy / LAPACK dpotf2 order) are therefore the reference's.  Single level
    (Gaussian target of test/test_adaptive.py, LV) and as the coarse proposal of two-level delayed acceptance.
    Proposals through a dense factor differ from numpy's `L @ z` by at most an ulp (BLAS fuses the dot product),
    hence 1e-12 instead of bitwise."""
    meta, a = load(name)
    out = cport.run_injected(cport.Problem(meta, a), a["theta0"], a["z"], a["u_c"], a["u_f"])
    assert np.array_equal(out["accepted"], a["accepted"]), name
    assert rel_err(out["traj"], a["traj"]).max() <= 1e-12, name
    assert rel_err(out["logpost_L0"], a["logpost_L0"]).max() <= LOGPOST_RTOL, name
    if meta["levels"] == 2:
        assert rel_err(out["logpost_L1"], a["logpost_L1"]).max() <= LOGPOST_RTOL, name
    np.testing.assert_allclose(out["am_mean"], a["am_mean"], rtol=1e-12, atol=1e-14)
    np.testing.assert_allclose(out["am_m2"], a["am_m2"], rtol=1e-11, atol=1e-14)
    np.testing.assert_allclose(out["am_L"], a["am_L"], rtol=1e-11, atol=1e-14)
    assert np.all(a["am_refreshes"] > 0) and np.all(a["am_L"][:, 1, 0] != 0.0)      # the factor did switch


def test_three_level_fixture_ignores_the_first_sub_chain_length():
    """mlda.py:112-117: with two surrogates the MRW sub-chain has subChainLengths[1] steps; [0] is ignored."""
    meta, a = load("mlda3_gauss2d_hier")
    assert meta["subChainLengths"] == [9, 4] and meta["J"] == 4 and a["z"].shape[2] == 4
    for order in meta["rng_order"]:
        assert order.count('N') == 4 * a["u_f"].shape[1]


@pytest.mark.parametrize("name", ["aem_linear", "aem_linear_noheuristic"])
def test_adaptive_error_model_matches_reference(name):
    """AEM (chain/method/aem.py): trajectory, decisions, the error model's Welford state and even the
    number of coarse model evaluations (which depends on the LRU(3) cache behaviour, memoisation.py:76-149)
    equal the unmodified reference's."""
    meta, a = load(name)
    out = cport.run_injected(cport.Problem(meta, a), a["theta0"], a["z"], a["u_c"], a["u_f"])
    assert np.array_equal(out["accepted"], a["accepted"])
    assert rel_err(out["traj"], a["traj"]).max() <= 1e-13
    assert np.array_equal(out["aem_n"], a["aem_n"])
    np.testing.assert_allclose(out["aem_mean"], a["aem_mean"], rtol=1e-12, atol=1e-15)
    np.testing.assert_allclose(out["aem_var"], a["aem_var"], rtol=1e-12, atol=1e-15)
    assert np.array_equal(out["aem_model_evals"], a["n_model_evals"][:, 0])


def test_rng_call_order_of_reference_is_what_the_restatement_assumes():
    """(N u)*J then U only if the sub-chain moved (SURVEY Appendix A)."""
    meta, a = load("mlda_gauss2d")
    J = meta["J"]
    for c, order in enumerate(meta["rng_order"]):
        # strip per fine step
        i = 0
        for n in range(a["u_f"].shape[1]):
            moved = False
            for j in range(J):
                assert order[i] == 'N'; i += 1
                if i < len(order) and order[i] == 'u':
                    i += 1
                else:
                    assert np.all(a["z"][c, n, j] == 0.0)     # equality skip: no uniform drawn
            if i < len(order) and order[i] == 'U':
                i += 1
                moved = True
            same = np.array_equal(a["traj"][c, n + 1], a["traj"][c, n])
            assert moved or same
        assert i == len(order)


def test_nonfinite_policy():
    meta, a = load("mlda_lv_nonfinite")
    # chain 0 starts where RK4(16) overflows: logpost = -inf on both levels
    assert np.isneginf(a["logpost_L1"][0, 0]) and np.isneginf(a["logpost_L0"][0, 0])
    pb = cport.Problem(meta, a)
    assert np.isneginf(cport.logpost(pb, 1, a["theta0"][0]))
    F = cport.forward(pb, 1, a["theta0"][0])
    assert np.all(np.isposinf(F) | np.isfinite(F)) and np.isposinf(F).any()


def test_iat_welford_dense_match_reference():
    _, a = load("postprocessing")
    for i in range(5):
        s = a[f"seq{i}"]
        assert cport.iat(s, 'max') == int(a["iat_max"][i])
        assert cport.iat(s, 'mean') == int(a["iat_mean"][i])
        np.testing.assert_allclose(cport.acf(s[:, 0])[:64], a[f"acf{i}"], rtol=0, atol=1e-12)
    m, v = cport.welford(a["welford_x"])
    np.testing.assert_allclose(m, a["welford_mean"], rtol=1e-13)
    np.testing.assert_allclose(v, a["welford_var"], rtol=1e-13)
    L = cport.cholesky(a["dense_C"])
    for x, y1, y2, n2 in zip(a["dense_v"], a["dense_chol_apply"], a["dense_inv_apply"], a["dense_norm2"]):
        np.testing.assert_allclose(cport.chol_apply(L, x), y1, rtol=1e-13, atol=1e-15)
        inv = cport.chol_solve(L, x)
        np.testing.assert_allclose(inv, y2, rtol=1e-12, atol=1e-15)
        np.testing.assert_allclose(np.dot(x, inv), n2, rtol=1e-12)


def test_rk4_forward_matches_the_reference_solver():
    """The RK4 forward map (north_star's replacement of scipy.solve_ivp) against the reference's OWN
    LotkaVolterraSolver (test/testSetup.py:101-141; DOP853, rtol 1e-12, scipy's default atol 1e-6),
    evaluated in the container by oracle/make_golden.py: the C oracle equals the numpy RK4 plugin to
    rounding and the reference solver to 1e-4 (N = 64) / 2e-5 (N = 512) relative -- the style of
    test/test_solver_invoke.py:64-94 (rtol 1e-3), tighter."""
    import bench_problems as bp
    _, a = load("lv_forward")
    meta, arrays = bp.lv_problem(True)
    np.testing.assert_array_equal(arrays["L0_design"], a["design"])
    pb = cport.Problem(meta, arrays)
    for i, th in enumerate(a["thetas"]):
        Fc, Ff = cport.forward(pb, 0, th), cport.forward(pb, 1, th)
        np.testing.assert_allclose(Fc, a["rk4_64"][i], rtol=1e-13)
        np.testing.assert_allclose(Ff, a["rk4_512"][i], rtol=1e-13)
        np.testing.assert_allclose(Fc, a["ref_forward"][i], rtol=1e-4)
        np.testing.assert_allclose(Ff, a["ref_forward"][i], rtol=2e-5)
        np.testing.assert_allclose(a["rk4_1024"][i], a["ref_forward"][i], rtol=2e-5)


def test_stage_point_rk4_step_is_the_textbook_step():
    """The device integrates with the 20-instruction "stage-point" form of the RK4 step (csrc/lv_model.cuh):
    x' = k1/6 + (2/3) x3 + x4 (1/3 + (ha - hb y4)/6) with x2 = x + k1/2, x3 = x + k2/2, x4 = x + k3.  Restated
    here in numpy (same operation order as the kernel, FMAs unfused) against the textbook form the oracle uses:
    an algebraic identity, so the two agree to rounding after 512 steps."""
    import bench_problems as bp
    _, a = load("lv_forward")
    design, (alpha, gamma, T) = a["design"], a["lv"]
    for th in a["thetas"]:
        for N in (64, 512):
            h = T / N
            hb, hd, ha, hg = h * np.exp(th[0]), h * np.exp(th[1]), h * alpha, h * gamma
            x, y = design[:, 0].copy(), design[:, 1].copy()
            for _ in range(N):
                tx, ty = x * (-hb / 6 * y + ha / 6), y * (hd / 6 * x - hg / 6)
                x2, y2 = 3.0 * tx + x, 3.0 * ty + y
                x3, y3 = x2 * (-hb / 2 * y2 + ha / 2) + x, y2 * (hd / 2 * x2 - hg / 2) + y
                x4, y4 = x3 * (-hb * y3 + ha) + x, y3 * (hd * x3 - hg) + y
                wx, wy = -hb / 6 * y4 + (ha / 6 + 1.0 / 3.0), hd / 6 * x4 + (1.0 / 3.0 - hg / 6)
                x, y = x4 * wx + (2.0 / 3.0 * x3 + tx), y4 * wy + (2.0 / 3.0 * y3 + ty)
            want = bp.lv_forward_numpy(th, design, alpha, gamma, T, N)
            np.testing.assert_allclose(np.stack([x, y], axis=1), want, rtol=5e-13)


def test_philox_known_answers():
    """Random123 kat_vectors for philox4x32-10."""
    assert cport.philox4x32_10([0, 0, 0, 0], [0, 0]) == [0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8]
    assert cport.philox4x32_10([0xffffffff] * 4, [0xffffffff] * 2) == \
        [0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd]
    assert cport.philox4x32_10([0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344], [0xa4093822, 0x299f31d0]) == \
        [0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1]


def test_philox_streams_statistics():
    z = np.array([cport.philox_normals(7, c, s, 0, 2) for c in range(50) for s in range(100)])
    u = np.array([cport.philox_uniform(7, c, s, 0xFFFF) for c in range(50) for s in range(100)])
    assert abs(z.mean()) < 0.05 and abs(z.var() - 1) < 0.05
    assert abs(u.mean() - 0.5) < 0.02 and 0 <= u.min() and u.max() < 1
