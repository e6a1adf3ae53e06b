"""GPU: the drop-in Python surface (builders -> run -> trajectory / diagnostics), written like the
reference's own tests (yagremcmc/test/test_mcmc_1d.py, test_mcmc_2d.py, test_mlda.py,
test_inference_mcmc_singleLevel.py) with the same targets and tolerances."""
import numpy as np
import pytest
import torch

import bench_problems as bp
from support import ensemble
from yagre_mcmc_b200.parameter import ParameterVector, ScalarParameter
from yagre_mcmc_b200.model import ForwardModel, LinearModelSolver, LotkaVolterraRK4Solver, LotkaVolterraParameter
from yagre_mcmc_b200.statistics import (IIDCovarianceMatrix, DiagonalCovarianceMatrix, DenseCovarianceMatrix,
                                        Gaussian, CentredGaussianNoise, Data, AdditiveGaussianNoiseLikelihood,
                                        BayesianRegressionModel, BayesianRegressionModelHierarchy,
                                        GaussianTargetDensity2d, GaussianTargetDensity1d)
from yagre_mcmc_b200.utility import Hierarchy, SharedComponent
from yagre_mcmc_b200.chain.method import MRWBuilder, MLDABuilder, AMBuilder, PCNBuilder, AEMBuilder
from yagre_mcmc_b200.statistics import AEMLikelihood
from yagre_mcmc_b200.chain.target import UnnormalisedPosterior
from yagre_mcmc_b200.chain.diagnostics import DummyDiagnostics, AcceptanceRateDiagnostics, FullDiagnostics
from yagre_mcmc_b200.postprocessing.autocorrelation import integrated_autocorrelation, effective_sample_size

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("diagnostics", [DummyDiagnostics, AcceptanceRateDiagnostics, FullDiagnostics])
def test_mcmc_1d_single_chain(diagnostics):
    """reference test/test_mcmc_1d.py:58-116 (target N(1, 1.5^2)... here example_mcmc_1d.py's N(1.5, 1))."""
    tgtMean, tgtVar = ScalarParameter.from_coefficient(np.array([1.5])), 1.0
    b = MRWBuilder()
    b.explicitTarget = GaussianTargetDensity1d(tgtMean, tgtVar)
    b.proposalCovariance = DiagonalCovarianceMatrix(np.array([1.5]))
    b.diagnostics = diagnostics()
    b.seed = 18
    mc = b.build_method()
    nSteps = 15000
    mc.run(nSteps, ScalarParameter.from_coefficient(np.array([-3.0])), verbose=False)
    states = np.asarray(mc.chain.trajectory)
    assert len(mc.chain.trajectory) == nSteps and mc.chain.length == nSteps        # test_mcmc_1d.py:89
    assert states.shape == (nSteps, 1) and states[0, 0] == -3.0
    burnIn = 200
    thin = integrated_autocorrelation(states[burnIn:], 'max')
    assert 2 <= thin <= 30
    sel = states[burnIn::thin]
    MTOL = VTOL = 0.1                                                               # test_mcmc_1d.py:109-110
    assert abs(sel.mean() - 1.5) < MTOL and abs(sel.var() - tgtVar) < VTOL
    if diagnostics is not DummyDiagnostics:
        moved = (states[1:] != states[:-1]).any(axis=1).mean()
        assert abs(mc.diagnostics.global_acceptance_rate() - moved) < 1e-12
    if diagnostics is FullDiagnostics:                 # Welford of the pre-transition states
        np.testing.assert_allclose(mc.diagnostics.mean(), states[:-1].mean(0), rtol=1e-10)
        np.testing.assert_allclose(mc.diagnostics.marginal_variance(), states[:-1].var(0, ddof=1), rtol=1e-9)


@pytest.mark.parametrize("proposal", ["iid", "diag", "dense"])
def test_mcmc_2d_ensemble(proposal):
    """reference test/test_mcmc_2d.py:18-81, run as 256 chains x 2,000 steps."""
    tgtMean = ParameterVector(np.array([1.0, 1.5]))
    tgtCov = np.array([[2.4, -0.5], [-0.5, 0.7]])
    b = MRWBuilder()
    b.explicitTarget = GaussianTargetDensity2d(tgtMean, tgtCov)
    b.proposalCovariance = {"iid": IIDCovarianceMatrix(2, 0.75),
                            "diag": DiagonalCovarianceMatrix(np.array([1.2, 0.4])),
                            "dense": DenseCovarianceMatrix(np.array([[1.2, -0.3], [-0.3, 0.5]]))}[proposal]
    b.diagnostics = FullDiagnostics()
    b.nChains, b.seed = 256, 116
    mc = b.build_method()
    mc.run(2000, ParameterVector(np.array([-8.0, -7.0])), verbose=False)
    states = np.asarray(mc.chain.trajectory)
    assert states.shape == (2000, 256, 2)
    assert np.all(states[0] == np.array([-8.0, -7.0]))
    x = states[300:].reshape(-1, 2)
    MTOL, CTOL = 5e-2, 1e-1                                                         # test_mcmc_2d.py:66-67
    assert np.all(np.abs(x.mean(0) - tgtMean.coefficient) < MTOL)
    assert np.all(np.abs(np.cov(x.T) - tgtCov) < CTOL)
    rate = mc.diagnostics.global_acceptance_rate()
    assert 0.2 < rate < 0.8
    assert mc.diagnostics.acceptance_rates().shape == (256,)
    pooled = mc.pooled()
    assert pooled["n_chains"] == 256 and np.all(np.abs(pooled["rhat"] - 1.0) < 0.2)
    iat = integrated_autocorrelation(mc.chain.trajectory, 'max')
    assert iat.shape == (256,) and np.all(iat >= 1)


def test_pooled_proposal_covariance_through_the_builder():
    """Burn-in restart idiom of the reference (example_inference_linearModel_twoLevel.py:228,236) with the
    pooled proposal covariance in between: burn-in from a far start with a small iid proposal, pool, restart
    from chain.trajectory[-1]."""
    tgtMean = np.array([1.0, 1.5])
    tgtCov = np.array([[2.4, -0.5], [-0.5, 0.7]])
    b = MRWBuilder()
    b.explicitTarget = GaussianTargetDensity2d(ParameterVector(tgtMean), tgtCov)
    b.proposalCovariance = IIDCovarianceMatrix(2, 0.02)
    b.nChains, b.seed = 512, 9
    mc = b.build_method()
    mc.run(3000, ParameterVector(np.array([0.0, 0.0])), verbose=False)
    rate0 = mc.diagnostics.global_acceptance_rate()
    pooled = mc.pool_proposal_covariance()
    L = pooled["prop_L"]
    assert L.shape == (2, 2) and L[0, 1] == 0.0
    last = np.asarray(mc.chain.trajectory)[-1]                                      # [nChains, d]
    mc.clear()              # diagnostics accumulate across run() until clear(), as in the reference (:122-125)
    mc.run(3000, ParameterVector(last), verbose=False)
    rate1 = mc.diagnostics.global_acceptance_rate()
    assert rate0 > 0.7 and 0.25 < rate1 < 0.45                                      # tiny steps -> tuned steps
    x = np.asarray(mc.chain.trajectory)[500:].reshape(-1, 2)
    assert np.all(np.abs(x.mean(0) - tgtMean) < 5e-2)
    assert np.all(np.abs(np.cov(x.T) - tgtCov) < 1e-1)


def _mlda_targets(surrMeanShift, surrCov):
    tgtMean = ParameterVector(np.array([1.0, 1.5]))
    tgtCov = np.array([[2.5, -0.3], [-0.3, 0.9]])
    tgt = GaussianTargetDensity2d(tgtMean, tgtCov)
    sur = GaussianTargetDensity2d(ParameterVector(tgtMean.coefficient + surrMeanShift), surrCov)
    return tgtMean, tgtCov, tgt, sur


def test_mlda_two_level():
    """reference test/test_mlda.py:133-186: surrogate mean +[0.1,-0.2], cov 1.5 x target, J = 10."""
    tgtMean, tgtCov, tgt, sur = _mlda_targets(np.array([0.1, -0.2]), 1.5 * np.array([[2.5, -0.3], [-0.3, 0.9]]))
    b = MLDABuilder()
    b.explicitTarget = tgt
    b.surrogateTargets = [sur]
    b.baseProposalCovariance = IIDCovarianceMatrix(2, 1.0)
    b.subChainLengths = [10]
    b.nChains, b.seed = 128, 456
    mc = b.build_method()
    mc.run(1500, ParameterVector(np.array([-5.0, 4.0])), verbose=False)
    states = np.asarray(mc.chain.trajectory)
    x = states[500::5].reshape(-1, 2)
    assert np.allclose(x.mean(0), tgtMean.coefficient, atol=0.1)                    # test_mlda.py:181
    assert 0.1 < mc.diagnostics.global_acceptance_rate() < 0.9                      # test_mlda.py:184-186
    coarse, fine = mc.evaluation_counts()
    assert fine <= 128 * 1499 and coarse <= 10 * 128 * 1499


def test_mlda_perfect_surrogate_always_accepts():
    """reference test/test_mlda.py:94-130: surrogate == target => fine acceptance rate 1."""
    tgtMean, tgtCov, tgt, _ = _mlda_targets(np.zeros(2), np.eye(2))
    b = MLDABuilder()
    b.explicitTarget = tgt
    b.surrogateTargets = [GaussianTargetDensity2d(tgtMean, tgtCov)]
    b.baseProposalCovariance = IIDCovarianceMatrix(2, 0.01)     # tiny steps: the sub-chain nearly always moves
    b.subChainLengths = [5]
    b.nChains, b.seed = 64, 123
    mc = b.build_method()
    mc.run(1000, tgtMean, verbose=False)
    assert abs(mc.diagnostics.global_acceptance_rate() - 1.0) < 1e-3                # test_mlda.py:128-130


def test_mlda_two_surrogates_through_the_builder():
    """reference test/test_mlda.py:14-91 (two surrogates, subChainLengths [6, 6]; passes at HEAD): chain length,
    acceptance in (0.1, 0.9), mean within 0.1 -- here over an ensemble.  Three surrogates crash in the reference
    (AttributeError in SurrogateTransition) and are refused."""
    tgtMean = np.array([1.0, 1.5])
    tgtCov = np.array([[2.4, -0.5], [-0.5, 0.7]])
    tgt = GaussianTargetDensity2d(ParameterVector(tgtMean), tgtCov)
    base = GaussianTargetDensity2d(ParameterVector(tgtMean + [-0.05, 0.01]), 3.0 * np.array([[2.8, -0.1], [-0.1, 1.7]]))
    fine = GaussianTargetDensity2d(ParameterVector(tgtMean + [0.0, -0.01]), 1.5 * np.array([[2.4, -0.3], [-0.3, 1.1]]))
    b = MLDABuilder()
    b.explicitTarget = tgt
    b.surrogateTargets = [base, fine]
    b.baseProposalCovariance = IIDCovarianceMatrix(2, 1.0)
    b.subChainLengths = [6, 6]
    b.nChains, b.seed = 512, 42
    mc = b.build_method()
    assert mc.nSurrogates == 2
    mc.run(2000, ParameterVector(np.array([-8.0, -7.0])), verbose=False)
    states = np.asarray(mc.chain.trajectory)
    assert states.shape == (2000, 512, 2)
    assert 0.1 < mc.diagnostics.global_acceptance_rate() < 0.9
    np.testing.assert_allclose(states[500::5].reshape(-1, 2).mean(0), tgtMean, atol=0.1)
    # The reference's two-surrogate recursion is not an exact delayed-acceptance sampler (the screen uses the
    # finest surrogate although the sub-chain ran on the base one, mlda.py:130,146-154): the UNMODIFIED reference,
    # run here for 3 x 30,000 steps (seeds 1-3), gives covariance [[3.86, -0.86], [-0.86, 1.00]] and acceptance
    # 0.52-0.53 on this problem, not the target's [[2.4, -0.5], [-0.5, 0.7]].  The drop-in reproduces that.
    np.testing.assert_allclose(np.cov(states[500::5].reshape(-1, 2).T), [[3.86, -0.86], [-0.86, 1.0]], atol=0.12)
    assert 0.50 < mc.diagnostics.global_acceptance_rate() < 0.55
    coarse, fine_ev = mc.evaluation_counts()
    assert coarse > 5.9 * 512 * 1999 and fine_ev <= 512 * 1999
    b3 = MLDABuilder()
    b3.explicitTarget = tgt
    b3.surrogateTargets = [base, fine, fine]
    b3.baseProposalCovariance = IIDCovarianceMatrix(2, 1.0)
    b3.subChainLengths = [3, 3, 3]
    with pytest.raises(NotImplementedError):
        b3.build_method()


def test_consecutive_runs_use_fresh_noise_and_diagnostics_accumulate():
    """ADVICE r1: the reference's generator keeps advancing across run() calls and its diagnostics accumulate
    until clear() (chain/metropolisHastings.py:103-125)."""
    b = MRWBuilder()
    b.explicitTarget = GaussianTargetDensity2d(ParameterVector(np.array([1.0, 1.5])), np.array([[2.4, -0.5], [-0.5, 0.7]]))
    b.proposalCovariance = IIDCovarianceMatrix(2, 1.0)
    b.nChains, b.seed = 64, 3
    b.diagnostics = FullDiagnostics()
    mc = b.build_method()
    start = ParameterVector(np.array([1.0, 1.5]))
    mc.run(200, start, verbose=False)
    t1 = np.asarray(mc.chain.trajectory).copy()
    n1 = mc.ensemble.counters()
    mc.run(200, start, verbose=False)
    t2 = np.asarray(mc.chain.trajectory)
    n2 = mc.ensemble.counters()
    assert np.array_equal(t1[0], t2[0]) and not np.array_equal(t1[1:], t2[1:])
    assert n1["step_index"] == 199 and n2["step_index"] == 398
    assert n2["transitions"] == 2 * n1["transitions"] and n2["welford_n"] == 398          # accumulated
    mc.clear()
    mc.run(100, start, verbose=False)
    n3 = mc.ensemble.counters()
    assert n3["welford_n"] == 99 and n3["transitions"] == 64 * 99 and n3["step_index"] == 497


def test_adaptive_coarse_proposal_through_the_mlda_builder():
    """Extension (INTEGRATION.md): an AdaptiveCovarianceMatrix descriptor as baseProposalCovariance makes the
    coarse MRW of delayed acceptance adaptive per chain (the reference's AdaptiveMRWProposal as the surrogate's
    proposal method, pinned by tests/golden/am_mlda_*.npz).  C5 problem through the builders."""
    from yagre_mcmc_b200.chain.adaptive import AdaptiveCovarianceMatrix
    meta, arr, hierarchy, lik, prior = _lv_hierarchy()
    b = MLDABuilder()
    b.bayesModel = hierarchy
    b.baseProposalCovariance = AdaptiveCovarianceMatrix(IIDCovarianceMatrix(2, 0.1), idleSteps=30, collectionSteps=150,
                                                       eps=1e-8, refresh=5)
    b.subChainLengths = [3]
    b.nChains, b.seed, b.storeTrajectory = 2048, 11, False
    mc = b.build_method()
    th0 = bp.lv_initial_states(2048)
    mc.run(400, LotkaVolterraParameter(th0), verbose=False)
    L = mc.proposal_factors()
    assert L.shape == (2048, 2, 2) and np.all(L[:, 0, 1] == 0.0) and np.all(L[:, 0, 0] < np.sqrt(0.1))
    assert mc.ensemble.counters()["am_steps"] == 399
    assert 0.1 <= mc.diagnostics.global_acceptance_rate() <= 0.8


def test_tempered_surrogate_through_the_builder():
    """TemperedUnnormalisedPosterior (reference chain/target.py:25-43) as the explicit surrogate of MLDABuilder."""
    from yagre_mcmc_b200.chain.target import TemperedUnnormalisedPosterior
    meta, a = bp.linear_problem(True)
    noise = CentredGaussianNoise(IIDCovarianceMatrix(2, 0.3))
    prior = Gaussian(ParameterVector(a["L0_prior_mean"]), IIDCovarianceMatrix(2, 5.0))
    likC, likF = [AdditiveGaussianNoiseLikelihood(Data(a["L0_data"]), ForwardModel(LinearModelSolver(a[f"L{l}_G"], a[f"L{l}_b"])), noise)
                  for l in range(2)]
    b = MLDABuilder()
    b.explicitTarget = UnnormalisedPosterior(likF, prior)
    b.surrogateTargets = [TemperedUnnormalisedPosterior(likC, prior, 0.35)]
    b.baseProposalCovariance = IIDCovarianceMatrix(2, 0.5)
    b.subChainLengths = [5]
    b.nChains, b.seed = 4096, 5
    mc = b.build_method()
    mc.run(3000, ParameterVector(np.zeros(2)), verbose=False)
    x = np.asarray(mc.chain.trajectory)[1000::20].reshape(-1, 2)
    mean, cov = bp.linear_posterior('f')
    np.testing.assert_allclose(x.mean(0), mean, atol=0.02)           # the fine screen keeps the target exact
    np.testing.assert_allclose(np.cov(x.T), cov, rtol=0.1, atol=5e-3)
    with pytest.raises(ValueError):
        TemperedUnnormalisedPosterior(likC, prior, 1.5)


def _lv_hierarchy():
    meta, arr = bp.lv_problem(True)
    design, data = arr["L0_design"], arr["L0_data"]
    cfg = dict(T=10., alpha=0.8, gamma=0.4, nData=10, dataDim=2)
    noise = CentredGaussianNoise(IIDCovarianceMatrix(2, 0.04))
    prior = Gaussian(LotkaVolterraParameter.from_coefficient(np.zeros(2)), IIDCovarianceMatrix(2, 1.4))
    lik = [AdditiveGaussianNoiseLikelihood(Data(data), ForwardModel(LotkaVolterraRK4Solver(design, dict(cfg, rk4Steps=N))), noise)
           for N in (64, 512)]
    return meta, arr, BayesianRegressionModelHierarchy(Hierarchy(lik), SharedComponent(prior, 2)), lik, prior


def test_lv_two_level_inference_through_builders_equals_direct_backend():
    """The builder path lowers to exactly the arrays of bench_problems.lv_problem, so the trajectory
    equals the one of the bare C-ABI handle with the same seed (bitwise)."""
    meta, arr, hier, lik, prior = _lv_hierarchy()
    nc, n = 96, 25
    th0 = bp.lv_initial_states(nc)
    b = MLDABuilder()
    b.bayesModel = hier
    b.baseProposalCovariance = IIDCovarianceMatrix(2, 0.1)
    b.subChainLengths = [3]
    b.nChains, b.seed = nc, 77
    mc = b.build_method()
    mc.run(n, LotkaVolterraParameter(th0), verbose=False)
    states = np.asarray(mc.chain.trajectory)
    assert states.shape == (n, nc, 2) and np.array_equal(states[0], th0)
    ens = ensemble(meta, arr, nc, seed=77)
    ens.set_state(th0)
    direct = ens.run(n - 1, samples=True)["samples"].permute(0, 2, 1).cpu().numpy()
    assert np.array_equal(states[1:], direct)
    # target.evaluate_log is served by the device
    lp = mc.target.evaluate_log(LotkaVolterraParameter(th0[0]))
    assert np.isfinite(lp) and abs(lp - float(ens.logpost(1, th0[:1])[0])) == 0.0
    # ESS idiom of example_inference_lotkaVolterra_twoLevel.py:117-118,132
    ess = effective_sample_size(mc.chain.trajectory, burnIn=5)
    assert ess.shape == (nc,) and np.all(ess >= 1)


def test_lv_single_level_mrw_through_builder():
    """reference test/test_inference_mcmc_singleLevel.py:77-119 style (MRW with iid / diag proposal)."""
    meta, arr, hier, lik, prior = _lv_hierarchy()
    for cov in (IIDCovarianceMatrix(2, 0.02), DiagonalCovarianceMatrix(np.array([0.02, 0.01]))):
        b = MRWBuilder()
        b.bayesModel = BayesianRegressionModel(lik[1], prior)
        b.proposalCovariance = cov
        b.diagnostics = FullDiagnostics()
        b.nChains, b.seed = 128, 16
        mc = b.build_method()
        mc.run(200, LotkaVolterraParameter(bp.LV_TRUTH), verbose=False)
        states = np.asarray(mc.chain.trajectory)
        assert states.shape == (200, 128, 2) and np.all(np.isfinite(states))
        assert 0.05 < mc.diagnostics.global_acceptance_rate() < 0.95
        assert np.all(np.abs(states[100:].reshape(-1, 2).mean(0) - bp.LV_TRUTH) < 0.15)


def test_lv_pcn_through_builder():
    """reference test/test_inference_mcmc_singleLevel.py:121-148 (pCN on the LV posterior)."""
    meta, arr, hier, lik, prior = _lv_hierarchy()
    b = PCNBuilder()
    b.bayesModel = BayesianRegressionModel(lik[1], prior)
    b.stepSize = 0.004
    b.diagnostics = FullDiagnostics()
    b.nChains, b.seed = 256, 17
    mc = b.build_method()
    mc.run(400, LotkaVolterraParameter(bp.LV_TRUTH), verbose=False)
    states = np.asarray(mc.chain.trajectory)
    assert states.shape == (400, 256, 2) and np.all(np.isfinite(states))
    assert 0.1 < mc.diagnostics.global_acceptance_rate() < 0.9
    assert np.all(np.abs(states[200:].reshape(-1, 2).mean(0) - bp.LV_TRUTH) < 0.1)
    # the pCN target is the likelihood alone (pcn.py:52-57): evaluate_log has no prior term
    th = bp.LV_TRUTH + 0.01
    from yagre_mcmc_b200.chain.method import MRWBuilder as _M
    m = _M()
    m.bayesModel = BayesianRegressionModel(lik[1], prior)
    m.proposalCovariance = IIDCovarianceMatrix(2, 0.1)
    post = m.build_method().target.evaluate_log(LotkaVolterraParameter(th))
    like = mc.target.evaluate_log(LotkaVolterraParameter(th))
    assert abs((post - like) - (-0.5 * float(th @ th) / 1.4)) < 1e-9


def test_linear_two_level_through_builders_matches_closed_form():
    """example_inference_linearModel_twoLevel.py:33-74,157-177 (C3) through the builders."""
    meta, a = bp.linear_problem(True)
    noise = CentredGaussianNoise(IIDCovarianceMatrix(2, 0.3))
    prior = Gaussian(ParameterVector(a["L0_prior_mean"]), IIDCovarianceMatrix(2, 5.0))
    lik = [AdditiveGaussianNoiseLikelihood(Data(a["L0_data"]), ForwardModel(LinearModelSolver(a[f"L{l}_G"], a[f"L{l}_b"])), noise)
           for l in range(2)]
    b = MLDABuilder()
    b.bayesModel = BayesianRegressionModelHierarchy(Hierarchy(lik), SharedComponent(prior, 2))
    b.baseProposalCovariance = IIDCovarianceMatrix(2, 0.5)
    b.subChainLengths = [5]
    b.nChains, b.seed, b.thin = 2048, 5, 500
    mc = b.build_method()
    # acceptance is ~0.04 and the IAT ~4e3 for this pair of models (SURVEY section 6): long burn-in
    mc.run(40001, ParameterVector(np.zeros(2)), verbose=False)
    states = np.asarray(mc.chain.trajectory)                   # init + 80 thinned states
    assert states.shape == (81, 2048, 2)
    mean, cov = bp.linear_posterior('f')
    x = states[61:].reshape(-1, 2)
    # slow mixer (see tests/test_backend_gpu.py::test_c3_linear_posterior_moments): loose tolerances
    np.testing.assert_allclose(x.mean(0), mean, atol=0.03)
    np.testing.assert_allclose(np.cov(x.T), cov, rtol=0.15, atol=5e-3)


def test_large_linear_model_through_builders():
    """d = 24, dataDim = 40 (beyond the one-chain-per-thread kernels): the builder path lands on the DMMA
    kernel; posterior moments against the closed form, FullDiagnostics from the diagonal Welford state."""
    meta, a = bp.big_linear_problem(24, 40, 2, two_level=True, J=2)
    d, dd = 24, 40
    noise = CentredGaussianNoise(IIDCovarianceMatrix(dd, 0.05))
    prior = Gaussian(ParameterVector(np.zeros(d)), IIDCovarianceMatrix(d, 2.0))
    lik = [AdditiveGaussianNoiseLikelihood(Data(a["L0_data"]), ForwardModel(LinearModelSolver(a[f"L{l}_G"], a[f"L{l}_b"])), noise)
           for l in range(2)]
    b = MLDABuilder()
    b.bayesModel = BayesianRegressionModelHierarchy(Hierarchy(lik), SharedComponent(prior, 2))
    b.baseProposalCovariance = IIDCovarianceMatrix(d, float(a["prop_L"][0, 0]) ** 2)
    b.subChainLengths = [2]
    b.targetDiagnostics = FullDiagnostics()
    b.nChains, b.seed, b.thin = 2048, 3, 100
    mc = b.build_method()
    mean, cov = bp.linear_gaussian_posterior(a, 1)
    mc.run(3001, ParameterVector(mean), verbose=False)
    assert mc.ensemble.last_launch()["block"] == 512          # linear_dmma_mh_kernel (16 warps)
    states = np.asarray(mc.chain.trajectory)
    assert states.shape == (31, 2048, d)
    x = states[11:].reshape(-1, d)
    se = np.sqrt(np.diag(cov))
    assert np.all(np.abs(x.mean(0) - mean) < 0.05 * se + 5 * se / np.sqrt(2048))
    np.testing.assert_allclose(x.var(0, ddof=1), np.diag(cov), rtol=0.1)
    assert 0.1 < mc.diagnostics.global_acceptance_rate() < 0.8
    np.testing.assert_allclose(mc.diagnostics.mean().mean(0), mean, atol=0.05)
    assert mc.diagnostics.marginal_variance().shape == (2048, d)
    lp = mc.target.evaluate_log(ParameterVector(mean))
    assert np.isfinite(lp)


def test_adaptive_error_model_through_builders():
    """example_inference_linearModel_twoLevel.py:95-102,183-191: AEM on the C3 linear pair lifts the fine
    acceptance rate (0.04 -> 0.35 in the reference's script, SURVEY 8f) and still samples the fine posterior."""
    meta, a = bp.linear_problem(True)
    noise = CentredGaussianNoise(IIDCovarianceMatrix(2, 0.3))
    prior = Gaussian(ParameterVector(a["L0_prior_mean"]), IIDCovarianceMatrix(2, 5.0))
    lik = [AEMLikelihood(Data(a["L0_data"]), ForwardModel(LinearModelSolver(a[f"L{l}_G"], a[f"L{l}_b"])), noise, 100, True)
           for l in range(2)]
    b = AEMBuilder()
    b.bayesModel = BayesianRegressionModelHierarchy(Hierarchy(lik), SharedComponent(prior, 2))
    b.baseProposalCovariance = IIDCovarianceMatrix(2, 0.5)
    b.subChainLengths = [5]
    b.targetDiagnostics = FullDiagnostics()
    b.nChains, b.seed, b.thin = 2048, 9, 50
    mc = b.build_method()
    mc.run(6001, ParameterVector(np.zeros(2)), verbose=False)
    em = mc.error_model()
    # a per-chain error model can also go wrong for an individual chain (a poor early estimate freezes it),
    # exactly as a single reference chain can: judge the ensemble by its bulk
    assert em["nData"].shape == (2048,) and np.median(em["nData"]) > 1000 and (em["nData"] > 200).mean() > 0.95
    mean, cov = bp.linear_posterior('f')
    # the error model estimates E[F_f - F_c] over the posterior: (G_f - G_c) mean + (b_f - b_c)
    expect = (a["L1_G"] - a["L0_G"]) @ mean + (a["L1_b"] - a["L0_b"])
    np.testing.assert_allclose(np.median(em["mean"], axis=0), expect, atol=0.05)
    assert mc.diagnostics.global_acceptance_rate() > 0.2
    good = em["nData"] > 200
    x = np.asarray(mc.chain.trajectory)[60:][:, good].reshape(-1, 2)
    np.testing.assert_allclose(x.mean(0), mean, atol=0.03)
    np.testing.assert_allclose(np.cov(x.T), cov, rtol=0.15, atol=5e-3)
    coarse, fine = mc.evaluation_counts()
    assert coarse >= 5 * 2048 * 6000 * 0.99                    # J proposals per step + cache-miss re-evaluations


def test_adaptive_metropolis_builder():
    """thresholds of the reference's skipped test/test_adaptive.py (mean 0.03 / cov 0.05 / acceptance)."""
    mean, cov = np.array([1.0, 1.5]), np.array([[3.2, -0.4], [-0.4, 0.2]])
    b = AMBuilder()
    b.explicitTarget = GaussianTargetDensity2d(ParameterVector(mean), cov)
    b.idleSteps, b.collectionSteps, b.regularisationParameter = 100, 500, 1e-4
    b.initialCovariance = IIDCovarianceMatrix(2, 1.0)
    b.nChains, b.seed, b.thin = 1024, 20, 5
    mc = b.build_method()
    mc.run(6001, ParameterVector(np.array([-3.0, 4.0])), verbose=False)
    x = np.asarray(mc.chain.trajectory)[300:].reshape(-1, 2)
    np.testing.assert_allclose(x.mean(0), mean, atol=0.03)
    np.testing.assert_allclose(np.cov(x.T), cov, atol=0.05)
    assert 0.1 <= mc.diagnostics.global_acceptance_rate() <= 0.8
    L = mc.proposal_factors()
    assert L.shape == (1024, 2, 2) and np.all(L[:, 0, 1] == 0.0)
    with pytest.raises(NotImplementedError):                   # chain/adaptive.py:41-43
        b1 = AMBuilder()
        b1.explicitTarget = GaussianTargetDensity1d(ScalarParameter.from_coefficient(np.array([0.0])), 1.0)
        b1.idleSteps, b1.collectionSteps, b1.regularisationParameter = 1, 2, 1e-4
        b1.initialCovariance = DiagonalCovarianceMatrix(np.array([1.0]))
        b1.build_method()


def test_verbose_run_and_clear(capsys):
    b = MRWBuilder()
    b.explicitTarget = GaussianTargetDensity2d(ParameterVector(np.zeros(2)), np.eye(2))
    b.proposalCovariance = IIDCovarianceMatrix(2, 1.0)
    b.nChains = 8
    mc = b.build_method()
    mc.run(100, ParameterVector(np.zeros(2)), verbose=True)
    assert mc.chain.length == 100
    mc.clear()
    assert mc.chain.length == 0 and mc.diagnostics.global_acceptance_rate() == 0.0
    mc.run(1, ParameterVector(np.zeros(2)), verbose=False)      # chainLength 1 = just the initial state
    assert np.asarray(mc.chain.trajectory).shape == (1, 8, 2)


def test_surrogate_diagnostics_record_the_coarse_acceptance():
    """ADVICE r1: user-supplied surrogateDiagnostics are fed (reference: the MRW of the surrogate hierarchy processes
    every coarse step, chain/method/mlda.py:58-62).  The kernels count accepted coarse sub-steps of the ensemble."""
    tgtMean, tgtCov, tgt, sur = _mlda_targets(np.array([0.1, -0.2]), 1.5 * np.array([[2.5, -0.3], [-0.3, 0.9]]))
    b = MLDABuilder()
    b.explicitTarget = tgt
    b.surrogateTargets = [sur]
    b.baseProposalCovariance = IIDCovarianceMatrix(2, 1.0)
    b.subChainLengths = [10]
    b.surrogateDiagnostics = [AcceptanceRateDiagnostics()]
    b.nChains, b.seed = 256, 1
    mc = b.build_method()
    mc.run(500, ParameterVector(np.array([1.0, 1.5])), verbose=False)
    coarse = b.surrogateDiagnostics[0].global_acceptance_rate()
    c = mc.ensemble.counters()
    assert c["coarse_accepted"] > 0 and coarse == c["coarse_accepted"] / (c["transitions"] * 10)
    assert 0.3 < coarse < 0.8 and coarse != mc.diagnostics.global_acceptance_rate()
    mc.clear()
    mc.run(100, ParameterVector(np.array([1.0, 1.5])), verbose=False)
    assert mc.ensemble.counters()["transitions"] == 256 * 99          # clear() restarted the device counters too
