"""GPU: pooled statistics from a stored sample buffer (yg_pooled_samples) and the pooled path it opens for d > 8.

  * the statistics vector against the long-double reference of tests/pooled_samples_reference.py, within its derived
    per-entry bounds, over a sweep of d, samples and chains, and on data with a large common offset;
  * bitwise repeatability;
  * agreement with the Welford path (yg_pooled_stats) at d <= 8 on the pre-transition states of real runs;
  * the tensor path end to end through the builders: pooled() and pool_proposal_covariance() at 64 x 256 and 32 x 96
    two-level, which switches the handle to the dense kernel instance;
  * the refusals that stay."""
import numpy as np
import pytest
import torch

import bench_problems as bp
import diag_reference as dr
import pooled_samples_reference as psr
from support import check_closed_form, ensemble, linear_chain
from yagre_mcmc_b200 import _lib
from yagre_mcmc_b200.ensemble import pooled_sample_stats, iat_ess
from yagre_mcmc_b200.parallel import moments_from_stats
from yagre_mcmc_b200.parameter import ParameterVector

pytestmark = pytest.mark.gpu


def _stats(x):
    return pooled_sample_stats(torch.from_numpy(np.ascontiguousarray(x)).cuda()).cpu().numpy()


def _data(rng, ns, d, nc, offset=0.0):
    return (offset + rng.standard_normal((ns, d, nc)) * rng.uniform(0.2, 2.0, (1, d, 1))
            + rng.standard_normal((1, d, nc)))


def _check_moments(v, x, label):
    """moments_from_stats of the vector against the long-double pooled moments (check_pooled's POOLED_RTOL)."""
    ns, d, nc = x.shape
    if ns * nc < 2:
        return
    pm = moments_from_stats(v, d)
    mu, cov = psr.pooled_moments(x)
    amax = np.abs(x).max(axis=(0, 2))
    assert np.all(np.abs(pm["mean"] - mu) <= dr.POOLED_RTOL * amax), (label, "mean")
    sd = np.sqrt(np.diag(cov))
    assert np.all(np.abs(pm["covariance"] - cov) <= dr.POOLED_RTOL * np.outer(sd, sd)), (label, "covariance")


@pytest.mark.parametrize("d", [1, 2, 3, 8, 9, 16, 17, 33, 63, 64])
def test_vector_against_long_double_reference(d):
    rng = np.random.default_rng(100 + d)
    worst = 0.0
    for ns in (1, 2, 5, 40):
        for nc in (1, 3, 8, 9, 1000):
            x = _data(rng, ns, d, nc)
            v = _stats(x)
            label = f"d={d} ns={ns} nc={nc}"
            worst = max(worst, psr.check_vector(v, x, label))
            _check_moments(v, x, label)
    assert worst <= 1.0


def test_large_ensemble_offset_data_and_repeatability():
    rng = np.random.default_rng(7)
    x = _data(rng, 5, 17, 65536)
    s = torch.from_numpy(x).cuda()
    v1, v2 = pooled_sample_stats(s), pooled_sample_stats(s)
    assert torch.equal(v1, v2)                                          # fixed-order sums: bitwise repeatable
    psr.check_vector(v1.cpu().numpy(), x, "65536 chains")
    _check_moments(v1.cpu().numpy(), x, "65536 chains")
    # a common offset of 1e4: raw moments would miss the M2 bound by orders of magnitude (test_pooled_samples_cpu)
    x = _data(rng, 40, 9, 1000, offset=1e4)
    psr.check_vector(_stats(x), x, "offset 1e4")


def _welford_vector_bound(pre):
    """Bound on |yg_pooled_stats - truth| for entries 3: of the vector, from the Welford bounds of every chain
    (diag_reference.welford_tolerance) plus the n_chains-term sums over chains."""
    nc, n, d = pre.shape
    mu, R = dr.welford_reference(pre)
    tm, t2 = dr.welford_tolerance(pre, (mu, R))
    mu, R = np.abs(mu.astype(np.float64)), np.abs(R.astype(np.float64))
    g = psr.gamma(nc + 1)
    t_mean = tm.sum(0) + g * (mu + tm).sum(0)
    t_mm = (np.einsum('ci,cj->ij', mu, tm) + np.einsum('ci,cj->ij', tm, mu) + np.einsum('ci,cj->ij', tm, tm)
            + g * np.einsum('ci,cj->ij', mu + tm, mu + tm))
    t_m2 = t2.sum(0) + g * (R + t2).sum(0)
    t_var = (np.einsum('cii->i', t2) + g * np.einsum('cii->i', R + t2)) / (n - 1)
    return np.concatenate([t_mean, t_mm.ravel(), t_m2.ravel(), t_var])


@pytest.mark.parametrize("case", ["gauss2d", "lv_two_level"])
def test_agrees_with_welford_path_on_pre_transition_states(case):
    """The Welford states of a run are its pre-transition states theta_0 .. theta_{n-1}, i.e. the stored trajectory
    (initial state first) without its last state.  The sample vector of that slice and yg_pooled_stats must each be
    within their own bound of the same long-double truth."""
    if case == "gauss2d":
        (meta, arrays), nc, ns = bp.gauss2d_problem(), 1000, 200
        th0 = bp.GAUSS2D_MEAN + np.random.default_rng(3).standard_normal((nc, 2))
    else:
        (meta, arrays), nc, ns = bp.lv_problem(True), 256, 40
        th0 = bp.lv_initial_states(nc)
    ens = ensemble(meta, arrays, nc, seed=21)
    ens.set_state(th0)
    samples = ens.run(ns, samples=True)["samples"]
    traj = torch.cat([torch.from_numpy(th0.T.copy()).cuda()[None], samples])
    pre = traj[:-1].contiguous()
    x = pre.cpu().numpy()
    v = pooled_sample_stats(pre).cpu().numpy()
    assert psr.check_vector(v, x, case) <= 1.0
    st = {k: val.cpu().numpy() if torch.is_tensor(val) else val for k, val in ens.state().items()}
    assert st["welford_n"] == ns
    w = ens.pooled_stats().cpu().numpy()
    pre_c = x.transpose(2, 0, 1)                                        # [nc, n, d]
    dr.check_pooled(w, st, st["welford_n"], pre_c, case)
    ref, _ = psr.reference(x)
    err = np.abs(w[3:].astype(np.longdouble) - ref[3:]).astype(np.float64)
    assert np.all(err <= _welford_vector_bound(pre_c)), (case, "yg_pooled_stats vs the sample truth")
    assert w[0] == v[0] == nc and w[1] == v[1] == ns


def _rhat_restated(vec, d):
    v = np.asarray(vec, dtype=np.float64)
    C, n = v[0], v[1]
    s_mean, s_mm = v[3:3 + d], v[3 + d:3 + d + d * d].reshape(d, d)
    s_var = v[3 + d + 2 * d * d:]
    W = s_var / C
    between = np.diag(s_mm) - s_mean * s_mean / C
    return np.sqrt(((n - 1) / n * W + between / (C - 1)) / W)


@pytest.mark.parametrize("case", ["single_64x256", "two_level_32x96"])
def test_tensor_path_pooling_through_the_builders(case):
    d, dd, two = (64, 256, False) if case == "single_64x256" else (32, 96, True)
    C, thin, n1, n2 = 4096, 10, 1001, 10001
    rng = np.random.default_rng(17)
    mc, (mean, cov) = linear_chain(d, dd, two, C, seed=5, thin=thin)
    iso, _ = linear_chain(d, dd, two, C, seed=5, thin=thin)
    draws1, draws2 = rng.multivariate_normal(mean, cov, size=C), rng.multivariate_normal(mean, cov, size=C)

    mc.run(n1, ParameterVector(draws1), verbose=False)
    traj = mc.chain.trajectory.device_tensor
    assert traj.shape == (1 + (n1 - 1) // thin, d, C)
    out = mc.pooled()
    c = mc.ensemble.counters()
    assert out["n_chains"] == C and out["samples_per_chain"] == traj.shape[0]
    assert abs(out["acceptance_rate"] - c["accepted"] / c["transitions"]) < 1e-12
    check_closed_form(out, mean, cov, C, case + " isotropic")
    vec = pooled_sample_stats(traj).cpu().numpy()
    np.testing.assert_allclose(out["rhat"], _rhat_restated(vec, d), rtol=1e-10)

    pooled = mc.pool_proposal_covariance()
    L = pooled["prop_L"]
    assert np.count_nonzero(np.tril(L, -1)) > 0
    np.testing.assert_array_equal(mc.ensemble.problem.arrays["prop_L"], L)
    mc.run(n2, ParameterVector(draws2), verbose=False)
    if d == 64:
        assert mc.ensemble.last_launch()["block"] == 4 * 32          # the dense-factor instance
    out2 = mc.pooled()
    check_closed_form(out2, mean, cov, C, case + " pooled dense")
    iat_dense = np.median(iat_ess(mc.chain.trajectory.device_tensor)[0].cpu().numpy())

    iso.run(n1, ParameterVector(draws1), verbose=False)
    iso.run(n2, ParameterVector(draws2), verbose=False)
    iat_iso = np.median(iat_ess(iso.chain.trajectory.device_tensor)[0].cpu().numpy())
    # Sokal's window M >= 5 tau must close inside the series for the IATs to be estimates at all
    assert 1 < iat_dense < iat_iso < (1 + (n2 - 1) // thin) / 5, (case, iat_dense, iat_iso)


def test_refusals():
    mc, (mean, _) = linear_chain(64, 256, False, 64, seed=1, thin=5, store=False)
    mc.run(11, ParameterVector(mean), verbose=False)
    with pytest.raises(NotImplementedError, match="storeTrajectory"):
        mc.pooled()
    with pytest.raises(NotImplementedError, match="storeTrajectory"):
        mc.pool_proposal_covariance()
    with pytest.raises(NotImplementedError):                          # still no full second moment on the tensor path
        mc.ensemble.pooled_stats()
    stored, _ = linear_chain(64, 256, False, 64, seed=1, thin=5)
    with pytest.raises(NotImplementedError, match="storeTrajectory"):  # nothing run yet
        stored.pooled()
    stored.run(11, ParameterVector(mean), verbose=False)
    stored.clear()
    with pytest.raises(NotImplementedError, match="storeTrajectory"):  # trajectory cleared
        stored.pooled()
    with pytest.raises(ValueError):
        stored.ensemble.rebuild_proposal_factor(np.ones((64, 64)))     # not lower triangular
    pcn, (mean, _) = linear_chain(32, 96, False, 64, seed=1, thin=5, pcn=True)
    pcn.run(11, ParameterVector(mean), verbose=False)
    with np.errstate(divide="ignore", invalid="ignore"):             # R-hat of chains that have not moved: 0 / 0
        assert pcn.pooled()["n_chains"] == 64
        with pytest.raises(NotImplementedError):                      # the pCN factor is the prior's
            pcn.pool_proposal_covariance()
    with pytest.raises(NotImplementedError):
        pcn.ensemble.set_proposal_factor(np.eye(32))
    with pytest.raises(ValueError):
        pooled_sample_stats(torch.zeros(3, 65, 4, dtype=torch.float64))   # host tensor
    with pytest.raises(NotImplementedError):
        pooled_sample_stats(torch.zeros(3, 65, 4, dtype=torch.float64, device="cuda"))
    assert _lib.YG_BIG_MAX_DIM == 64
