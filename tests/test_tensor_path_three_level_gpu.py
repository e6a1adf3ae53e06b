"""GPU: MLDA with two surrogates and tempered levels on the FP64 tensor path (linear_dmma_kernel.cu, NL = 3; abi.cu's
tempering fold).

  1. recorded Philox noise replayed through the C oracle: identical accept decisions, trajectories to 1e-12, every
     level's stored log-posterior within the tensor-path bound (three_level_reference.py), coarse / mid / fine
     evaluation counters and accept counts equal to the oracle's; the production instance equals the recording one bit
     for bit (support.check_case);
  2. forced decisions (logpost_reference.forced_schedule, with the tempered tensor bound) at eta = the smallest
     allowed, 1e-7 and 1e-3;
  3. composition: short launches equal one long launch, two handles split by chain_offset equal one, load_state and
     set_state(keep_diagnostics) resume bit for bit with three logpost rows;
  4. chains started from exact draws of mu ~ pi_2 pi_0 / pi_1 keep mu's moments; a tempered surrogate of two levels
     keeps the target's;
  5. the pooled dense factor (rebuild_proposal_factor) on three-level 64 x 256 runs the general streamed instance and
     replays through the oracle;
  6. MLDABuilder with two surrogate targets, one tempered, on a 64-parameter hierarchy."""
import numpy as np
import pytest
import torch

import bench_problems as bp
import logpost_reference as R
from golden_io import rel_err
import three_level_reference as TL
from support import check_case, check_closed_form, ensemble, replay, schedule_noise
from three_level_reference import mlda_invariant_gaussian

pytestmark = pytest.mark.gpu

SHAPES = {
    # name: (d, data_dims, generator kwargs, dense factor)
    "9x20_L0_tempered": (9, (20, 20, 20), dict(tempering={0: 0.5}), False),
    "23x45": (23, (45, 45, 45), {}, False),
    "32x96_dense_prior": (32, (96, 96, 96), dict(dense_prior=True), False),
    "32x256": (32, (256, 256, 256), {}, False),                                 # level 1's G streamed at d <= 32
    "48_40_97_256": (48, (40, 97, 256), {}, False),
    "64x256": (64, (256, 256, 256), {}, False),                                 # G1 and G2 streamed
    "64x256_dense_prior_dense_factor": (64, (256, 256, 256), dict(dense_prior=True), True),
}

TEMPERED = {
    # name: (d, data_dim, levels, tempering of level 0)
    "single_24x40_t0.6": (24, 40, 1, 0.6),
    "single_24x40_t0": (24, 40, 1, 0.0),
    "two_24x40_t0.35": (24, 40, 2, 0.35),
    "two_24x40_t0": (24, 40, 2, 0.0),
}


def problem(name):
    """(meta, arrays, operand rows per level, dense factor)."""
    if name in TEMPERED:
        d, dd, levels, t = TEMPERED[name]
        meta, arrays = bp.big_linear_problem(d, dd, 2, two_level=levels == 2, J=3, seed=17)
        return meta, dict(arrays, L0_tempering=np.array(t)), [dd] * levels, False
    d, dims, kw, dense_L = SHAPES[name]
    meta, arrays = bp.big_linear_three_level_problem(d, dims, 2, J=3, **kw)
    if dense_L:
        _, cov, _ = mlda_invariant_gaussian(arrays, 3)
        arrays = dict(arrays, prop_L=np.linalg.cholesky(2.4 ** 2 / d * 0.3 * cov))
    rows = [dd + (d if kw.get("dense_prior") else 0) for dd in dims]
    return meta, arrays, rows, dense_L


def start(meta, arrays, nc, seed):
    mean, cov, _ = mlda_invariant_gaussian(arrays, meta["levels"])
    return np.random.default_rng(seed).multivariate_normal(mean, cov, size=nc)


def tensor_plan(d, rows, dense_L, welford=True):
    """smem_plan.h's big_tensor_plan restated for up to three levels: (stream bits, warps, dynamic shared memory)."""
    kp = 16 if d <= 16 else (32 if d <= 32 else 64)
    ks, kq = kp + 4, kp // 4
    nps = [(r + 15) & ~15 for r in rows] + [0] * (3 - len(rows))
    raw = sum(n * ks + n + 2 * kp for n in nps if n) + 2 * kp + (kp * ks if dense_L else 0)
    tile, noise = 8 * 8 * ks, 4 * 8 * (4 * kq + 4)
    plain, budget = tile * (2 if dense_L else 1) + noise, 227 * 1024

    def plan(doubles):
        blob = 8 * ((doubles + 1) & ~1)
        warps = min(12 if kq == 16 else 16, max(0, budget - blob) // plain)
        wsm = welford and warps >= 4 and blob + warps * (plain + 2 * tile) <= budget
        return warps, blob + warps * (plain + (2 * tile if wsm else 0))
    stream, staged = 0, raw
    warps, smem = plan(raw)
    for bit, size in ((1, nps[1] * ks), (4, nps[2] * ks), (2, kp * ks if dense_L else 0)):
        if warps >= 4:
            break
        if size:
            stream, staged = stream | bit, staged - size
            warps, smem = plan((staged + 3) & ~3)
    return stream, warps, smem


def traj_err(got, ref, dense_L):
    """As in test_tensor_path_streamed_gpu: relative per coordinate; with a dense factor relative to the larger of the
    value and the coordinate's magnitude over the run (p = s + L z sums in a different order on the two sides)."""
    if not dense_L:
        return rel_err(got, ref).max()
    scale = np.maximum(np.abs(ref), np.abs(ref).max(axis=(0, 1), keepdims=True))
    return float((np.abs(got - ref) / scale).max())


def check_levels(meta, arrays, states, lp, label):
    """states [m, d], lp [m, levels]: every level within the tensor-path bound."""
    for l in range(meta["levels"]):
        want, b = TL.tensor_logpost_bound(meta, arrays, l, states)
        e = np.abs(lp[:, l].astype(np.longdouble) - want).astype(np.float64)
        assert np.all(e <= b), (label, l, float((e / b).max()))


REPLAY = [(n, 33, 1) for n in sorted(SHAPES) + sorted(TEMPERED)] + [
    ("9x20_L0_tempered", 2500, 3), ("23x45", 5, 1), ("32x96_dense_prior", 2500, 1), ("32x256", 2500, 3),
    ("48_40_97_256", 2500, 3), ("64x256", 20011, 1), ("64x256_dense_prior_dense_factor", 2500, 3),
    ("two_24x40_t0.35", 2500, 3), ("single_24x40_t0", 2500, 1)]


@pytest.mark.parametrize("name,nc,thin", REPLAY)
def test_three_level_replay(name, nc, thin):
    meta, arrays, rows, dense_L = problem(name)
    d = meta["dim"]
    stream, warps, smem = tensor_plan(d, rows, dense_L)
    th0 = start(meta, arrays, nc, nc)
    label = f"{name} nc={nc}"
    check_case(meta, arrays, th0, [("run", 1), ("run", 2), ("run", 3)], seed=41, smem=smem, label=label)
    ns = 3 * thin
    ens = ensemble(meta, arrays, nc, seed=43)
    ens.set_state(th0)
    check_levels(meta, arrays, th0, ens.state()["logpost"].cpu().numpy().T, f"{label} set_state")
    out = ens.run(ns, thin=thin, samples=True, accepted=True, logpost=True, record=True)
    torch.cuda.synchronize()
    launch = ens.last_launch()
    assert launch["smem"] == smem and launch["block"] == 32 * warps, (label, launch, stream, warps, smem)
    ref = replay(meta, arrays, th0, out)
    acc = out["accepted"].cpu().numpy().T
    assert np.array_equal(acc, ref["accepted"]), label
    got = out["samples"].cpu().numpy().transpose(2, 0, 1)                      # [nc, ns / thin, d]
    keep = np.arange(thin, ns + 1, thin)
    assert traj_err(got, ref["traj"][:, keep], dense_L) <= 1e-12, label
    lp = out["logpost"].cpu().numpy().transpose(2, 0, 1)                      # [nc, ns / thin, levels]
    assert lp.shape[2] == meta["levels"]
    check_levels(meta, arrays, got.reshape(-1, d), lp.reshape(-1, meta["levels"]), label)
    c = ens.counters()
    ev = [int(v) - nc for v in ref["n_evals"]]
    assert c["transitions"] == acc.size and c["accepted"] == int(acc.sum()), label
    want = {1: dict(fine_evals=ev[0]), 2: dict(coarse_evals=ev[0], fine_evals=ev[1]),
            3: dict(coarse_evals=ev[0], mid_evals=ev[1], fine_evals=ev[2])}[meta["levels"]]
    assert {k: c[k] for k in want} == want, (label, c, want)
    if meta["levels"] >= 2:
        assert c["coarse_accepted"] == int(ref["coarse_accepted"].sum()), label
    if meta["levels"] == 3:
        assert c["mid_evals"] == c["fine_evals"] > 0, label


# ------------------------------------------------------------------------------------------------------------------
# forced decisions
# ------------------------------------------------------------------------------------------------------------------
def _inject(z, sch):
    return dict(z=np.ascontiguousarray(z.transpose(1, 2, 3, 0)), u_c=np.ascontiguousarray(sch["u_c"].transpose(1, 2, 0)),
                u_f=np.ascontiguousarray(sch["u_f"].transpose(1, 0)))


@pytest.mark.parametrize("name", ["9x20_L0_tempered", "32x96_dense_prior", "64x256", "two_24x40_t0.35"])
@pytest.mark.parametrize("eta", [0.0, 1e-7, 1e-3])
def test_three_level_forced_decisions(name, eta, monkeypatch):
    # forced_schedule's tensor-path bounds with the tempering fold (untempered levels: the same function)
    monkeypatch.setattr(R, "_tensor_logpost_and_bound", TL.tensor_logpost_and_bound)
    meta, arrays, _, _ = problem(name)
    nc, ns = 96, 4
    th0 = start(meta, arrays, nc, 7)
    z = schedule_noise(meta, nc, ns, 11)
    sch = R.forced_schedule(meta, arrays, th0, z, R.random_pattern(nc, ns, z.shape[2], seed=13), eta)
    ens = ensemble(meta, arrays, nc, seed=5)
    ens.set_state(th0)
    out = ens.run(ns, samples=True, accepted=True, logpost=True, inject=_inject(z, sch))
    torch.cuda.synchronize()
    acc = out["accepted"].cpu().numpy().T
    assert np.array_equal(acc, sch["accepted"]), (name, eta, np.argwhere(acc != sch["accepted"])[:5])
    c = ens.counters()
    assert np.array_equal(ens.state()["n_accept"].cpu().numpy(), sch["n_accept"])
    assert c["coarse_accepted"] == int(sch["coarse_accepted"].sum())
    assert c["transitions"] == acc.size and c["accepted"] == int(acc.sum())
    ev = sch["evals"]
    want = {2: dict(coarse_evals=ev[0], fine_evals=ev[1]),
            3: dict(coarse_evals=ev[0], mid_evals=ev[1], fine_evals=ev[2])}[meta["levels"]]
    assert {k: c[k] for k in want} == {k: int(v) for k, v in want.items()}, (c, want)
    assert 0.05 < acc.mean() < 0.95


# ------------------------------------------------------------------------------------------------------------------
# composition
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["64x256", "32x256", "9x20_L0_tempered"])
def test_three_level_launches_compose(name):
    meta, arrays, _, _ = problem(name)
    for nc in (5, 2500, 20011):
        th0 = start(meta, arrays, nc, nc)
        a = ensemble(meta, arrays, nc, seed=2)
        a.set_state(th0)
        whole = a.run(6, samples=True, accepted=True, logpost=True)
        b = ensemble(meta, arrays, nc, seed=2)
        b.set_state(th0)
        parts = [b.run(k, samples=True, accepted=True, logpost=True) for k in (1, 2, 3)]
        for k in ("samples", "accepted", "logpost"):
            assert torch.equal(whole[k], torch.cat([p[k] for p in parts])), (nc, k)
        sa, sb = a.state(), b.state()
        assert sa["logpost"].shape == (3, nc)
        for k in ("theta", "logpost", "n_accept"):
            assert torch.equal(sa[k], sb[k]), (nc, k)
        sa_counts = a.counters()
        assert sa_counts == b.counters()
        # two handles split by chain_offset
        off = nc // 3
        split = []
        for lo, hi in ((0, off), (off, nc)):
            if hi > lo:
                e = ensemble(meta, arrays, hi - lo, seed=2, chain_offset=lo)
                e.set_state(th0[lo:hi])
                split.append(e.run(6, samples=True, accepted=True, logpost=True))
        for k in ("samples", "accepted", "logpost"):
            assert torch.equal(torch.cat([p[k] for p in split], dim=-1), whole[k]), (nc, k)
        # load_state into a fresh handle after 3 transitions resumes the 6-transition run
        c = ensemble(meta, arrays, nc, seed=2)
        c.set_state(th0)
        c.run(3, samples=False)
        f = ensemble(meta, arrays, nc, seed=2)
        f.load_state(c.state())
        rest = f.run(3, samples=True, accepted=True, logpost=True)
        for k in ("samples", "accepted", "logpost"):
            assert torch.equal(rest[k], whole[k][3:]), (nc, k)
        assert torch.equal(f.state()["logpost"], sa["logpost"])
        # set_state(keep_diagnostics) = a fresh handle set to the same state at the same stream position
        x = sa["theta"].t().cpu().numpy()
        a.set_state(x, keep_diagnostics=True)
        g = ensemble(meta, arrays, nc, seed=2)
        g.set_state(x, step_index=6)
        assert torch.equal(a.state()["logpost"], g.state()["logpost"])
        ra, rg = a.run(4, samples=True, accepted=True, logpost=True), g.run(4, samples=True, accepted=True, logpost=True)
        for k in ("samples", "accepted", "logpost"):
            assert torch.equal(ra[k], rg[k]), (nc, k)
        ca, cg = a.counters(), g.counters()
        assert ca["transitions"] == 10 * nc and cg["transitions"] == 4 * nc       # the diagnostics were kept
        for k in ("mid_evals", "fine_evals", "coarse_evals", "accepted"):
            assert ca[k] == sa_counts[k] + cg[k], (nc, k)
        for e in (a, b, c, f, g):
            e.close()


# ------------------------------------------------------------------------------------------------------------------
# statistics
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["64x256", "32x96_dense_prior"])
def test_three_level_invariant_law(name):
    """Chains started from exact draws of mu ~ pi_2 pi_0 / pi_1 stay there."""
    meta, arrays, _, _ = problem(name)
    d, C = meta["dim"], 4096
    mean, cov, _ = mlda_invariant_gaussian(arrays, 3)
    ens = ensemble(meta, arrays, C, seed=8)
    ens.set_state(start(meta, arrays, C, 19))
    s = ens.run(2000, thin=20, samples=True)["samples"].cpu().numpy()         # [100, d, C]
    flat = s.transpose(0, 2, 1).reshape(-1, d)
    check_closed_form(dict(mean=flat.mean(0), covariance=np.cov(flat.T)), mean, cov, C, name)
    c = ens.counters()
    assert 0.05 < c["accepted"] / c["transitions"] < 0.95
    assert c["mid_evals"] == c["fine_evals"] < c["coarse_evals"]


def test_tempered_surrogate_keeps_the_target():
    """Two levels, level 0 tempered at 0.35: delayed acceptance stays exact for the (untempered) target."""
    meta, arrays, _, _ = problem("two_24x40_t0.35")
    C = 4096
    mean, cov = bp.linear_gaussian_posterior(arrays, 1)
    ens = ensemble(meta, arrays, C, seed=9)
    ens.set_state(np.random.default_rng(4).multivariate_normal(mean, cov, size=C))
    s = ens.run(2000, thin=20, samples=True)["samples"].cpu().numpy()
    flat = s.transpose(0, 2, 1).reshape(-1, 24)
    check_closed_form(dict(mean=flat.mean(0), covariance=np.cov(flat.T)), mean, cov, C, "tempered surrogate")


# ------------------------------------------------------------------------------------------------------------------
# the pooled dense factor on three levels
# ------------------------------------------------------------------------------------------------------------------
def test_three_level_rebuild_to_a_dense_factor():
    meta, arrays, rows, _ = problem("64x256")
    nc = 2500
    ens = ensemble(meta, arrays, nc, seed=3)
    ens.set_state(start(meta, arrays, nc, 3))
    ens.run(5, samples=False)
    _, cov, _ = mlda_invariant_gaussian(arrays, 3)
    L = np.linalg.cholesky(2.4 ** 2 / 64 * 0.3 * cov)
    ens.rebuild_proposal_factor(L)
    th0 = ens.state()["theta"].cpu().numpy().T.copy()
    out = ens.run(4, samples=True, accepted=True, logpost=True, record=True)
    torch.cuda.synchronize()
    stream, warps, smem = tensor_plan(64, rows, True)
    assert stream != 0 and ens.last_launch()["smem"] == smem and ens.last_launch()["block"] == 32 * warps
    p = ens.problem
    ref = replay(meta, p.arrays, th0, out)
    acc = out["accepted"].cpu().numpy().T
    assert np.array_equal(acc, ref["accepted"]) and 0.05 < acc.mean() < 0.95
    assert traj_err(out["samples"].cpu().numpy().transpose(2, 0, 1), ref["traj"][:, 1:], True) <= 1e-12
    lp = out["logpost"].cpu().numpy().transpose(2, 0, 1)
    for l in range(3):
        assert rel_err(lp[:, :, l], ref[f"logpost_L{l}"][:, 1:]).max() <= 1e-10, l


# ------------------------------------------------------------------------------------------------------------------
# public API
# ------------------------------------------------------------------------------------------------------------------
def test_mlda_two_surrogates_one_tempered_through_the_builder():
    from yagre_mcmc_b200.parameter import ParameterVector
    from yagre_mcmc_b200.model import ForwardModel, LinearModelSolver
    from yagre_mcmc_b200.statistics import (IIDCovarianceMatrix, Gaussian, CentredGaussianNoise, Data,
                                            AdditiveGaussianNoiseLikelihood)
    from yagre_mcmc_b200.chain.method import MLDABuilder
    from yagre_mcmc_b200.chain.target import UnnormalisedPosterior, TemperedUnnormalisedPosterior
    d, dims = 64, (256, 256, 256)
    meta, a = bp.big_linear_three_level_problem(d, dims, 1, J=3, tempering={1: 0.9})
    prior = Gaussian(ParameterVector(np.zeros(d)), IIDCovarianceMatrix(d, 2.0))
    lik = [AdditiveGaussianNoiseLikelihood(Data(a[f"L{l}_data"]), ForwardModel(LinearModelSolver(a[f"L{l}_G"], a[f"L{l}_b"])),
                                           CentredGaussianNoise(IIDCovarianceMatrix(dd, 0.05)))
           for l, dd in enumerate(dims)]
    b = MLDABuilder()
    b.explicitTarget = UnnormalisedPosterior(lik[2], prior)
    b.surrogateTargets = [UnnormalisedPosterior(lik[0], prior), TemperedUnnormalisedPosterior(lik[1], prior, 0.9)]
    b.baseProposalCovariance = IIDCovarianceMatrix(d, 0.25 * float(a["prop_L"][0, 0]) ** 2)
    b.subChainLengths = [3, 3]
    b.nChains, b.seed, b.storeTrajectory = 4096, 21, False
    mc = b.build_method()
    assert mc.nSurrogates == 2 and mc.ensemble.levels == 3
    mean, cov, _ = mlda_invariant_gaussian(a, 3)
    mc.run(300, ParameterVector(np.random.default_rng(1).multivariate_normal(mean, cov, size=4096)), verbose=False)
    assert 0.1 < mc.diagnostics.global_acceptance_rate() < 0.9
    c = mc.ensemble.counters()
    assert c["mid_evals"] == c["fine_evals"] > 0 and c["coarse_evals"] > c["fine_evals"]
