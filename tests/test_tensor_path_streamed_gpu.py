"""GPU: the tensor path on shapes whose blob does not fit shared memory, with operands streamed from L2
(smem_plan.h: big_tensor_plan; linear_dmma_kernel.cu: logpost_tile_streamed, lz_streamed).

  1. recorded noise replayed through the C oracle: identical accept decisions, trajectories to 1e-12, both levels'
     log-posteriors to 1e-10, the counters and the per-chain accept counts exactly, the Welford moments within
     tests/diag_reference.py's bounds;
  2. the production instance (Philox) equals the recording one bit for bit, and chains split over two handles with
     chain_offset equal the same chains of one handle;
  3. launches of 1 + 2 + 3 transitions compose to one of 6 bit for bit (tile hand-overs with streamed operands);
  4. yg_logpost and the kernel's log-posteriors within the long-double bound of tests/logpost_reference.py;
  5. two-level 64 x 256 samples the fine level's closed-form posterior;
  6. the builders: isotropic burn-in -> pool_proposal_covariance() -> run on a two-level 64 x 160 model;
  7. the launch report (dynamic shared memory, block size) is the plan's."""
import numpy as np
import pytest
import torch

import bench_problems as bp
from golden_io import rel_err
from support import LOGPOST_RTOL, check_case, check_closed_form, ensemble, linear_chain, replay, value_case
from yagre_mcmc_b200.parameter import ParameterVector

pytestmark = pytest.mark.gpu

def traj_err(got, ref, dense_L):
    """Trajectory error: relative per coordinate; with a dense factor relative to the larger of the value and the
    coordinate's magnitude over the run.  p = s + L z sums d products that the device forms in DMMA order and the oracle
    in its own: where the sum nearly cancels, the per-element relative error of the state is unbounded though its error
    is a few ulps of the coordinate's scale."""
    if not dense_L:
        return rel_err(got, ref).max()
    scale = np.maximum(np.abs(ref), np.abs(ref).max(axis=(0, 1), keepdims=True))
    return float((np.abs(got - ref) / scale).max())


def tensor_plan(d, rows, dense_L, welford=True):
    """smem_plan.h's big_tensor_plan restated: (stream bits, warps, dynamic shared memory) for a model with d parameters
    and `rows` operand rows per level (data_dim, + d for a dense prior)."""
    kp = 16 if d <= 16 else (32 if d <= 32 else 64)
    ks, kq = kp + 4, kp // 4
    nps = [(r + 15) & ~15 for r in rows]
    raw = sum(np_ * ks + np_ + 2 * kp for np_ in nps) + 2 * kp + (kp * ks if dense_L else 0)
    tile, noise = 8 * 8 * ks, 4 * 8 * (4 * kq + 4)
    plain, budget = tile * (2 if dense_L else 1) + noise, 227 * 1024

    def plan(doubles):
        blob = 8 * ((doubles + 1) & ~1)
        warps = min(12 if kq == 16 else 16, max(0, budget - blob) // plain)
        wsm = welford and warps >= 4 and blob + warps * (plain + 2 * tile) <= budget
        return warps, blob + warps * (plain + (2 * tile if wsm else 0))
    stream, staged = 0, raw
    warps, smem = plan(raw)
    for bit, size in ((1, nps[1] * ks if len(nps) == 2 else 0), (2, kp * ks if dense_L else 0)):
        if warps >= 4:
            break
        if size:
            stream, staged = stream | bit, staged - size
            warps, smem = plan((staged + 3) & ~3)
    return stream, warps, smem


def _problem(name):
    """The streamed shapes: (meta, arrays, operand rows per level, dense factor)."""
    d, dd, two, dense_L, dense_prior = STREAMED[name]
    meta, arrays = bp.big_linear_problem(d, dd, 2, two_level=two, J=3, seed=7)
    arrays = dict(arrays)
    rng = np.random.default_rng(d * 1000 + dd)
    if dense_L or dense_prior:
        A = rng.standard_normal((d, d))
        cov = A @ A.T / d + 0.5 * np.eye(d)
    if dense_L:
        arrays["prop_L"] = np.linalg.cholesky(2.4 ** 2 / d * 0.02 * cov)
    if dense_prior:
        prec = np.linalg.inv(2.0 * cov)
        for l in range(meta["levels"]):
            arrays[f"L{l}_prior_prec"] = 0.5 * (prec + prec.T)
            arrays[f"L{l}_prior_mean"] = 0.1 * rng.standard_normal(d)
    rows = [dd + (d if dense_prior else 0)] * meta["levels"]
    return meta, arrays, rows, dense_L


STREAMED = {
    # name: (d, data_dim, two level, dense factor, dense prior)
    "two_64x256": (64, 256, True, False, False),
    "two_64x200_dense_factor": (64, 200, True, True, False),
    "two_48x140_dense_factor_dense_prior": (48, 140, True, True, True),
    "two_33x177": (33, 177, True, False, False),
    "single_64x256_dense_factor_dense_prior": (64, 256, False, True, True),
}

REPLAY = [("two_64x256", 1, 1), ("two_64x256", 2500, 3), ("two_64x256", 20011, 1),
          ("two_64x200_dense_factor", 7, 3), ("two_64x200_dense_factor", 2500, 1),
          ("two_48x140_dense_factor_dense_prior", 33, 1), ("two_48x140_dense_factor_dense_prior", 2500, 3),
          ("two_33x177", 7, 1), ("two_33x177", 20011, 3),
          ("single_64x256_dense_factor_dense_prior", 1, 3), ("single_64x256_dense_factor_dense_prior", 33, 1),
          ("single_64x256_dense_factor_dense_prior", 2500, 3)]


@pytest.mark.parametrize("name,nc,thin", REPLAY)
def test_streamed_replay_counters_and_diagnostics(name, nc, thin):
    meta, arrays, rows, dense_L = _problem(name)
    d = meta["dim"]
    stream, warps, smem = tensor_plan(d, rows, dense_L)
    assert stream != 0, name                                         # the shape does stream
    th0 = 0.01 * np.random.default_rng(nc).standard_normal((nc, d))
    label = f"{name} nc={nc}"
    # production == recording instance, counters / n_accept / coarse_accepted against the oracle, Welford, the launch
    check_case(meta, arrays, th0, [("run", 1), ("run", 2), ("run", 3)], seed=41, smem=smem, label=label)
    # a thinned recorded run replayed through the oracle
    ns = 3 * thin
    ens = ensemble(meta, arrays, nc, seed=43)
    ens.set_state(th0)
    out = ens.run(ns, thin=thin, samples=True, accepted=True, logpost=True, record=True)
    torch.cuda.synchronize()
    launch = ens.last_launch()
    assert launch["smem"] == smem and launch["block"] == 32 * warps, (label, launch, warps, smem)
    ref = replay(meta, arrays, th0, out)
    acc = out["accepted"].cpu().numpy().T
    assert np.array_equal(acc, ref["accepted"]), label
    got = out["samples"].cpu().numpy().transpose(2, 0, 1)           # [nc, ns / thin, d]
    keep = np.arange(thin, ns + 1, thin)                              # reference rows: the initial state, then every step
    assert traj_err(got, ref["traj"][:, keep], dense_L) <= 1e-12, label
    lp = out["logpost"].cpu().numpy().transpose(2, 0, 1)             # [nc, ns / thin, levels]
    for l in range(meta["levels"]):
        key = f"logpost_L{l}"
        assert rel_err(lp[:, :, l], ref[key][:, keep]).max() <= LOGPOST_RTOL, (label, key)
    c = ens.counters()
    ev = [int(v) - nc for v in ref["n_evals"]]
    assert c["transitions"] == acc.size and c["accepted"] == int(acc.sum()), label
    if meta["levels"] == 2:
        assert (c["coarse_evals"], c["fine_evals"]) == (ev[0], ev[1]), label
        assert c["coarse_accepted"] == int(ref["coarse_accepted"].sum()), label
    else:
        assert c["fine_evals"] == ev[0], label


@pytest.mark.parametrize("name", ["two_64x256", "single_64x256_dense_factor_dense_prior"])
def test_streamed_philox_equals_recorded_and_shards(name):
    meta, arrays, rows, _ = _problem(name)
    d, nc, ns = meta["dim"], 20000, 7
    th0 = 0.01 * np.random.default_rng(3).standard_normal((nc, d))
    runs = []
    for record in (False, True):
        ens = ensemble(meta, arrays, nc, seed=12)
        ens.set_state(th0)
        runs.append((ens.run(ns, samples=True, accepted=True, logpost=True, record=record), ens.state(), ens.counters()))
    for k in ("samples", "accepted", "logpost"):
        assert torch.equal(runs[0][0][k], runs[1][0][k]), k
    for k in ("theta", "logpost", "n_accept", "w_mean", "w_m2"):
        assert torch.equal(runs[0][1][k], runs[1][1][k]), k
    assert runs[0][2] == runs[1][2]
    off = 8000
    parts = []
    for lo, hi in ((0, off), (off, nc)):
        sub = ensemble(meta, arrays, hi - lo, seed=12, chain_offset=lo)
        sub.set_state(th0[lo:hi])
        parts.append(sub.run(ns, samples=True, accepted=True, logpost=True))
    for k in ("samples", "accepted", "logpost"):
        assert torch.equal(torch.cat([p[k] for p in parts], dim=-1), runs[0][0][k]), k


def test_streamed_short_launches_compose():
    meta, arrays, _, _ = _problem("two_64x256")
    for nc in (5, 2500, 20011):
        th0 = 0.01 * np.random.default_rng(nc).standard_normal((nc, 64))
        a = ensemble(meta, arrays, nc, seed=2)
        a.set_state(th0)
        whole = a.run(6, samples=True, accepted=True, logpost=True)
        b = ensemble(meta, arrays, nc, seed=2)
        b.set_state(th0)
        parts = [b.run(k, samples=True, accepted=True, logpost=True) for k in (1, 2, 3)]
        for k in ("samples", "accepted", "logpost"):
            assert torch.equal(whole[k], torch.cat([p[k] for p in parts])), (nc, k)
        sa, sb = a.state(), b.state()
        assert torch.equal(sa["theta"], sb["theta"]) and torch.equal(sa["n_accept"], sb["n_accept"])
        np.testing.assert_allclose(sa["w_mean"].cpu().numpy(), sb["w_mean"].cpu().numpy(), rtol=1e-11, atol=1e-14)
        assert a.counters() == b.counters()


@pytest.mark.parametrize("name", ["two_64x256", "two_48x140_dense_factor_dense_prior",
                                  "single_64x256_dense_factor_dense_prior"])
def test_streamed_logpost_values(name):
    meta, arrays, _, _ = _problem(name)
    value_case(meta, arrays, 0.01 * np.random.default_rng(4).standard_normal((2500, meta["dim"])), sample=512)


def test_streamed_two_level_posterior_moments():
    """Delayed acceptance is exact: chains started from draws of the fine level's posterior stay there."""
    meta, arrays = bp.big_linear_problem(64, 256, 1, two_level=True, J=3)
    mean, cov = bp.linear_gaussian_posterior(arrays, 1)
    C = 4096
    th0 = np.random.default_rng(19).multivariate_normal(mean, cov, size=C)
    ens = ensemble(meta, arrays, C, seed=8)
    ens.set_state(th0)
    s = ens.run(2000, thin=20, samples=True)["samples"].cpu().numpy()     # [100, d, C]
    flat = s.transpose(0, 2, 1).reshape(-1, 64)
    check_closed_form(dict(mean=flat.mean(0), covariance=np.cov(flat.T)), mean, cov, C, "two_64x256")
    c = ens.counters()
    assert 0.05 < c["accepted"] / c["transitions"] < 0.95 and c["fine_evals"] < c["coarse_evals"]


def test_streamed_pooled_factor_through_the_builders():
    """Two-level 64 x 160: the isotropic burn-in runs with the whole blob in shared memory; pooling switches the handle
    to the dense factor, whose blob no longer fits (its rebuild was refused while it had to) and streams level 1's G;
    the run after it samples the posterior and replays through the oracle."""
    C, thin = 4096, 10
    mc, (mean, cov) = linear_chain(64, 160, True, C, seed=5, thin=thin)
    draws = np.random.default_rng(23).multivariate_normal(mean, cov, size=C)
    mc.run(501, ParameterVector(draws), verbose=False)
    pooled = mc.pool_proposal_covariance()
    assert np.count_nonzero(np.tril(pooled["prop_L"], -1)) > 0
    ens = mc.ensemble
    stream, warps, smem = tensor_plan(64, [160, 160], True)
    assert stream == 1
    mc.run(1001, ParameterVector(draws), verbose=False)
    assert ens.last_launch()["smem"] == smem and ens.last_launch()["block"] == 32 * warps
    check_closed_form(mc.pooled(), mean, cov, C, "pooled dense factor")
    # a short recorded run on the pooled factor, replayed through the oracle
    th0 = ens.state()["theta"].cpu().numpy().T.copy()
    out = ens.run(4, samples=True, accepted=True, logpost=True, record=True)
    torch.cuda.synchronize()
    p = ens.problem
    meta = dict(model=p.model, dim=p.dim, levels=p.levels, J=p.J, eq=p.eq)
    ref = replay(meta, p.arrays, th0, out)
    assert np.array_equal(out["accepted"].cpu().numpy().T, ref["accepted"])
    assert traj_err(out["samples"].cpu().numpy().transpose(2, 0, 1), ref["traj"][:, 1:], True) <= 1e-12
    lp = out["logpost"].cpu().numpy().transpose(2, 0, 1)
    assert rel_err(lp[:, :, 1], ref["logpost_L1"][:, 1:]).max() <= LOGPOST_RTOL


def test_every_envelope_problem_is_accepted():
    """yg_set_problem takes every linear problem up to 64 x 256, one or two levels, dense and diagonal prior and
    factor."""
    for d, dd in ((64, 256), (33, 256), (64, 1), (48, 241)):
        for two in (False, True):
            for dense_L in (False, True):
                for dense_prior in (False, True):
                    meta, arrays = bp.big_linear_problem(d, dd, 1, two_level=two, J=2)
                    arrays = dict(arrays)
                    if dense_L:
                        arrays["prop_L"] = np.tril(np.full((d, d), 0.001)) + 0.01 * np.eye(d)
                    if dense_prior:
                        for l in range(meta["levels"]):
                            arrays[f"L{l}_prior_prec"] = 0.5 * np.eye(d) + 0.01
                    ens = ensemble(meta, arrays, 17, seed=1)
                    ens.set_state(np.zeros((17, d)))
                    ens.run(2, samples=False)
                    ens.close()
