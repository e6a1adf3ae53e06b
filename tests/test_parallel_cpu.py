"""CPU, world_size 2 over gloo: the N > 1 host path.  Chains shard by contiguous global-id ranges
with no data-path collective; the only exchange is an all-reduce(sum) of the sufficient-statistics
vector (yagre_mcmc_b200/parallel.py).  The device kernels that PRODUCE the per-rank vectors are
covered by the -m gpu tests; here the per-rank vectors are built with numpy in yg_pooled_stats'
layout so that the reduction, the restore of the per-chain sample count and the R-hat algebra
are exercised across two real processes."""
import os

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from support import free_port
from yagre_mcmc_b200.parallel import (shard_range, all_reduce_stats, moments_from_stats,
                                      split_rhat_from_moments, pooled_proposal_covariance)


class _RankEnsemble:
    """Stands in for ChainEnsemble on CPU: the statistics vector of this rank's chains and a recorder for
    the proposal factor (the device side, yg_pooled_stats / yg_set_proposal_factor, is covered by -m gpu)."""

    def __init__(self, vec, d):
        self._vec, self.dim, self.L = vec, d, None

    def pooled_stats(self):
        return self._vec.clone()

    def set_proposal_factor(self, L):
        self.L = np.array(L)


def _ensemble(seed=3, C=48, n=400, d=2):
    rng = np.random.default_rng(seed)
    return (rng.standard_normal((C, n, d)) * np.array([1.0, 2.5]) + np.array([0.4, -1.0])
            + 0.3 * rng.standard_normal((C, 1, d)))


def _stats_vector(x, n_accept):
    """numpy restatement of yg_pooled_stats' layout for chains x[C, n, d]."""
    C, n, d = x.shape
    mean_c = x.mean(axis=1)
    dx = x - mean_c[:, None]
    m2_c = np.einsum('cni,cnj->cij', dx, dx)
    var_c = x.var(axis=1, ddof=1)
    return np.concatenate([[C, n, float(n_accept)], mean_c.sum(0), np.einsum('ci,cj->ij', mean_c, mean_c).ravel(),
                           m2_c.sum(0).ravel(), var_c.sum(0)])


def _worker(rank, world, port, q):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        x = _ensemble()
        lo, hi = shard_range(x.shape[0], rank, world)
        vec = torch.from_numpy(_stats_vector(x[lo:hi], 100 * (hi - lo) + rank))
        out = moments_from_stats(all_reduce_stats(vec), x.shape[2])
        half = x.shape[1] // 2
        xs = x[lo:hi]
        hm = torch.from_numpy(np.stack([xs[:, :half].mean(1).T, xs[:, half:2 * half].mean(1).T]))
        hv = torch.from_numpy(np.stack([xs[:, :half].var(1, ddof=1).T, xs[:, half:2 * half].var(1, ddof=1).T]))
        rh = split_rhat_from_moments(hm, hv, half)
        ens = _RankEnsemble(torch.from_numpy(_stats_vector(x[lo:hi], 100 * (hi - lo) + rank)), x.shape[2])
        pooled = pooled_proposal_covariance(ens, eps=1e-6)
        out["prop_L"], out["prop_L_set"] = pooled["prop_L"], ens.L
        q.put((rank, lo, hi, out, rh))
    finally:
        dist.destroy_process_group()


@pytest.mark.timeout(180)
def test_two_rank_pooling_equals_single_process():
    world, port = 2, free_port()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_worker, args=(r, world, port, q)) for r in range(world)]
    for p in procs:
        p.start()
    res = sorted([q.get(timeout=150) for _ in range(world)], key=lambda t: t[0])
    for p in procs:
        p.join(30)
        assert p.exitcode == 0
    x = _ensemble()
    C, n, d = x.shape
    assert res[0][1] == 0 and res[0][2] == res[1][1] and res[1][2] == C        # contiguous, complete shards
    flat = x.reshape(-1, d)
    single = moments_from_stats(_stats_vector(x, 100 * C + 1), d)
    for _, _, _, out, rh in res:                                               # every rank holds the pooled answer
        assert out["n_chains"] == C and out["samples_per_chain"] == n
        np.testing.assert_allclose(out["mean"], flat.mean(0), rtol=1e-12)
        np.testing.assert_allclose(out["covariance"], np.cov(flat.T), rtol=1e-10)
        np.testing.assert_allclose(out["rhat"], single["rhat"], rtol=1e-12)
        assert abs(out["acceptance_rate"] - single["acceptance_rate"]) < 1e-15
        # split R-hat against the textbook formula on 2C half chains
        half = n // 2
        halves = np.concatenate([x[:, :half], x[:, half:2 * half]], axis=0)
        W = halves.var(axis=1, ddof=1).mean(0)
        B_over_n = halves.mean(axis=1).var(axis=0, ddof=1)
        np.testing.assert_allclose(rh, np.sqrt(((half - 1) / half * W + B_over_n) / W), rtol=1e-12)
        # pooled proposal covariance: every rank installs chol(2.4^2/d (Sigma_pooled + eps I))
        want = np.linalg.cholesky(2.4 * 2.4 / d * (np.cov(flat.T) + 1e-6 * np.eye(d)))
        np.testing.assert_allclose(out["prop_L_set"], want, rtol=1e-9)
    np.testing.assert_array_equal(res[0][3]["mean"], res[1][3]["mean"])
    np.testing.assert_array_equal(res[0][3]["prop_L_set"], res[1][3]["prop_L_set"])    # bitwise the same factor
