"""Multi-GPU: chains shard trivially (one process per GPU, torch.distributed / NCCL over NVLink);
the ONLY collective on the path is an all-reduce(sum) of a few dozen doubles of sufficient
statistics, from which pooled moments, the pooled acceptance rate and R-hat follow.
Nothing like this exists in the reference (single chain, single process): parity of R-hat is
pinned against a numpy restatement in the tests, not against the reference.

Layout of the statistics vector (yg_pooled_stats, length 3 + d + 2 d^2 + d):
  [0] chains  [1] samples per chain n  [2] sum accepts
  sum_c mean_c [d] | sum_c mean_c mean_c' [d,d] | sum_c M2_c [d,d] | sum_c var_c [d]
yg_pooled_stats builds it from the chains' Welford moments (d <= 8); yg_pooled_samples builds the same vector from a
stored sample buffer for any d <= 64 (the tensor path keeps a diagonal Welford M2 only).
"""
import numpy as np
import torch


def shard_range(n_global, rank, world):
    return (n_global * rank) // world, (n_global * (rank + 1)) // world


def all_reduce_stats(vec):
    """Sums the statistics vector over ranks; entry [1] (samples per chain) is identical on
    every rank and is restored after the sum."""
    import torch.distributed as dist
    if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
        n = vec[1].clone()
        dist.all_reduce(vec, op=dist.ReduceOp.SUM)
        vec[1] = n
    return vec


def moments_from_stats(vec, d):
    """Pooled mean / covariance / acceptance / R-hat from the (all-reduced) statistics vector."""
    v = np.asarray(vec.detach().cpu().numpy() if torch.is_tensor(vec) else vec, dtype=np.float64)
    C, n, acc = v[0], v[1], v[2]
    o = 3
    s_mean = v[o:o + d]; o += d
    s_mm = v[o:o + d * d].reshape(d, d); o += d * d
    s_m2 = v[o:o + d * d].reshape(d, d); o += d * d
    s_var = v[o:o + d]
    mu = s_mean / C
    between = s_mm - C * np.outer(mu, mu)                  # sum_c (mean_c - mu)(mean_c - mu)'
    cov = (0.5 * (s_m2 + s_m2.T) + n * between) / (C * n - 1.0) if C * n > 1 else np.full((d, d), np.nan)
    out = dict(n_chains=int(C), samples_per_chain=int(n), mean=mu, covariance=cov,
               acceptance_rate=acc / (C * n) if n > 0 else 0.0)
    if C > 1 and n > 1:
        W = s_var / C                                      # mean within-chain variance
        B_over_n = np.diag(between) / (C - 1.0)            # variance of the chain means
        var_plus = (n - 1.0) / n * W + B_over_n
        out['rhat'] = np.sqrt(var_plus / W)
    else:
        out['rhat'] = np.full(d, np.nan)
    return out


def pooled_diagnostics(ensemble):
    """ensemble: ChainEnsemble of THIS rank.  Returns pooled moments / R-hat over all ranks."""
    vec = all_reduce_stats(ensemble.pooled_stats())
    return moments_from_stats(vec, ensemble.dim)


def proposal_factor_from_covariance(cov, scale=None, eps=1e-8):
    """Lower Cholesky factor of scale * (cov + eps I); scale defaults to the adaptive-Metropolis 2.4^2 / d
    (the scaling of DESIGN.md section 5).  Host-side, d x d."""
    cov = np.asarray(cov, dtype=np.float64)
    d = cov.shape[0]
    s = 2.4 * 2.4 / d if scale is None else float(scale)
    return np.linalg.cholesky(s * (0.5 * (cov + cov.T) + eps * np.eye(d)))


def pooled_proposal_covariance(ensemble, scale=None, eps=1e-8):
    """Optional pooled proposal covariance (north_star): the covariance of ALL chains of ALL ranks, from the
    same all-reduced sufficient statistics as the diagnostics (one all-reduce of 3 + 2d + 2d^2 doubles over
    NCCL / NVLink), becomes the proposal covariance of every chain: L = chol(scale (Sigma_pooled + eps I)).
    Every rank computes the same factor from the same reduced vector, so the ensemble stays reproducible
    and invariant to the GPU count.  Call it between runs, after a burn-in: the Welford statistics it pools
    cover the steps since the last set_state.  Returns the moments dict with the factor under 'prop_L'."""
    out = pooled_diagnostics(ensemble)
    L = proposal_factor_from_covariance(out['covariance'], scale, eps)
    ensemble.set_proposal_factor(L)
    out['prop_L'] = L
    return out


def pooled_diagnostics_from_samples(samples, accepted, transitions):
    """Pooled moments and R-hat over all ranks from THIS rank's stored samples [n_samples, d, n_chains] (a device
    tensor in yg_run's samples layout, e.g. Trajectory.device_tensor; d <= 64).  accepted: accepted transitions summed
    over this rank's chains; transitions: transitions per chain, the same on every rank.  The acceptance entry is
    written as accepted n_samples / transitions before the all-reduce, so 'acceptance_rate' is the pooled accepted
    transitions over the pooled transitions."""
    from .ensemble import pooled_sample_stats
    vec = pooled_sample_stats(samples)
    vec[2] = float(accepted) * samples.shape[0] / transitions if transitions > 0 else 0.0
    return moments_from_stats(all_reduce_stats(vec), samples.shape[1])


def pooled_proposal_covariance_from_samples(ensemble, samples, accepted, transitions, scale=None, eps=1e-8):
    """pooled_proposal_covariance from stored samples (pooled_diagnostics_from_samples): the factor
    L = chol(scale (Sigma_pooled + eps I)) is installed with ensemble.rebuild_proposal_factor, so a tensor-path
    ensemble built with a diagonal factor switches to the dense one.  Returns the moments dict with 'prop_L'."""
    out = pooled_diagnostics_from_samples(samples, accepted, transitions)
    L = proposal_factor_from_covariance(out['covariance'], scale, eps)
    ensemble.rebuild_proposal_factor(L)
    out['prop_L'] = L
    return out


def split_rhat_from_moments(hm, hv, half):
    """Split-R-hat per coordinate from per-chain half moments hm, hv [2, d, n] (torch tensors on any
    device) of THIS rank; all-reduced over ranks when torch.distributed is initialised.  The two
    halves of every chain are treated as 2n chains of length `half`."""
    d, n = hm.shape[1], hm.shape[2]
    stats = torch.stack([torch.full((d,), float(2 * n), dtype=torch.float64, device=hm.device),
                         hm.sum(dim=(0, 2)), (hm * hm).sum(dim=(0, 2)), hv.sum(dim=(0, 2))])
    import torch.distributed as dist
    if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
        dist.all_reduce(stats)
    m, s1, s2, sv = [x.cpu().numpy() for x in stats]
    W = sv / m
    B_over_n = (s2 - s1 * s1 / m) / (m - 1.0)
    return np.sqrt(((half - 1.0) / half * W + B_over_n) / W)


def split_rhat(samples):
    """Split-R-hat per coordinate from stored samples [N, d, n] of THIS rank (+ all ranks when
    torch.distributed is initialised): every chain is cut in two halves (yg_split_moments)."""
    from .ensemble import split_moments
    hm, hv = split_moments(samples)                        # [2, d, n] each
    return split_rhat_from_moments(hm, hv, samples.shape[0] // 2)
