"""High-precision reference of the chain diagnostics the step kernels keep (FullDiagnostics, chain/diagnostics.py:91-94):
the Welford mean and co-moment of the pre-transition states since the last reset, and the bounds a kernel's
double-precision accumulation must stay within.

Layouts: device arrays are [d, n_chains] / [d, d, n_chains] (or [d, n_chains] for the tensor path's diagonal M2);
the reference works chain by chain, pre[n_chains, n, d].
"""
import numpy as np

U = 2.0 ** -53          # unit roundoff of binary64


def pre_states(theta0, samples_per_run, restarts=None):
    """Pre-transition states of every chain since the last reset: [n_chains, n, d] float64.

    theta0: [n_chains, d], the state set by the last set_state without keep_diagnostics.
    samples_per_run: the samples of each run since then, in the device layout [ns, d, n_chains], unthinned.
    restarts: optional list as long as samples_per_run; entry k is None (run k continues where run k-1 ended,
    which is also what a load_state of the state() in between does) or the [n_chains, d] state given to
    set_state(..., keep_diagnostics=True) before run k.

    A run of ns transitions from x0 sees x0, samples[0], ..., samples[ns-2]: the last sample is the next run's first
    pre-state (or is replaced by the restart state)."""
    x = np.asarray(theta0, dtype=np.float64)
    parts = []
    for k, s in enumerate(samples_per_run):
        if restarts is not None and restarts[k] is not None:
            x = np.asarray(restarts[k], dtype=np.float64)
        s = np.asarray(s, dtype=np.float64)
        if s.shape[0] == 0:
            continue
        chain = s.transpose(2, 0, 1)                        # [n_chains, ns, d]
        parts += [x[:, None, :], chain[:, :-1]]
        x = chain[:, -1]
    return np.concatenate(parts, axis=1)


def welford_reference(pre):
    """Mean [n_chains, d] and full co-moment R[n_chains, d, d] = sum_t (x_t - mu)(x_t - mu)' by two passes in long
    double (64-bit significand: its own error is 2^-11 of the bounds below)."""
    x = np.asarray(pre, dtype=np.longdouble)
    mu = x.sum(axis=1) / x.shape[1]
    dev = x - mu[:, None, :]
    return mu, np.einsum('cti,ctj->cij', dev, dev)


def welford_tolerance(pre, ref, traj_rtol=0.0):
    """Bounds (mean [n_chains, d], M2 [n_chains, d, d]) on |kernel - reference| for n pre-states, u = 2^-53:

        |d mu_i|   <= 4 n u max_t|x_i|
        |d M2_ij|  <= 1e-11 sqrt(R_ii R_jj) + 8 n u (max|x_i| max|x_j - mu_j| + max|x_j| max|x_i - mu_i|)

    Derivation.  Step t of Welford's recurrence (m' = m + (x - m)/t, M2' = M2 + (x - m)(x - m')) commits a
    rounding error of at most ~3u max|x| to the mean: the subtraction (u |x - m| <= 2u max|x|), the division and the
    addition (u |m'|).  The recurrence passes an earlier error e of the mean on as e (1 - 1/t), so the errors add up
    to at most n times the local one.  The co-moment term (x - m)(x - m') carries the mean's error into both factors;
    bounding |x - m| by max|x - mu| + |mu - m| and the accumulated error of the sum by n u |terms| gives the second
    part.  The first part is the relative rounding of the n additions into M2 itself (n u R_ii at most, far below
    1e-11 R for the n here), kept as a floor so that an exactly-zero M2 of a coordinate that moved still fails.
    The run-length form of the tensor path (m steps at once: mean += (x - mean) m / n', M2 += (x - mean)^2 n m / n')
    is the same recurrence with fewer roundings, so the same bound holds.

    traj_rtol: the pre-states are another computation's trajectory, equal to the kernel's to this relative error
    (the oracle replay of a thinned run): adds traj_rtol max|x| to the mean and traj_rtol n max|x| max|x - mu| per
    factor to M2."""
    x = np.asarray(pre, dtype=np.float64)
    mu, R = ref
    n = x.shape[1]
    amax = np.abs(x).max(axis=1)                                            # [n_chains, d]
    dmax = np.abs(x - np.asarray(mu, dtype=np.float64)[:, None, :]).max(axis=1)
    cross = amax[:, :, None] * dmax[:, None, :] + amax[:, None, :] * dmax[:, :, None]
    Rd = np.asarray(np.einsum('cii->ci', R), dtype=np.float64)
    tol_mean = (4.0 * n * U + traj_rtol) * amax
    tol_m2 = 1e-11 * np.sqrt(Rd[:, :, None] * Rd[:, None, :]) + (8.0 * n * U + traj_rtol * n) * cross
    return tol_mean, tol_m2


def check_welford(w_mean, w_m2, welford_n, pre, label="", traj_rtol=0.0):
    """Asserts that the kernel's w_mean [d, nc] and w_m2 ([d, d, nc], or [d, nc] diagonal) are the Welford moments of
    pre [nc, n, d] within welford_tolerance, and exact for a chain that never left its state: w_mean equal to that
    state, w_m2 zero (the first update of either form is exact, and every later one adds exact zeros)."""
    pre = np.asarray(pre, dtype=np.float64)
    nc, n, d = pre.shape
    assert welford_n == n, (label, welford_n, n)
    wm = np.asarray(w_mean, dtype=np.float64).T                            # [nc, d]
    w2 = np.asarray(w_m2, dtype=np.float64)
    diag_only = w2.ndim == 2
    w2 = w2.T if diag_only else w2.transpose(2, 0, 1)                      # [nc, d] or [nc, d, d]
    mu, R = welford_reference(pre)
    tm, t2 = welford_tolerance(pre, (mu, R), traj_rtol)
    em = np.abs(wm - mu.astype(np.float64))
    assert np.all(em <= tm), (label, "w_mean", float((em / np.maximum(tm, 1e-300)).max()))
    if diag_only:
        R, t2 = np.einsum('cii->ci', R), np.einsum('cii->ci', t2)
    e2 = np.abs(w2 - R.astype(np.float64))
    assert np.all(e2 <= t2), (label, "w_m2", float((e2 / np.maximum(t2, 1e-300)).max()),
                              np.unravel_index(int(np.argmax(e2 - t2)), e2.shape))
    still = (pre == pre[:, :1]).all(axis=(1, 2))
    if traj_rtol == 0.0 and still.any():
        assert np.array_equal(wm[still], pre[still, 0]), (label, "w_mean of a chain that never moved")
        assert np.all(w2[still] == 0.0), (label, "w_m2 of a chain that never moved")
    return int(still.sum())


POOLED_RTOL = 1e-9      # moments_from_stats against the long-double moments of all pre-states


def pooled_reference(st, welford_n):
    """The statistics vector of yg_pooled_stats (parallel.py's layout) as long-double sums of the state arrays."""
    wm = np.asarray(st["w_mean"], dtype=np.longdouble)                    # [d, nc]
    w2 = np.asarray(st["w_m2"], dtype=np.longdouble)                      # [d, d, nc]
    d, nc = wm.shape
    n = np.longdouble(welford_n)
    mm = wm[:, None, :] * wm[None, :, :]
    var = np.einsum('iic->ic', w2) / (n - 1) if welford_n > 1 else np.zeros_like(wm)
    terms = [np.ones((1, nc), dtype=np.longdouble), None,
             np.asarray(st["n_accept"], dtype=np.longdouble)[None, :],
             wm, mm.reshape(d * d, nc), w2.reshape(d * d, nc), var]
    ref, mag = [], []
    for t in terms:
        if t is None:
            ref.append([n]); mag.append([0.0])
        else:
            ref.append(t.sum(axis=1)); mag.append(np.abs(t).sum(axis=1))
    return np.concatenate(ref), np.concatenate(mag).astype(np.float64)


def check_pooled(vec, st, welford_n, pre, label=""):
    """yg_pooled_stats against long-double sums of the state (tolerance per entry: n_chains u sum|terms|, the bound of
    any summation order), and moments_from_stats against the long-double mean / covariance of all pre-states of all
    chains (POOLED_RTOL of max|x_i| for the mean, of sqrt(cov_ii cov_jj) for the covariance)."""
    from yagre_mcmc_b200.parallel import moments_from_stats
    v = np.asarray(vec, dtype=np.float64)
    nc = np.asarray(st["n_accept"]).shape[0]
    ref, mag = pooled_reference(st, welford_n)
    err = np.abs(v.astype(np.longdouble) - ref).astype(np.float64)
    tol = nc * U * mag
    assert np.all(err <= tol), (label, "pooled vector", np.nonzero(err > tol)[0])
    assert v[0] == nc and v[1] == welford_n, label
    d = np.asarray(st["w_mean"]).shape[0]
    pm = moments_from_stats(v, d)
    flat = np.asarray(pre, dtype=np.longdouble).reshape(-1, d)
    mu = flat.sum(axis=0) / flat.shape[0]
    dev = flat - mu
    cov = (dev.T @ dev / (flat.shape[0] - 1)).astype(np.float64)
    mu = mu.astype(np.float64)
    assert np.all(np.abs(pm["mean"] - mu) <= POOLED_RTOL * np.abs(flat.astype(np.float64)).max(axis=0)), (label, pm["mean"], mu)
    sd = np.sqrt(np.diag(cov))
    assert np.all(np.abs(pm["covariance"] - cov) <= POOLED_RTOL * np.outer(sd, sd)), (label, pm["covariance"], cov)


def check_replay_diagnostics(st, counters, ref, pre, label="", traj_rtol=0.0):
    """A run replayed through the oracle (cport.run_injected of its recorded noise, from a fresh state): the kernel's
    Welford moments against the reference of pre [nc, n, d] (check_welford), its w_mean and diag(w_m2) / (n - 1)
    against the oracle's own float64 welford_mean / welford_var (both within the bound of the same truth: twice the
    bound apart at most), and coarse_accepted against the oracle's per-chain count of accepted coarse sub-steps."""
    s = {k: np.asarray(v.cpu().numpy() if hasattr(v, "cpu") else v) for k, v in st.items() if k in ("w_mean", "w_m2")}
    n = counters["welford_n"]
    check_welford(s["w_mean"], s["w_m2"], n, pre, label, traj_rtol)
    mu, R = welford_reference(pre)
    tm, t2 = welford_tolerance(pre, (mu, R), traj_rtol)
    assert np.all(np.abs(s["w_mean"].T - ref["welford_mean"]) <= 2 * tm), (label, "w_mean vs the oracle")
    w2 = s["w_m2"]
    diag = (w2 if w2.ndim == 2 else np.einsum('iic->ic', w2)).T
    if n > 1:
        assert np.all(np.abs(diag / (n - 1) - ref["welford_var"]) <= 2 * np.einsum('cii->ci', t2) / (n - 1)), \
            (label, "w_m2 vs the oracle")
    assert counters["coarse_accepted"] == int(ref["coarse_accepted"].sum()), (label, counters["coarse_accepted"])
