"""Long-double reference of yg_pooled_samples (parallel.py's statistics vector from a stored sample buffer) and the bound
each entry of the kernel's double-precision result must meet.

Layout: samples x[ns, d, nc] as the device stores them (chain index fastest).  mean_c is the mean of chain c's ns
samples and M2_c = sum_t (x_ct - mean_c)(x_ct - mean_c)'.

The kernel's formulation (yagre_mcmc_b200/csrc/diag_kernels.cu, pooled_samples_kernel), restated in double by
`kernel_formulation` below: chain c is shifted by its first sample s_c, y = fl(x - s_c), S1_c = sum_t y,
mean_c = s_c + S1_c / ns, M2_c = sum_t y y' - S1_c (S1_c / ns)', var_c = (sum_t y_i^2 - S1_i (S1_i / ns)) / (ns - 1);
every sum over chains is a plain sum.

Bounds (u = 2^-53, gamma_k = k u / (1 - k u); A1_c = sum_t |y_t|, Q_c = sum_t y_t^2, all in exact arithmetic):
  * Sums.  Every floating-point sum the kernel forms adds each term through at most h additions (a lane's chain
    groups one after the other -- at most nc + 3 k-steps of four products each --, then the CTA's 4 warps, then at
    most nc / 16 + 1 CTA partials in stage 2), so |error| <= gamma_h sum|terms| (Higham, Accuracy and Stability,
    (4.4), which holds for any order).  Vector and pass-2 sums: h_vec = 2 nc + 20.  The M2 sum has (ns + 1) k-steps
    per chain group: h_m2 = (ns + 1)(nc + 3) + nc + 20.
  * mean_c: y carries u |y|, S1 gamma_ns A1 on top, the division and the addition u each:
        e_c = gamma_{ns+3} (|mean_c| + A1_c / ns).
    sum_c mean_c:             sum_c e_c + gamma_{h_vec} sum_c (|mean_c| + e_c)
    sum_c mean_c mean_c':     sum_c (|m_i| e_j + e_i |m_j| + e_i e_j) + gamma_{h_vec+1} sum_c (|m_i| + e_i)(|m_j| + e_j)
  * M2: a product y_i y_j of rounded y carries gamma_3; S1_i (S1_j / ns) carries gamma_{2 ns + 4} A1_i A1_j / ns.  With
    the summation on top:
        sum_c M2_c:           gamma_{h_m2 + 2 ns + 8} (sum_{t,c} |y_i y_j| + 3 sum_c A1_i A1_j / ns)
  * var_c: Q carries gamma_{ns+2} Q, S1_i (S1_i / ns) gamma_{2 ns + 4} A1_i^2 / ns, the subtraction and the division u
    each:  e_var_c = gamma_{2 ns + 8} (Q + A1^2 / ns + |M2_c,ii|) / (ns - 1)
        sum_c var_c:          sum_c e_var_c + gamma_{h_vec+1} sum_c (|var_c| + e_var_c)
  [0] (chains), [1] (ns) and [2] (0) are exact.
The reference itself is computed in long double (64-bit significand), 2^-11 of u: far inside these bounds.

A raw-moment formulation (sum_t x x' - ns mean mean') loses u |x|^2 per term instead of u |y|^2: with a common offset of
1e4 on unit-scale data it exceeds the M2 bound by orders of magnitude, which the CPU test shows."""
import numpy as np

U = 2.0 ** -53


def gamma(k):
    return k * U / (1.0 - k * U)


def _ld(x):
    return np.asarray(x, dtype=np.longdouble)


def reference(x):
    """(vector in long double, tolerance vector in float64) for samples x[ns, d, nc]."""
    X = _ld(x)
    ns, d, nc = X.shape
    Y = X - X[0][None]                                         # [ns, d, nc]
    S1, A1 = Y.sum(axis=0), np.abs(Y).sum(axis=0)               # [d, nc]
    Q = (Y * Y).sum(axis=0)
    mean = X[0] + S1 / ns
    m2 = np.einsum('tic,tjc->ij', Y, Y) - np.einsum('ic,jc->ij', S1, S1) / ns
    m2_abs = np.einsum('tic,tjc->ij', np.abs(Y), np.abs(Y)) + 3.0 * np.einsum('ic,jc->ij', A1, A1) / ns
    m2_diag_c = Q - S1 * S1 / ns                                # [d, nc]
    var_c = m2_diag_c / (ns - 1) if ns > 1 else np.zeros_like(m2_diag_c)

    h_vec, h_m2 = 2 * nc + 20, (ns + 1) * (nc + 3) + nc + 20
    am = np.abs(mean)
    e = gamma(ns + 3) * (am + A1 / ns)
    tol_mean = e.sum(axis=1) + gamma(h_vec) * (am + e).sum(axis=1)
    tol_mm = (np.einsum('ic,jc->ij', am, e) + np.einsum('ic,jc->ij', e, am) + np.einsum('ic,jc->ij', e, e)
              + gamma(h_vec + 1) * np.einsum('ic,jc->ij', am + e, am + e))
    tol_m2 = gamma(h_m2 + 2 * ns + 8) * m2_abs
    if ns > 1:
        e_var = gamma(2 * ns + 8) * (Q + A1 * A1 / ns + np.abs(m2_diag_c)) / (ns - 1)
        tol_var = e_var.sum(axis=1) + gamma(h_vec + 1) * (np.abs(var_c) + e_var).sum(axis=1)
    else:
        tol_var = np.zeros(d, dtype=np.longdouble)
    ref = np.concatenate([_ld([nc, ns, 0]), mean.sum(axis=1), np.einsum('ic,jc->ij', mean, mean).ravel(),
                          m2.ravel(), var_c.sum(axis=1)])
    tol = np.concatenate([np.zeros(3), tol_mean, tol_mm.ravel(), tol_m2.ravel(), tol_var]).astype(np.float64)
    return ref, tol


def check_vector(vec, x, label=""):
    """Asserts that vec (float64, parallel.py's layout) is the statistics vector of x within the bounds above, with the
    M2 block exactly symmetric.  Returns the worst error / bound ratio."""
    v = np.asarray(vec, dtype=np.float64)
    ref, tol = reference(x)
    assert v.shape == ref.shape, (label, v.shape, ref.shape)
    err = np.abs(v.astype(np.longdouble) - ref).astype(np.float64)
    bad = np.nonzero(err > tol)[0]
    assert bad.size == 0, (label, "entries outside the bound", bad[:10], err[bad[:10]], tol[bad[:10]])
    d = np.asarray(x).shape[1]
    o = 3 + d
    for blk in (v[o:o + d * d], v[o + d * d:o + 2 * d * d]):
        m = blk.reshape(d, d)
        assert np.array_equal(m, m.T), (label, "block not symmetric")
    nz = tol > 0
    return float((err[nz] / tol[nz]).max()) if nz.any() else 0.0


def pooled_moments(x):
    """Long-double pooled mean and covariance of all samples of all chains of x[ns, d, nc] (float64)."""
    X = _ld(x)
    flat = X.transpose(0, 2, 1).reshape(-1, X.shape[1])
    mu = flat.sum(axis=0) / flat.shape[0]
    dev = flat - mu
    cov = dev.T @ dev / (flat.shape[0] - 1) if flat.shape[0] > 1 else np.full((X.shape[1],) * 2, np.nan)
    return mu.astype(np.float64), cov.astype(np.float64)


def kernel_formulation(x):
    """The kernel's arithmetic in double precision (one summation order of many), for the CPU tests of the bound."""
    x = np.asarray(x, dtype=np.float64)
    ns, d, nc = x.shape
    y = x - x[0][None]
    S1 = y.sum(axis=0)
    nS = S1 / ns
    mean = x[0] + nS
    m2 = np.einsum('tic,tjc->ij', y, y) - S1 @ nS.T
    var = ((y * y).sum(axis=0) - S1 * nS) / (ns - 1) if ns > 1 else np.zeros((d, nc))
    return np.concatenate([[nc, ns, 0.0], mean.sum(axis=1), _lower_mirrored(mean @ mean.T).ravel(),
                           _lower_mirrored(m2).ravel(), var.sum(axis=1)])


def _lower_mirrored(a):
    return np.tril(a) + np.tril(a, -1).T


def raw_formulation(x):
    """The same vector from raw moments, sum_t x x' - ns mean mean' (what the kernel must NOT do)."""
    x = np.asarray(x, dtype=np.float64)
    ns, d, nc = x.shape
    mean = x.mean(axis=0)
    m2 = np.einsum('tic,tjc->ij', x, x) - ns * mean @ mean.T
    var = ((x * x).sum(axis=0) - ns * mean * mean) / (ns - 1)
    return np.concatenate([[nc, ns, 0.0], mean.sum(axis=1), _lower_mirrored(mean @ mean.T).ravel(),
                           _lower_mirrored(m2).ravel(), var.sum(axis=1)])
