"""Long-double reference of the log-posterior every level of a lowered problem returns (yo_logpost,
oracle/yagre_oracle.c), absolute bounds a double-precision evaluation must stay within, and accept uniforms placed at
known distances from each decision's threshold (forced_schedule).

Layouts: meta / arrays are the lowered problem (ensemble.LoweredProblem); theta is [n, d].  Everything here is numpy
on the host; no torch.

Rule of the forced schedules: a uniform is never placed where a correct double-precision kernel could decide either
way.  Every decision gets eta >= ETA_FACTOR x a bound on the error of its delta, and a point whose forward model comes
near the double range is undecidable and raises.
"""
import numpy as np

LD = np.longdouble
assert np.finfo(LD).nmant >= 63, "the reference needs an 80-bit (or wider) long double"

U = 2.0 ** -53                       # unit roundoff of binary64
DBL_MAX = float(np.finfo(np.float64).max)
RANGE_MARGIN = 2.0 ** 16             # a value within this factor of DBL_MAX (either side) is undecidable
ETA_FACTOR = 100.0                   # eta of a forced decision >= ETA_FACTOR x the bound on the error of its delta

# c_rk4: |(x, y)_double - (x, y)_long double| <= c_rk4 * N * u * max over the trajectory of max(|x|, |y|) for one
# N-step RK4 integration of the LV model, double precision in either order the project uses (the oracle's textbook
# order, lv_rk4; the kernel's stage-point form, lv_model.cuh lv_rk4_step, ported with fma emulated in long double).
# Measured by measure_c_rk4(n_draws=10000, Ns=(16, 64, 512, 4096), seed=2026) on theta in LV_TRUTH + [-1.5, 1.5]^2,
# design points in [0.5, 1.5]^2, T = 10, alpha = 0.8, gamma = 0.4 (40,000 integrations per order):
#   worst ratio          N = 16   N = 64   N = 512   N = 4096
#     textbook           0.598    0.281    0.115     0.027
#     stage-point        0.922    0.716    0.322     0.544
# c_rk4 is 4x the worst: 3.7 (rounded up from 3.69).  The 4x also covers CUDA's exp (<= 1 ulp) against numpy's.
C_RK4 = 3.7
C_RK4_REGION = 1.5                   # half-width of the measured theta box around LV_TRUTH


def gamma(n):
    """Higham's gamma_n = n u / (1 - n u): the relative bound of n roundings in any order."""
    n = np.asarray(n, dtype=np.float64)
    return n * U / (1.0 - n * U)


class Undecidable(ValueError):
    """A point whose double-precision evaluation may or may not overflow."""


def _lvl(arrays, level):
    pre = f"L{level}_"
    return {k[len(pre):]: np.asarray(v) for k, v in arrays.items() if k.startswith(pre)}


def _tempering(L):
    return float(np.asarray(L["tempering"]).reshape(-1)[0]) if "tempering" in L else 1.0


def _quad_ld(P, x):
    """x' P x over the last axis, long double.  P [m, m], x [..., m]."""
    P = np.asarray(P, dtype=LD)
    return np.einsum('...k,kl,...l->...', x, P, x)


def _quad_bound(P, x, dx, m):
    """Bound on |fl(x~' P x~) - x' P x| for |x~ - x| <= dx, evaluated in m terms per dot product:
    2 (|P||x|)'dx + dx'|P|dx (the perturbation of x) + gamma_{m+1} |x|'|P||x| (the roundings of the quad form,
    Higham 3.5: a dot product of m terms is within gamma_m of its sum of magnitudes; the outer sum adds one)."""
    A = np.abs(np.asarray(P, dtype=np.float64))
    ax = np.abs(np.asarray(x, dtype=np.float64))
    dx = np.asarray(dx, dtype=np.float64)
    Px = ax @ A.T
    return 2.0 * (Px * dx).sum(-1) + ((dx @ A.T) * dx).sum(-1) + gamma(m + 1) * (Px * ax).sum(-1)


def _check_range(mag):
    """+1: beyond DBL_MAX by more than the margin (the double evaluation has overflowed: -inf); -1: undecidable;
    0: far inside the double range."""
    mag = np.asarray(mag, dtype=LD)
    over = ~(mag <= LD(DBL_MAX) * LD(RANGE_MARGIN))           # includes inf / nan
    band = ~over & (mag > LD(DBL_MAX) / LD(RANGE_MARGIN))
    return np.where(over, 1, np.where(band, -1, 0))


# ------------------------------------------------------------------------------------------------------------------
# the LV forward model (discrete RK4, same h = T / N and exp(theta) rates as the oracle and the kernel)
# ------------------------------------------------------------------------------------------------------------------
def lv_rk4_ld(beta, delta, x, y, alpha, gamma_, T, N):
    """Textbook RK4 in long double over broadcast arrays.  Returns (x, y, peak): peak is the largest magnitude of any
    stage point and of any x*y product on the way (inf / nan once the long double itself overflowed)."""
    x, y = LD(1) * x, LD(1) * y
    beta, delta = LD(1) * beta, LD(1) * delta
    a, g = LD(alpha), LD(gamma_)
    h = LD(T) / LD(N)
    h2, h6 = h / 2, h / 6
    peak = np.maximum(np.abs(x), np.abs(y))
    with np.errstate(over='ignore', invalid='ignore'):
        for _ in range(int(N)):
            xy = x * y
            k1x, k1y = a * x - beta * xy, delta * xy - g * y
            xa, ya = x + h2 * k1x, y + h2 * k1y
            xya = xa * ya
            k2x, k2y = a * xa - beta * xya, delta * xya - g * ya
            xb, yb = x + h2 * k2x, y + h2 * k2y
            xyb = xb * yb
            k3x, k3y = a * xb - beta * xyb, delta * xyb - g * yb
            xc, yc = x + h * k3x, y + h * k3y
            xyc = xc * yc
            k4x, k4y = a * xc - beta * xyc, delta * xyc - g * yc
            x = x + h6 * (((k1x + 2 * k2x) + 2 * k3x) + k4x)
            y = y + h6 * (((k1y + 2 * k2y) + 2 * k3y) + k4y)
            for v in (xy, xa, ya, xya, xb, yb, xyb, xc, yc, xyc, x, y):
                peak = np.fmax(peak, np.abs(v))
            bad = ~np.isfinite(x) | ~np.isfinite(y)
            peak = np.where(bad, LD(np.inf), peak)
    return x, y, peak


def lv_rk4_textbook_f64(beta, delta, x, y, alpha, gamma_, T, N):
    """The oracle's lv_rk4 in double (numpy does not fuse)."""
    h = T / N
    h2, h6 = 0.5 * h, h / 6.0
    with np.errstate(over='ignore', invalid='ignore'):
        for _ in range(int(N)):
            k1x, k1y = alpha * x - beta * x * y, delta * x * y - gamma_ * y
            xa, ya = x + h2 * k1x, y + h2 * k1y
            k2x, k2y = alpha * xa - beta * xa * ya, delta * xa * ya - gamma_ * ya
            xb, yb = x + h2 * k2x, y + h2 * k2y
            k3x, k3y = alpha * xb - beta * xb * yb, delta * xb * yb - gamma_ * yb
            xc, yc = x + h * k3x, y + h * k3y
            k4x, k4y = alpha * xc - beta * xc * yc, delta * xc * yc - gamma_ * yc
            x = x + h6 * (((k1x + 2.0 * k2x) + 2.0 * k3x) + k4x)
            y = y + h6 * (((k1y + 2.0 * k2y) + 2.0 * k3y) + k4y)
    return x, y


def _fma(a, b, c):
    """fma emulated: the long double product and sum, rounded once more to double (a 64-bit significand holds the
    product to 2^-11 of an ulp of double; the double rounding is within an ulp of the true fma)."""
    return np.asarray(LD(1) * a * b + c, dtype=np.float64)


def lv_rk4_stage_point_f64(beta, delta, x, y, alpha, gamma_, T, N, consts_f32=False):
    """Port of lv_model.cuh: lv_step_consts, lv_rates and lv_rk4_step (the kernel's stage-point form).
    consts_f32 rounds the chain-independent constants to float32 (a wrong evaluation the bounds must catch)."""
    h = T / N
    ha, hg = h * alpha, h * gamma_
    ha1, ha2, ha6 = ha, 0.5 * ha, ha / 6.0
    ha6p = ha6 + 1.0 / 3.0
    mhg1, mhg2, mhg6 = -hg, -0.5 * hg, -(hg / 6.0)
    mhg6p = 1.0 / 3.0 + mhg6
    if consts_f32:
        ha1, ha2, ha6, ha6p, mhg1, mhg2, mhg6, mhg6p = (float(np.float32(v)) for v in
                                                        (ha1, ha2, ha6, ha6p, mhg1, mhg2, mhg6, mhg6p))
    hb, hd = h * beta, h * delta
    mb1, mb2, mb6 = -hb, -0.5 * hb, -(hb * (1.0 / 6.0))
    hd1, hd2, hd6 = hd, 0.5 * hd, hd * (1.0 / 6.0)
    with np.errstate(over='ignore', invalid='ignore'):
        for _ in range(int(N)):
            tx = x * _fma(mb6, y, ha6)
            ty = y * _fma(hd6, x, mhg6)
            x2, y2 = _fma(3.0, tx, x), _fma(3.0, ty, y)
            x3 = _fma(x2, _fma(mb2, y2, ha2), x)
            y3 = _fma(y2, _fma(hd2, x2, mhg2), y)
            x4 = _fma(x3, _fma(mb1, y3, ha1), x)
            y4 = _fma(y3, _fma(hd1, x3, mhg1), y)
            wx, wy = _fma(mb6, y4, ha6p), _fma(hd6, x4, mhg6p)
            sx, sy = _fma(2.0 / 3.0, x3, tx), _fma(2.0 / 3.0, y3, ty)
            x, y = _fma(x4, wx, sx), _fma(y4, wy, sy)
    return x, y


def measure_c_rk4(n_draws, Ns, seed, alpha=0.8, gamma_=0.4, T=10.0, half_width=C_RK4_REGION):
    """Worst |double - long double| / (N u peak) per order and N over n_draws (theta, design point) draws:
    {(order, N): ratio}.  Points whose long-double trajectory leaves the double range (by any margin) are skipped."""
    rng = np.random.default_rng(seed)
    truth = np.log(np.array([0.4, 0.6]))
    th = truth + rng.uniform(-half_width, half_width, (n_draws, 2))
    x0, y0 = rng.uniform(0.5, 1.5, n_draws), rng.uniform(0.5, 1.5, n_draws)
    beta, delta = np.exp(th[:, 0]), np.exp(th[:, 1])
    out = {}
    for N in Ns:
        xr, yr, peak = lv_rk4_ld(beta, delta, x0, y0, alpha, gamma_, T, N)
        ok = _check_range(peak) == 0
        scale = N * U * np.asarray(peak, dtype=np.float64)
        for name, f in (("textbook", lv_rk4_textbook_f64), ("stage_point", lv_rk4_stage_point_f64)):
            x, y = f(beta, delta, x0.copy(), y0.copy(), alpha, gamma_, T, N)
            e = np.maximum(np.abs(np.asarray(x - xr, dtype=np.float64)), np.abs(np.asarray(y - yr, dtype=np.float64)))
            out[(name, N)] = float(np.max(e[ok] / scale[ok]))
    return out


# ------------------------------------------------------------------------------------------------------------------
# log-posterior and its bound
# ------------------------------------------------------------------------------------------------------------------
def _lv_misfits(L, theta):
    """Per point and design point: residuals r [n, nD, 2] (long double), trajectory peaks [n, nD] and range flags."""
    design = np.asarray(L["design"], dtype=np.float64)
    alpha, gamma_, T, N = (float(v) for v in np.asarray(L["lv"]).reshape(-1)[:4])
    th = np.asarray(theta, dtype=LD)
    beta, delta = np.exp(th[:, 0:1]), np.exp(th[:, 1:2])                    # [n, 1]
    x, y, peak = lv_rk4_ld(beta, delta, design[None, :, 0], design[None, :, 1], alpha, gamma_, T, int(N))
    data = np.asarray(L["data"], dtype=LD)
    r = np.stack([x - data[None, :, 0], y - data[None, :, 1]], axis=-1)
    return r, peak, int(N)


def logpost_ld(meta, arrays, level, theta):
    """The log-posterior of `level` at theta [n, d] in long double (yo_logpost's formula): -inf where the double
    evaluation certainly overflows; raises Undecidable where it may or may not."""
    lp, _ = _logpost_and_bound(meta, arrays, level, theta, path="generic")
    return lp


def logpost_bound(meta, arrays, level, theta, path=None):
    """Absolute bound per point on |lp_double - lp_ld| for a double-precision evaluation of `level` at theta [n, d]:
    (lp_ld [n] long double, bound [n] float64; bound 0 where lp_ld is -inf: there the kernel must return -inf too).

    path: "generic" (the oracle and the one-chain-per-thread kernels: yo_logpost's formula), "lv" (the LV kernel;
    the same formula with the misfits of RK4 integrations in either order) or "tensor" (linear_dmma_kernel.cu);
    default from the model and the shape.

    Derivation (u = 2^-53, gamma_n = n u / (1 - n u); every sum or dot product of n terms in any order is within
    gamma_n of the sum of the magnitudes of its terms, Higham, Accuracy and Stability, 3.1-3.5):

    * Quad form x' P x (Gaussian target, prior, measurement misfit) at an input off by at most dx per entry:
      2 (|P||x|)' dx + dx'|P| dx + gamma_{m+1} |x|'|P||x|, m = the dimension (_quad_bound).
      The input x = theta - mean is one subtraction: dx = u |x|.
    * Linear misfit, generic path: F = G theta + b is a dot product of d + 1 terms, r = F - data_row one more
      rounding: dr_k <= gamma_{d+2} (sum_j |G_kj theta_j| + |b_k| + |data_k|).
    * LV misfit: the end state of each design point's RK4 integration is within C_RK4 N u peak of the long-double
      one (peak = largest stage magnitude on the trajectory; C_RK4 measured, see above), r = end - data one more
      rounding: dr <= C_RK4 N u peak + u |r|.
    * logL = -1/2 sum_n q_n: gamma_{n_data} sum|q_n| plus the sum of the misfits' own bounds, halved; tempering t
      multiplies it and rounds once: |t| (...) + u |t logL|.
    * The tensor path (linear_dmma_kernel.cu, abi.cu's host side) evaluates
          sum_rows ||F - d_row||^2_P = sum_r w_r (F_r - mean_r)^2 + q_const,  w_r = n_data P_rr,
          q_const = sum_r P_rr sum_i (d_ir - mean_r)^2,
      with sqrt(w_r) folded into G and b - mean on the host.  Per row e_r = sqrt(w_r) (G_r theta + b_r - mean_r):
      the fold (one sqrt, one product per entry of G, one subtraction and product for b - mean) and the DMMA chain of
      d fused products make |de_r| <= gamma_{d+n_data+6} sqrt(w_r) (sum_k |G_rk theta_k| + |b_r| + mean|d_r|),
      with mean|d_r| = sum_i |d_ir| / n (the computed mean is within gamma_{n_data} of it in that scale).
      sum_r e_r^2 then costs 2|e_r| de_r + de_r^2 per row and gamma_{rows+1} sum e_r^2.  The identity drops
      -2 n P_rr (F_r - mean_r)(mean_r - mean~_r), the centring error: <= 2 P_rr |F_r - mean_r| gamma_{n_data} sum_i |d_ir|.
      q_const is a sum of non-negative terms, each a product of two subtractions: gamma_{n_data+data_dim+4} q_const.
      A dense prior P = R'R, R = chol(P)' in double, is folded in as d more rows R theta - R m: a Cholesky factor
      in double satisfies R~'R~ = P + dP, |dP| <= gamma_{d+1} |R~|'|R~| (Higham 10.3), so x'(R~'R~)x is within
      gamma_{d+1} || |R~||x| ||^2 of x'Px; each such row is a dot product of 2 d terms:
      de <= gamma_{2d+1} (|R~||theta| + |R~||m|).  The symmetrisation (P_ij + P_ji) / 2 adds u |x|'|P||x|.
      Then -1/2 (q + q_const) rounds twice more: u (q + q_const).
    * The total adds the prior's bound and one rounding of every sum of terms (u per term).
    """
    if path is None:
        path = _default_path(meta, arrays)
    return _logpost_and_bound(meta, arrays, level, theta, path)


def _default_path(meta, arrays):
    if meta["model"] == "lv":
        return "lv"
    if meta["model"] == "linear":
        d = int(meta["dim"])
        dd = max(np.asarray(arrays[f"L{l}_data"]).shape[1] for l in range(int(meta["levels"])))
        if d > 8 or dd > 8:
            return "tensor"
    return "generic"


def _prior_bound(L, theta):
    x = np.asarray(theta, dtype=LD) - np.asarray(L["prior_mean"], dtype=LD)
    P = np.asarray(L["prior_prec"], dtype=np.float64)
    d = P.shape[0]
    lp = -_quad_ld(P, x) / 2
    b = 0.5 * _quad_bound(P, x, U * np.abs(np.asarray(x, dtype=np.float64)), d)
    return lp, b


def _logpost_and_bound(meta, arrays, level, theta, path):
    theta = np.asarray(theta, dtype=np.float64)
    assert theta.ndim == 2 and theta.shape[1] == int(meta["dim"]), theta.shape
    n, d = theta.shape
    L = _lvl(arrays, level)
    model = meta["model"]
    if model == "gauss":
        x = np.asarray(theta, dtype=LD) - np.asarray(L["g_mean"], dtype=LD)
        P = np.asarray(L["g_prec"], dtype=np.float64)
        c = LD(float(np.asarray(L["g_logconst"]).reshape(-1)[0]))
        q = _quad_ld(P, x)
        if np.any(_check_range(q) != 0):
            _raise_or_inf(q)
        lp = -q / 2 + c
        b = 0.5 * _quad_bound(P, x, U * np.abs(np.asarray(x, dtype=np.float64)), d)
        b = b + U * (np.abs(np.asarray(-q / 2, dtype=np.float64)) + abs(float(c)))
        return lp, b
    t = _tempering(L)
    Pn = np.asarray(L["noise_prec"], dtype=np.float64)
    data = np.asarray(L["data"], dtype=np.float64)
    nD, dd = data.shape
    if model == "lv":
        r, peak, N = _lv_misfits(L, theta)
        flag = _check_range(peak)
        dr = C_RK4 * N * U * np.asarray(np.where(flag == 0, peak, 0), dtype=np.float64)[..., None] \
            + U * np.abs(np.asarray(np.where(flag[..., None] == 0, r, 0), dtype=np.float64))
    elif path == "tensor":
        return _tensor_logpost_and_bound(meta, L, theta)
    else:
        G, bvec = np.asarray(L["G"], dtype=np.float64), np.asarray(L["b"], dtype=np.float64)
        F = np.asarray(theta, dtype=LD) @ np.asarray(G, dtype=LD).T + np.asarray(bvec, dtype=LD)     # [n, dd]
        r = F[:, None, :] - np.asarray(data, dtype=LD)[None]                                          # [n, nD, dd]
        mag = np.abs(theta) @ np.abs(G).T + np.abs(bvec)
        dr = gamma(d + 2) * (mag[:, None, :] + np.abs(data)[None])
        flag = _check_range(np.abs(r).max(axis=-1) ** 2 * np.abs(Pn).max())
    with np.errstate(over='ignore', invalid='ignore'):
        q = _quad_ld(Pn, np.where(flag[..., None] == 0, r, 0))                                         # [n, nD]
        qmag = _check_range(np.where(flag == 0, np.abs(np.asarray(r, dtype=LD)).max(axis=-1) ** 2
                                     * LD(np.abs(Pn).sum()) * nD, 0))
    flag = np.where(flag == 0, qmag, flag)
    point_flag = flag.max(axis=1)
    if np.any(flag == -1):
        raise Undecidable(f"level {level}: points {np.nonzero((flag == -1).any(axis=1))[0][:8]} come within "
                          f"2^16 of the double range")
    dr = np.where(flag[..., None] == 0, dr, 0.0)
    qb = _quad_bound(Pn, np.where(flag[..., None] == 0, np.asarray(r, dtype=np.float64), 0.0), dr, dd)    # [n, nD]
    S = q.sum(axis=1)
    logL = -S / 2
    bL = 0.5 * (qb.sum(axis=1) + gamma(nD) * np.asarray(S, dtype=np.float64))
    lpr, bpr = _prior_bound(L, theta)
    lp = LD(t) * logL + lpr
    b = abs(t) * bL + U * np.abs(np.asarray(LD(t) * logL, dtype=np.float64)) + bpr \
        + U * (np.abs(np.asarray(LD(t) * logL, dtype=np.float64)) + np.abs(np.asarray(lpr, dtype=np.float64)))
    inf = point_flag == 1
    if inf.any():
        if not t > 0:
            raise Undecidable("an overflowed likelihood at a non-positive tempering")
        lp = np.where(inf, LD(-np.inf), lp)
        b = np.where(inf, 0.0, b)
    return lp, b


def _raise_or_inf(q):
    raise Undecidable("a Gaussian quad form outside the double range")


def _tensor_q_const(arrays, level=0):
    """q_const of the tensor path in long double: sum_r P_rr sum_i (d_ir - mean_r)^2."""
    L = _lvl(arrays, level)
    dl = np.asarray(L["data"], dtype=LD)
    return float((((dl - dl.mean(axis=0)) ** 2) * np.diag(np.asarray(L["noise_prec"], dtype=LD))).sum())


def _tensor_logpost_and_bound(meta, L, theta):
    n, d = theta.shape
    G, bvec = np.asarray(L["G"], dtype=np.float64), np.asarray(L["b"], dtype=np.float64)
    data = np.asarray(L["data"], dtype=np.float64)
    nD, dd = data.shape
    Pn = np.diag(np.asarray(L["noise_prec"], dtype=np.float64)).copy()                  # diagonal noise only
    assert np.array_equal(np.diag(Pn), np.asarray(L["noise_prec"])), "the tensor path takes diagonal noise"
    # the reference: yo_logpost's formula in long double
    thl = np.asarray(theta, dtype=LD)
    F = thl @ np.asarray(G, dtype=LD).T + np.asarray(bvec, dtype=LD)                     # [n, dd]
    dl = np.asarray(data, dtype=LD)
    S = (((F[:, None, :] - dl[None]) ** 2) * np.asarray(Pn, dtype=LD)).sum(axis=(1, 2))
    lpr, _ = _prior_bound(L, theta)
    lp = -S / 2 + lpr
    if np.any(_check_range(S) != 0):
        raise Undecidable("tensor path: a misfit outside the double range")
    # the bound of the centred, folded evaluation
    mean = dl.mean(axis=0)
    sw = np.sqrt(nD * Pn)
    e = np.asarray((F - mean) * np.asarray(sw, dtype=LD), dtype=np.float64)             # [n, dd]
    mabs = np.abs(data).sum(axis=0) / nD
    de = gamma(d + nD + 6) * sw * (np.abs(theta) @ np.abs(G).T + np.abs(bvec) + mabs)
    q_const = float((((dl - mean) ** 2) * np.asarray(Pn, dtype=LD)).sum())
    rows = dd
    b_rows = (2.0 * np.abs(e) * de + de * de).sum(axis=1)
    b_sq = np.asarray((e * e).sum(axis=1), dtype=np.float64)
    b_centre = (2.0 * Pn * np.abs(np.asarray(F - mean, dtype=np.float64)) * gamma(nD) * np.abs(data).sum(axis=0)).sum(axis=1)
    b_qc = gamma(nD + dd + 4) * q_const
    P0 = np.asarray(L["prior_prec"], dtype=np.float64)
    m0 = np.asarray(L["prior_mean"], dtype=np.float64)
    x = np.asarray(theta - m0, dtype=np.float64)
    dense = np.count_nonzero(P0 - np.diag(np.diag(P0))) > 0
    if dense:
        R = np.linalg.cholesky(0.5 * (P0 + P0.T)).T                                     # R'R = P
        Rx = np.abs(R) @ np.abs(np.asarray(theta, dtype=np.float64)).T + (np.abs(R) @ np.abs(m0))[:, None]
        dR = gamma(2 * d + 1) * Rx.T                                                     # [n, d]
        ex = np.abs(x) @ np.abs(R).T                                                     # |R||x|
        b_prior = (2.0 * ex * dR + dR * dR).sum(axis=1) + gamma(d + 1) * (ex * ex).sum(axis=1) \
            + U * ((np.abs(x) @ np.abs(P0).T) * np.abs(x)).sum(axis=1)
        b_sq = b_sq + (ex * ex).sum(axis=1)
        rows += d
        prior_sum = np.zeros(n)
    else:
        b_prior = _quad_bound(P0, x, U * np.abs(x), 4)                                   # quad over 4 lanes + 2 shuffles
        b_prior = b_prior + gamma(d + 2) * ((np.abs(x) @ np.abs(P0).T) * np.abs(x)).sum(axis=1)
        prior_sum = ((np.abs(x) @ np.abs(P0).T) * np.abs(x)).sum(axis=1)
    b_q = b_rows + gamma(rows + 1) * b_sq + b_centre + b_qc
    tot = np.asarray(S, dtype=np.float64)
    b = 0.5 * b_q + 0.5 * b_prior + U * (tot + 2 * prior_sum) + U * np.abs(np.asarray(lp, dtype=np.float64))
    return lp, b


# ------------------------------------------------------------------------------------------------------------------
# forced decisions
# ------------------------------------------------------------------------------------------------------------------
def _grad_mag(meta, arrays, level, theta, path):
    """sum_i |d lp / d theta_i| |theta_i| by central differences in long double (step 1e-6 relative): the first-order
    change of lp when theta moves by a relative u in every coordinate."""
    theta = np.asarray(theta, dtype=np.float64)
    n, d = theta.shape
    out = np.zeros(n)
    for i in range(d):
        hstep = 1e-6 * np.maximum(np.abs(theta[:, i]), 1e-3)
        tp, tm = theta.copy(), theta.copy()
        tp[:, i] += hstep
        tm[:, i] -= hstep
        try:
            fp, _ = _logpost_and_bound(meta, arrays, level, tp, "generic")
            fm, _ = _logpost_and_bound(meta, arrays, level, tm, "generic")
        except Undecidable:
            return np.full(n, np.inf)
        with np.errstate(invalid='ignore'):
            g = np.asarray((fp - fm) / (2 * LD(1) * hstep), dtype=np.float64)
        g = np.where(np.isfinite(g), np.abs(g), 0.0)
        out += g * np.maximum(np.abs(theta[:, i]), 1e-300)
    return out


def _eval(meta, arrays, level, theta, path, n_moves):
    """lp_ld and the bound of a kernel's lp at a point its trajectory reaches after n_moves proposals, each of which
    may round differently from this simulation's: 4 u |theta| per move and coordinate (first order, via the gradient)."""
    lp, b = _logpost_and_bound(meta, arrays, level, theta, path)
    fin = np.isfinite(np.asarray(lp, dtype=np.float64))
    if fin.any():
        g = _grad_mag(meta, arrays, level, theta, path)
        b = b + np.where(fin, 2.0 * 4.0 * U * (n_moves + 1) * g, 0.0)     # 2x: the difference quotient's own error
    return lp, b


def _propose(meta, arrays, s, z, L=None):
    """propose() of the oracle in double: p = s + L z, or pCN's sqrt(1 - 2h) s + sqrt(2h) (m + L z).  L: the problem's
    factor by default, or one factor per chain [nc, d, d] (adaptive Metropolis); an exact zero of L is skipped, per
    chain, as the oracle and the kernels skip it."""
    Lp = np.asarray(arrays["prop_L"] if L is None else L, dtype=np.float64)
    d = s.shape[1]
    acc = np.zeros_like(s)
    for i in range(d):
        first = np.ones(s.shape[0], dtype=bool)
        for j in range(i + 1):
            l = Lp[..., i, j]
            use = (l != 0.0) | (j == i)
            t = l * z[:, j]
            acc[:, i] = np.where(use & first, t, np.where(use, acc[:, i] + t, acc[:, i]))
            first &= ~use
    if meta.get("proposal", "mrw") == "pcn":
        tt = 2.0 * float(meta["pcn_step"])
        a, b = np.sqrt(1.0 - tt), np.sqrt(tt)
        m = np.asarray(arrays.get("pcn_mean", np.zeros(d)), dtype=np.float64)
        return a * s + b * (m + acc)
    return s + acc


def _equal(meta, a, b):
    if meta.get("eq", "exact") == "isclose":
        x, y = a[:, 0], b[:, 0]
        with np.errstate(invalid='ignore'):
            diff = np.abs(y - x)
            close = (diff <= np.abs(1e-9 * y)) | (diff <= np.abs(1e-9 * x))
        return (x == y) | (~np.isinf(x) & ~np.isinf(y) & close)
    return (a == b).all(axis=1)


def _decide(delta, err, want, eta, exact_eta):
    """Uniforms forcing `want` (bool [n]) at distance max(eta, ETA_FACTOR err) from the threshold in log space.
    Returns (u, decided, eta_used): decided is the decision the uniform forces (the wanted one unless only one is
    possible).  delta is long double; NaN (both terms -inf) accepts for every u."""
    n = delta.shape[0]
    e = np.maximum(eta, ETA_FACTOR * err) if not exact_eta else np.full(n, float(eta))
    d = np.asarray(delta, dtype=np.float64)
    u = np.full(n, 0.5)
    out = np.array(want, dtype=bool)
    nan = np.isnan(d)
    out[nan] = True
    pinf = d == np.inf
    out[pinf] = True                                     # a = 1: every u in [0, 1] accepts
    u[pinf] = np.where(want[pinf], 0.5, 1.0)
    minf = d == -np.inf
    out[minf] = False                                    # a = 0: only u = 0 accepts
    fin = np.isfinite(d)
    only_acc = fin & (d >= -e)
    only_rej = fin & (d - e < -700.0)
    out[only_acc] = True
    out[only_rej] = False
    with np.errstate(over='ignore', under='ignore', invalid='ignore'):
        ua = np.asarray(np.exp(np.asarray(delta, dtype=LD) - LD(1) * e), dtype=np.float64)
        ur = np.asarray(np.exp(np.asarray(delta, dtype=LD) + LD(1) * e), dtype=np.float64)
    acc = fin & out
    rej = fin & ~out
    u[acc] = np.minimum(ua[acc], 1.0)
    u[rej] = np.where(d[rej] + e[rej] < -700.0, 2.0 ** -960, np.minimum(ur[rej], 1.0))
    # a reject needs u > a, impossible at u = 1 and a = 1: only when d >= -e, which is forced to accept above
    e_used = np.where(fin, e, np.inf)
    return u, out, e_used


def _follow(delta, err, u):
    """accept_rule on given uniforms, in long double: u <= min(exp(delta), 1), a NaN delta accepting.  Returns
    (u, decision, margin): margin = |delta - log u| - err - 8 u (exp's rounding), > 0 where any double-precision
    evaluation within err of delta decides the same way."""
    with np.errstate(over='ignore', divide='ignore', invalid='ignore'):
        dl = np.asarray(delta, dtype=LD)
        a = np.exp(dl)
        dec = ~(a < 1) | (np.asarray(u, dtype=LD) <= a)
        m = np.asarray(np.abs(dl - np.log(np.asarray(u, dtype=LD))), dtype=np.float64) - err - 8.0 * U
    m = np.where(np.isnan(m) & np.isnan(np.asarray(delta, dtype=np.float64)), np.inf, m)
    return np.asarray(u, dtype=np.float64), dec, m


def forced_schedule(meta, arrays, theta0, z, pattern, eta, exact_eta=False, factor=None, uniforms=None):
    """Simulates chain_step (oracle/yagre_oracle.c: MRW / pCN, two-level delayed acceptance, MLDA with two surrogates)
    in long double on the noise z [nc, ns, J, d] and returns uniforms that force the decisions of `pattern`.

    pattern: dict(coarse=bool [nc, ns, J] (ignored for one level), fine=bool [nc, ns]): the wanted decisions.
    eta: the distance of each uniform from its threshold in log space, at least ETA_FACTOR x the bound on the error of
    that delta (the terms' logpost_bound plus the trajectory term of _eval) -- pass 0 for the smallest allowed.
    exact_eta: use eta as given even below that bound (then no decision is certain; for on / off comparisons only).
    factor: optional per-chain proposal-factor hook, factor(n, j, s) -> L [nc, d, d], called before each proposal
    (transition n, sub-step j, 0 for one level) with the current (sub-)chain state s [nc, d]: adaptive Metropolis.
    uniforms: optional dict(u_c, u_f): decide by these uniforms and the long-double deltas instead of placing
    uniforms (a run playing a kernel on given noise; pattern and eta are ignored).  Then margin_min is the smallest
    margin of a decision beyond its bound (_follow; > 0: every decision is certain).

    Returns dict(u_c [nc, ns, J], u_f [nc, ns], accepted uint8 [nc, ns], coarse_accepted int64 [nc],
    n_accept int64 [nc], evals [3] (as counted by the oracle, without the initial ones), eta_min (smallest eta used
    at a decision that could go either way), coarse / fine: the decisions actually forced, traj [nc, ns, d]: the
    state after each transition, theta: the last one).  Raises Undecidable."""
    levels = int(meta["levels"])
    J = int(meta["J"]) if levels >= 2 else 1
    theta = np.array(theta0, dtype=np.float64)
    nc, d = theta.shape
    ns = z.shape[1]
    assert z.shape == (nc, ns, J, d)
    path = _default_path(meta, arrays)
    lpt = [None] * levels
    bt = [None] * levels
    for l in range(levels):
        lpt[l], bt[l] = _eval(meta, arrays, l, theta, path, 0)
    u_c = np.full((nc, ns, J), 0.5)
    u_f = np.full((nc, ns), 0.5)
    acc = np.zeros((nc, ns), dtype=np.uint8)
    cacc = np.zeros(nc, dtype=np.int64)
    evals = np.zeros(3, dtype=np.int64)
    coarse_forced = np.zeros((nc, ns, J), dtype=bool)
    traj = np.zeros((nc, ns, d))
    eta_min = margin_min = np.inf
    moves = 0

    def track(e, dlt):
        nonlocal eta_min
        fin = np.isfinite(np.asarray(dlt, dtype=np.float64))
        if fin.any():
            eta_min = min(eta_min, float(e[fin].min()))

    def decide(delta, err, which, idx, live):
        nonlocal margin_min
        if uniforms is None:
            return _decide(delta, err, pattern[which][idx], eta, exact_eta)
        u, dec, m = _follow(delta, err, uniforms["u_c" if which == "coarse" else "u_f"][idx])
        if live.any():
            margin_min = min(margin_min, float(m[live].min()))
        return u, dec, np.full(nc, np.inf)

    def propose(s, n, j):
        return _propose(meta, arrays, s, z[:, n, j], None if factor is None else factor(n, j, s))

    for n in range(ns):
        if levels == 1:
            moves += 1
            p = propose(theta, n, 0)
            eq = _equal(meta, p, theta)
            lpp, bp = _eval(meta, arrays, 0, p, path, moves)
            evals[0] += int((~eq).sum())
            with np.errstate(invalid='ignore'):
                delta = lpp - lpt[0]
            u, dec, e = decide(delta, bp + bt[0] + U * np.abs(np.asarray(delta, dtype=np.float64)),
                               "fine", (slice(None), n), ~eq)
            dec &= ~eq
            track(e[~eq], delta[~eq])
            u_f[:, n] = u
            acc[:, n] = dec
            theta = np.where(dec[:, None], p, theta)
            lpt[0] = np.where(dec, lpp, lpt[0])
            bt[0] = np.where(dec, bp, bt[0])
            traj[:, n] = theta
            continue
        s, lpc, bc = theta.copy(), lpt[0].copy(), bt[0].copy()
        for j in range(J):
            moves += 1
            p = propose(s, n, j)
            eq = _equal(meta, p, s)
            lpp, bp = _eval(meta, arrays, 0, p, path, moves)
            evals[0] += int((~eq).sum())
            with np.errstate(invalid='ignore'):
                delta = lpp - lpc
            u, dec, e = decide(delta, bp + bc + U * np.abs(np.asarray(delta, dtype=np.float64)),
                               "coarse", (slice(None), n, j), ~eq)
            dec &= ~eq
            track(e[~eq], delta[~eq])
            u_c[:, n, j] = u
            coarse_forced[:, n, j] = dec
            cacc += dec
            s = np.where(dec[:, None], p, s)
            lpc = np.where(dec, lpp, lpc)
            bc = np.where(dec, bp, bc)
        moved = ~_equal(meta, s, theta)
        top = levels - 1
        lpf, bf = _eval(meta, arrays, top, s, path, moves)
        evals[top] += int(moved.sum())
        if levels == 3:
            lpm, bm = _eval(meta, arrays, 1, s, path, moves)
            evals[1] += int(moved.sum())
            terms = [lpf, lpt[1], -lpm, -lpt[2]]
            bsum = bf + bt[1] + bm + bt[2]
        else:
            lpm, bm = None, None
            terms = [lpf, lpt[0], -lpc, -lpt[1]]
            bsum = bf + bt[0] + bc + bt[1]
        with np.errstate(invalid='ignore'):
            delta = ((terms[0] + terms[1]) + terms[2]) + terms[3]
            mag = sum(np.abs(np.asarray(t, dtype=np.float64)) for t in terms)
        mag = np.where(np.isfinite(mag), mag, 0.0)
        u, dec, e = decide(delta, bsum + 3.0 * U * mag, "fine", (slice(None), n), moved)
        dec &= moved
        track(e[moved], delta[moved])
        u_f[:, n] = u
        acc[:, n] = dec
        theta = np.where(dec[:, None], s, theta)
        lpt[0] = np.where(dec, lpc, lpt[0])
        bt[0] = np.where(dec, bc, bt[0])
        lpt[top] = np.where(dec, lpf, lpt[top])
        bt[top] = np.where(dec, bf, bt[top])
        if levels == 3:
            lpt[1] = np.where(dec, lpm, lpt[1])
            bt[1] = np.where(dec, bm, bt[1])
        traj[:, n] = theta
    return dict(u_c=u_c, u_f=u_f, accepted=acc, coarse_accepted=cacc, n_accept=acc.sum(axis=1, dtype=np.int64),
                evals=evals, eta_min=eta_min, margin_min=margin_min, coarse=coarse_forced, traj=traj, theta=theta)


def random_pattern(nc, ns, J, seed, p=0.5):
    rng = np.random.default_rng(seed)
    return dict(coarse=rng.random((nc, ns, J)) < p, fine=rng.random((nc, ns)) < p)
