"""References for MLDA with two surrogates and tempered levels on the tensor path: the Gaussian law the two-surrogate
recursion leaves invariant, and the tensor path's log-posterior bound for a TEMPERED level.

logpost_reference's tensor path (_tensor_logpost_and_bound) evaluates every level untempered.  tensor_logpost_and_bound
below is the same reference with the tempering fold of abi.cu; for t = 1 it IS logpost_reference's function, so
untempered levels keep their bound term for term.  forced_schedule reaches the tensor bound through
logpost_reference._tensor_logpost_and_bound: a test that forces decisions on tempered tensor-path levels puts this
function in its place for the test (pytest's monkeypatch).

Layouts as in logpost_reference: meta / arrays the lowered problem, theta [n, d]; numpy only."""
import numpy as np

import logpost_reference as R
from logpost_reference import LD, U, gamma

_UNTEMPERED = R._tensor_logpost_and_bound


# ------------------------------------------------------------------------------------------------------------------
# the invariant law
# ------------------------------------------------------------------------------------------------------------------
def level_gaussian_terms(arrays, level):
    """(A, a) of one level of a Gaussian or linear-Gaussian lowered problem: its log-density is -x'A x / 2 + a'x + const.
    A linear level has A = t n G'P G + Q and a = t G'P sum_n (d_n - b) + Q m (t its tempering, 1 when untempered)."""
    pre = f"L{level}_"
    if pre + "g_prec" in arrays:
        P = np.asarray(arrays[pre + "g_prec"], dtype=np.float64)
        return P, P @ np.asarray(arrays[pre + "g_mean"], dtype=np.float64)
    t = float(np.asarray(arrays.get(pre + "tempering", 1.0)).reshape(-1)[0])
    G, b, data = arrays[pre + "G"], arrays[pre + "b"], np.atleast_2d(arrays[pre + "data"])
    Pn, Q, m = arrays[pre + "noise_prec"], arrays[pre + "prior_prec"], arrays[pre + "prior_mean"]
    return t * data.shape[0] * G.T @ Pn @ G + Q, t * G.T @ Pn @ (data - b).sum(axis=0) + Q @ m


def mlda_invariant_gaussian(arrays, levels):
    """(mean, covariance, precision) of the law the device's MLDA leaves invariant on Gaussian levels.  Up to two levels
    it is the target's.  With two surrogates the sub-chain is pi_0-reversible and the screen uses pi_1 in place of pi_0,
    so the chain keeps mu ~ pi_2 pi_0 / pi_1: precision A_2 + A_0 - A_1, linear term a_2 + a_0 - a_1."""
    if levels < 3:
        A, a = level_gaussian_terms(arrays, levels - 1)
    else:
        (A0, a0), (A1, a1), (A2, a2) = (level_gaussian_terms(arrays, l) for l in range(3))
        A, a = A2 + A0 - A1, a2 + a0 - a1
    A = 0.5 * (A + A.T)
    cov = np.linalg.inv(A)
    return cov @ a, cov, A


# ------------------------------------------------------------------------------------------------------------------
# the tempered tensor-path bound
# ------------------------------------------------------------------------------------------------------------------
def tensor_logpost_and_bound(meta, L, theta):
    """logpost_reference._tensor_logpost_and_bound honouring L's tempering t: lp = t logL + logprior in long double.

    abi.cu folds fl(sqrt(t)) into the level's data rows (one more product in sqrt(w_r): the gamma index of de_r grows
    by one, and de_r scales with sqrt(t)) and multiplies q_const by t (one more rounding: gamma_{n_data + data_dim + 5}
    of t q_const).  fl(sqrt(t))^2 = t (1 + 2 delta + delta^2), |delta| <= u, so the data-row sum is off by <= 3 u of
    itself.  The centring term scales with t.  The dense prior's rows are not tempered."""
    t = R._tempering(L)
    if t == 1.0:
        return _UNTEMPERED(meta, L, theta)
    n, d = theta.shape
    G, bvec = np.asarray(L["G"], dtype=np.float64), np.asarray(L["b"], dtype=np.float64)
    data = np.asarray(L["data"], dtype=np.float64)
    nD, dd = data.shape
    Pn = np.diag(np.asarray(L["noise_prec"], dtype=np.float64)).copy()
    assert np.array_equal(np.diag(Pn), np.asarray(L["noise_prec"])), "the tensor path takes diagonal noise"
    thl = np.asarray(theta, dtype=LD)
    F = thl @ np.asarray(G, dtype=LD).T + np.asarray(bvec, dtype=LD)                     # [n, dd]
    dl = np.asarray(data, dtype=LD)
    S = LD(t) * (((F[:, None, :] - dl[None]) ** 2) * np.asarray(Pn, dtype=LD)).sum(axis=(1, 2))
    lpr, _ = R._prior_bound(L, theta)
    lp = -S / 2 + lpr
    if np.any(R._check_range(S) != 0):
        raise R.Undecidable("tensor path: a misfit outside the double range")
    mean = dl.mean(axis=0)
    sw = np.sqrt(nD * Pn)
    st = np.sqrt(t)
    e = st * np.asarray((F - mean) * np.asarray(sw, dtype=LD), dtype=np.float64)        # [n, dd]
    mabs = np.abs(data).sum(axis=0) / nD
    de = st * gamma(d + nD + 7) * sw * (np.abs(theta) @ np.abs(G).T + np.abs(bvec) + mabs)
    q_const = t * float((((dl - mean) ** 2) * np.asarray(Pn, dtype=LD)).sum())
    rows = dd
    b_rows = (2.0 * np.abs(e) * de + de * de).sum(axis=1)
    b_sq = np.asarray((e * e).sum(axis=1), dtype=np.float64)
    b_temper = 3.0 * U * b_sq
    b_centre = t * (2.0 * Pn * np.abs(np.asarray(F - mean, dtype=np.float64)) * gamma(nD)
                    * np.abs(data).sum(axis=0)).sum(axis=1)
    b_qc = gamma(nD + dd + 5) * q_const
    P0 = np.asarray(L["prior_prec"], dtype=np.float64)
    m0 = np.asarray(L["prior_mean"], dtype=np.float64)
    x = np.asarray(theta - m0, dtype=np.float64)
    if np.count_nonzero(P0 - np.diag(np.diag(P0))) > 0:
        Rc = np.linalg.cholesky(0.5 * (P0 + P0.T)).T                                    # R'R = P
        Rx = np.abs(Rc) @ np.abs(np.asarray(theta, dtype=np.float64)).T + (np.abs(Rc) @ np.abs(m0))[:, None]
        dR = gamma(2 * d + 1) * Rx.T
        ex = np.abs(x) @ np.abs(Rc).T
        b_prior = (2.0 * ex * dR + dR * dR).sum(axis=1) + gamma(d + 1) * (ex * ex).sum(axis=1) \
            + U * ((np.abs(x) @ np.abs(P0).T) * np.abs(x)).sum(axis=1)
        b_sq = b_sq + (ex * ex).sum(axis=1)
        rows += d
        prior_sum = np.zeros(n)
    else:
        b_prior = R._quad_bound(P0, x, U * np.abs(x), 4)
        b_prior = b_prior + gamma(d + 2) * ((np.abs(x) @ np.abs(P0).T) * np.abs(x)).sum(axis=1)
        prior_sum = ((np.abs(x) @ np.abs(P0).T) * np.abs(x)).sum(axis=1)
    b_q = b_rows + gamma(rows + 1) * b_sq + b_centre + b_qc + b_temper
    tot = np.asarray(S, dtype=np.float64)
    b = 0.5 * b_q + 0.5 * b_prior + U * (tot + 2 * prior_sum) + U * np.abs(np.asarray(lp, dtype=np.float64))
    return lp, b


def tensor_logpost_bound(meta, arrays, level, theta):
    """(lp_ld [n], bound [n]) of `level` on the tensor path, tempering honoured (logpost_reference.logpost_bound's
    layout)."""
    return tensor_logpost_and_bound(meta, R._lvl(arrays, level), np.asarray(theta, dtype=np.float64))
