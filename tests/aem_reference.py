"""Long-double reference of the adaptive-error-model chain (chain_step_aem, oracle/yagre_oracle.c; aem_mh_kernel,
yagre_mcmc_b200/csrc/generic_kernel.cuh), vectorised over chains, with absolute bounds on every value a
double-precision kernel computes.

The coarse log-posterior of an AEM chain is not a function of theta alone: it depends on the chain's error model
(the Welford mean and co-moment of e = F_fine - F_coarse over its accepted fine steps), on the inflated noise
precision derived from it, and on an LRU(3) cache whose values are NOT refreshed when the error model changes.  So
this module simulates the whole chain: the coarse sub-chain (proposal queried first, then the state, mrw.py), the
fine screen pi_f(P) + pi_c(theta) - pi_c(P) - pi_f(theta), the error-model update on an accepted fine step
(query_model_evaluation touches the cache on a hit and counts a model evaluation on a miss), and the cache.

What is exact and what is bounded.  Proposals are computed in double in the kernel's order (logpost_reference._propose:
p = s + L z, the products and sums rounded one by one, as __dmul_rn / __dadd_rn and the oracle's unfused C), so every
state and every cache key is the kernel's bit for bit: hit or miss is structural, and the cache keys, cache.n, aem_n
and the evaluation counts are exact expectations.  Every value is carried in long double with an absolute bound on
the distance of any double-precision evaluation in the kernel's or the oracle's order (u = 2^-53,
gamma_n = n u / (1 - n u), Higham 3.1-3.5):

* Forward model F = G theta + b, d products and d sums (fused or not): |dF_k| <= gamma_{d+1} mag_k,
  mag_k = sum_j |G_kj theta_j| + |b_k|.  Two levels whose rows k are identical compute F_f,k and F_c,k by the same
  operations on the same operands, so their error component is exactly 0.
* Error sample e = F_f - F_c is a cancellation, so its bound is relative to the operands, not to |e|:
  |de_k| <= dF_f,k + dF_c,k + u |e~_k| <= gamma_{d+2} (mag_f,k + mag_c,k)   (0 for identical rows).
* Welford over n samples e_i with errors de_i <= de_max (diag_reference.welford_tolerance's argument on the
  perturbed samples e~_i, plus the perturbation itself; amax = max|e_i|, S = sum|e_i|):
    |d mean| <= 4 n u (amax + de_max) + de_max
    |d M2|   <= gamma_n M2 + 16 n u (amax + de_max)(amax + |mean| + 2 de_max)
                + 4 de_max (S + n |mean|) + 4 n de_max^2
  (the first two terms are the recurrence's own roundings on samples of magnitude <= amax + de_max, the last two
  bound |sum (e~_i - mean~)^2 - sum (e_i - mean)^2| <= 2 sum|e_i - mean| 2 de_max + n (2 de_max)^2).
* Inflated precision p_k = 1 / (s mv_k + 1 / p0_k), mv_k = M2_k / (n - 1):  |d mv_k| <= (1 + u) |d M2_k| / (n - 1)
  + u mv_k; with beta = max_k |d mv_k|, min and max over k move by <= beta, max(., 1e-6) and min(., 100) are
  1-Lipschitz, and the quotient s = 2 mx / mnv (mnv = max(mn, 1e-6) >= 1e-6 > beta) moves by
  ds <= 2 beta (mnv + mx) / (mnv (mnv - beta)) + 2 u s; the clamp then moves by at most
  max(min(s + ds, 100) - min(s, 100), min(s, 100) - min(s - ds, 100)) (0 when s - ds > 100).  Then v = s mv + 1/p0 moves by
  dv <= (1 + 2u) (ds (mv + dmv) + s dmv + u (s mv + 1/p0 + v)), and 1/v by dv / (v (v - dv)) + u / v.
* Coarse log-posterior -1/2 sum_n sum_k p_k r_nk^2 + prior, r = F_c - data (+ mean once aem_n >= min_data):
  |dr| <= gamma_{d+3} (mag_c + |data| + |mean|) + |d mean|; each term moves by dp r^2 + (p + dp)(2 |r| dr + dr^2),
  the dd-term inner sum rounds within gamma_{dd+2} of sum p r^2 and the n_data-term outer sum (numpy's pairwise
  order, restated by np_stream_sum; any order) within gamma_{n_data} of its sum; -1/2 is exact and the prior
  (logpost_reference._prior_bound) is added with one more rounding: u (|S/2| + |prior|).
* A cache entry keeps the value and bound of the evaluation that filled it: that IS the stale semantics.
* The fine level is the plain level-1 log-posterior: logpost_reference.logpost_bound's generic path.
* Decisions: coarse delta = lp(P) - lp(s), bound b_P + b_s + u |delta|; fine delta = ((pi_f(P) + pi_c(theta))
  - pi_c(P)) - pi_f(theta), bound the sum of the four plus 3 u (sum of magnitudes).  A decision u <= min(exp(delta), 1)
  is certain when |delta - log u| exceeds that bound plus 8 u (exp's rounding, <= 2 ulp, in log space).

Layouts: theta [nc, d]; z [nc, ns, J, d]; u_c [nc, ns, J]; u_f [nc, ns]; accepted [nc, ns] (chain-major, as
cport.run_injected).  numpy only; no torch.
"""
import numpy as np

import logpost_reference as R
from logpost_reference import LD, U, ETA_FACTOR, gamma

EXP_SLACK = 8.0 * U              # exp(delta) rounded (<= 2 ulp), in log space
FLOOR, CLAMP = 1e-6, 100.0       # noise.py:41-46: scaling = min(2 max(var) / max(min(var), 1e-6), 100)

# plausible mistakes of an AEM step, each a flag of the simulation (the negative controls of test_aem_reference_cpu)
MISTAKES = ("invalidate_on_update",     # cache emptied when the error model changes (fresh values)
            "shift_after_min_data",     # mean shift from aem_n > min_data instead of >=
            "inflate_from_min_data",    # inflation from aem_n >= min_data instead of >
            "variance_over_n",          # M2 / n instead of M2 / (n - 1)
            "no_clamp",                 # heuristic without min(., 100)
            "no_floor",                 # heuristic without max(., 1e-6)
            "update_no_touch",          # the update's cache hit does not move the entry back
            "cache_2", "cache_4",       # LRU of 2 or 4 entries
            "error_sign",               # e = F_c - F_f
            "drop_data_row")            # the last data row left out of the likelihoods


def cap(x):
    """Capacity class of a parameter or data dimension (the kernel instances D, DD in {2, 4, 8})."""
    return 2 if x <= 2 else (4 if x <= 4 else 8)


class _Problem:
    def __init__(self, meta, arrays, mistakes):
        self.meta, self.mistakes = meta, frozenset(mistakes)
        assert self.mistakes <= set(MISTAKES), self.mistakes - set(MISTAKES)
        a = {k: np.asarray(v, dtype=np.float64) for k, v in arrays.items()}
        if "drop_data_row" in self.mistakes:
            a = dict(a, L0_data=a["L0_data"][:-1], L1_data=a["L1_data"][:-1])
        self.arrays = a
        self.d = int(meta["dim"])
        self.J = int(meta["J"])
        self.min_data = int(meta["aem"]["min_data"])
        self.heuristic = bool(meta["aem"]["heuristic"])
        self.Gc, self.bc, self.Gf, self.bf = a["L0_G"], a["L0_b"], a["L1_G"], a["L1_b"]
        self.data = a["L0_data"]
        self.dd = self.data.shape[1]
        P0 = a["L0_noise_prec"]
        assert np.array_equal(P0, np.diag(np.diag(P0))), "AEM takes diagonal noise"
        assert "L0_tempering" not in a or float(a["L0_tempering"]) == 1.0
        self.p0 = np.diag(P0).copy()
        self.c0 = 1.0 / np.asarray(self.p0, dtype=LD)
        self.prior = dict(prior_mean=a["L0_prior_mean"], prior_prec=a["L0_prior_prec"])
        self.same = (self.Gc == self.Gf).all(axis=1) & (self.bc == self.bf)
        self.cap = 2 if "cache_2" in self.mistakes else (4 if "cache_4" in self.mistakes else 3)


def _forward(G, b, x):
    F = np.asarray(x, dtype=LD) @ np.asarray(G, dtype=LD).T + np.asarray(b, dtype=LD)
    mag = np.abs(x) @ np.abs(G).T + np.abs(b)
    return F, mag


class _Chains:
    """Per-chain state of the simulation: the error model (long-double Welford plus the running magnitudes its bound
    needs), the inflated precision and the cache."""

    def __init__(self, pb, nc):
        d, dd, c = pb.d, pb.dd, pb.cap
        self.pb = pb
        self.en = np.zeros(nc, dtype=np.int64)
        self.mu = np.zeros((nc, dd), dtype=LD)
        self.m2 = np.zeros((nc, dd), dtype=LD)
        self.amax = np.zeros((nc, dd))
        self.demax = np.zeros((nc, dd))
        self.sabs = np.zeros((nc, dd))
        self.have = np.zeros(nc, dtype=bool)
        self.prec = np.tile(np.asarray(pb.p0, dtype=LD), (nc, 1))
        self.bprec = np.zeros((nc, dd))
        self.keys = np.zeros((nc, c, d))
        self.val = np.zeros((nc, c), dtype=LD)
        self.vb = np.zeros((nc, c))
        self.cn = np.zeros(nc, dtype=np.int64)
        self.model_evals = np.zeros(nc, dtype=np.int64)
        self.clamped = self.unclamped = self.floored = 0

    # ---- error model ------------------------------------------------------------------------------------------
    def mean_bound(self, rows):
        n = self.en[rows][:, None].astype(np.float64)
        a, de = self.amax[rows], self.demax[rows]
        return 4.0 * n * U * (a + de) + de

    def m2_bound(self, rows):
        n = self.en[rows][:, None].astype(np.float64)
        a, de, S = self.amax[rows], self.demax[rows], self.sabs[rows]
        mu = np.abs(np.asarray(self.mu[rows], dtype=np.float64))
        m2 = np.asarray(self.m2[rows], dtype=np.float64)
        return gamma(n) * m2 + 16.0 * n * U * (a + de) * (a + mu + 2.0 * de) + 4.0 * de * (S + n * mu) + 4.0 * n * de * de

    def update(self, rows, x):
        pb = self.pb
        Fc, mc = _forward(pb.Gc, pb.bc, x)
        Ff, mf = _forward(pb.Gf, pb.bf, x)
        e = (Fc - Ff) if "error_sign" in pb.mistakes else (Ff - Fc)
        de = np.where(pb.same[None, :], 0.0, gamma(pb.d + 2) * (mf + mc))
        self.en[rows] += 1
        n = self.en[rows][:, None].astype(LD)
        dl = e - self.mu[rows]
        self.mu[rows] += dl / n
        self.m2[rows] += dl * (e - self.mu[rows])
        ea = np.abs(np.asarray(e, dtype=np.float64))
        self.amax[rows] = np.maximum(self.amax[rows], ea)
        self.demax[rows] = np.maximum(self.demax[rows], de)
        self.sabs[rows] += ea
        self.refresh(rows)

    def refresh(self, rows):
        pb = self.pb
        md = pb.min_data
        on = self.en[rows] >= md if "inflate_from_min_data" in pb.mistakes else self.en[rows] > md
        rows = rows[on]
        if rows.size == 0:
            return
        n = self.en[rows][:, None]
        div = n if "variance_over_n" in pb.mistakes else n - 1
        with np.errstate(divide='ignore', invalid='ignore'):
            mv = self.m2[rows] / np.asarray(div, dtype=LD)
            bmv = (1.0 + U) * self.m2_bound(rows) / np.maximum(div, 1).astype(np.float64) \
                + U * np.abs(np.asarray(mv, dtype=np.float64))
            if pb.heuristic:
                mn, mx = mv.min(axis=1), mv.max(axis=1)
                beta = bmv.max(axis=1)
                mnv = mn if "no_floor" in pb.mistakes else np.maximum(mn, LD(FLOOR))
                s_raw = 2 * mx / mnv
                s = s_raw if "no_clamp" in pb.mistakes else np.minimum(s_raw, LD(CLAMP))
                mnf, mxf, sf = (np.asarray(v, dtype=np.float64) for v in (mnv, mx, s_raw))
                ds = np.where(mnf > beta, 2.0 * beta * (mnf + mxf) / (mnf * (mnf - beta)) + 2.0 * U * sf, np.inf)
                if "no_clamp" not in pb.mistakes:       # min(., 100) moves by no more than its argument, often by 0
                    ds = np.maximum(np.minimum(sf + ds, CLAMP) - np.minimum(sf, CLAMP),
                                    np.minimum(sf, CLAMP) - np.minimum(sf - ds, CLAMP))
                self.clamped += int((s_raw > CLAMP).sum())
                self.unclamped += int((s_raw <= CLAMP).sum())
                self.floored += int((mn < FLOOR).sum())
                s, ds = s[:, None], ds[:, None]
            else:
                s, ds = LD(1), np.zeros((rows.size, 1))
            v = s * mv + pb.c0[None, :]
            sf = np.asarray(s, dtype=np.float64)
            mvf = np.asarray(mv, dtype=np.float64)
            vf = np.asarray(v, dtype=np.float64)
            dv = (1.0 + 2.0 * U) * (ds * (mvf + bmv) + sf * bmv
                                    + U * (sf * mvf + np.asarray(pb.c0, dtype=np.float64)[None, :] + vf))
            self.prec[rows] = 1 / v
            self.bprec[rows] = np.where(vf > dv, dv / (vf * (vf - dv)) + U / vf, np.inf)
        self.have[rows] = True

    # ---- coarse log-posterior and the cache ----------------------------------------------------------------------
    def coarse(self, rows, x):
        """The AEM coarse log-posterior of the chains rows at x [m, d] with their current error model: (lp, bound)."""
        pb = self.pb
        F, mag = _forward(pb.Gc, pb.bc, x)
        data = np.asarray(pb.data, dtype=LD)
        r = F[:, None, :] - data[None]                                           # [m, nD, dd]
        shift = self.en[rows] > pb.min_data if "shift_after_min_data" in pb.mistakes else self.en[rows] >= pb.min_data
        mu = np.where(shift[:, None], self.mu[rows], LD(0))
        bmu = np.where(shift[:, None], self.mean_bound(rows), 0.0)
        r = r + mu[:, None, :]
        dr = gamma(pb.d + 3) * (mag[:, None, :] + np.abs(pb.data)[None] + np.abs(np.asarray(mu, dtype=np.float64))[:, None, :]) \
            + bmu[:, None, :]
        p = np.where(self.have[rows][:, None], self.prec[rows], np.asarray(pb.p0, dtype=LD)[None])
        bp = np.where(self.have[rows][:, None], self.bprec[rows], 0.0)
        t = p[:, None, :] * r * r
        S = t.sum(axis=(1, 2))
        rf, pf = np.abs(np.asarray(r, dtype=np.float64)), np.asarray(p, dtype=np.float64)
        bS = (bp[:, None, :] * rf * rf + (pf + bp)[:, None, :] * (2.0 * rf * dr + dr * dr)).sum(axis=(1, 2)) \
            + (gamma(pb.dd + 2) + gamma(pb.data.shape[0])) * np.asarray(S, dtype=np.float64)
        lpr, bpr = R._prior_bound(pb.prior, x)
        lp = -S / 2 + lpr
        b = 0.5 * bS + bpr + U * (0.5 * np.asarray(S, dtype=np.float64) + np.abs(np.asarray(lpr, dtype=np.float64)))
        self.model_evals[rows] += 1
        return lp, b

    def find(self, rows, x):
        c = self.pb.cap
        eq = (self.keys[rows] == x[:, None, :]).all(axis=2) & (np.arange(c)[None, :] < self.cn[rows][:, None])
        return np.where(eq.any(axis=1), eq.argmax(axis=1), -1)

    def touch(self, rows, idx):
        """AEMCache._move_to_back: entry idx of each chain in rows to the newest position."""
        n = self.cn[rows][:, None]
        i = idx[:, None]
        p = np.arange(self.pb.cap)[None, :]
        src = np.where(p < i, p, np.where(p < n - 1, p + 1, np.where(p == n - 1, i, p)))
        rr = rows[:, None]
        self.keys[rows] = self.keys[rr, src]
        self.val[rows] = self.val[rr, src]
        self.vb[rows] = self.vb[rr, src]

    def add(self, rows, x, v, b):
        c = self.pb.cap
        full = rows[self.cn[rows] >= c]
        if full.size:
            self.keys[full, :c - 1] = self.keys[full, 1:].copy()
            self.val[full, :c - 1] = self.val[full, 1:].copy()
            self.vb[full, :c - 1] = self.vb[full, 1:].copy()
            self.cn[full] = c - 1
        k = self.cn[rows]
        self.keys[rows, k] = x
        self.val[rows, k] = v
        self.vb[rows, k] = b
        self.cn[rows] += 1

    def query(self, rows, x, stale=None):
        """query_log_likelihood at x [m, d] for the chains rows: (lp, bound); a hit returns the cached (possibly
        stale) value and moves it back, a miss evaluates and adds.  stale: a bool array [m] set where a hit's value is
        more than 100x the bounds away from a fresh evaluation."""
        lp = np.zeros(rows.size, dtype=LD)
        b = np.zeros(rows.size)
        idx = self.find(rows, x)
        hit = idx >= 0
        if hit.any():
            hr = rows[hit]
            lp[hit] = self.val[hr, idx[hit]]
            b[hit] = self.vb[hr, idx[hit]]
            if stale is not None:
                evals = self.model_evals[hr].copy()
                fv, fb = self.coarse(hr, x[hit])
                self.model_evals[hr] = evals
                stale[hit] |= np.abs(np.asarray(fv - lp[hit], dtype=np.float64)) > 100.0 * (fb + b[hit])
            self.touch(hr, idx[hit])
        if (~hit).any():
            mr = rows[~hit]
            v, vb = self.coarse(mr, x[~hit])
            lp[~hit], b[~hit] = v, vb
            self.add(mr, x[~hit], v, vb)
        return lp, b

    def after_accept(self, rows, x):
        """query_model_evaluation of the accepted proposal, then the error-model update."""
        if rows.size == 0:
            return
        idx = self.find(rows, x)
        hit = idx >= 0
        if "update_no_touch" not in self.pb.mistakes and hit.any():
            self.touch(rows[hit], idx[hit])
        self.model_evals[rows[~hit]] += 1
        if "invalidate_on_update" in self.pb.mistakes:
            self.cn[rows] = 0
        self.update(rows, x)


def _fine(pb, x):
    meta = dict(pb.meta)
    meta.pop("aem", None)
    return R._logpost_and_bound(meta, pb.arrays, 1, x, "generic")


def _margin(delta, u):
    with np.errstate(divide='ignore'):
        lu = np.log(np.asarray(u, dtype=LD))
    return np.asarray(np.abs(np.asarray(delta, dtype=LD) - lu), dtype=np.float64)


def _accepts(delta, u):
    """accept_rule in long double: u <= min(exp(delta), 1) (a NaN delta accepts)."""
    with np.errstate(over='ignore'):
        a = np.exp(np.asarray(delta, dtype=LD))
    return ~(a < 1) | (np.asarray(u, dtype=LD) <= a)


def _simulate(meta, arrays, theta0, z, u_c=None, u_f=None, accepted=None, force=None, mistakes=(), stale=False):
    """The AEM chain on noise z.  Coarse decisions are taken from u_c by the reference's own delta, or forced;
    fine decisions follow `accepted` if given, else u_f by the reference's delta, or are forced.
    force: None or (pattern, eta, exact_eta): uniforms placed by logpost_reference._decide."""
    pb = _Problem(meta, arrays, mistakes)
    theta = np.array(theta0, dtype=np.float64)
    nc, d = theta.shape
    ns, J = z.shape[1], pb.J
    assert z.shape == (nc, ns, J, d), z.shape
    ch = _Chains(pb, nc)
    m0 = dict(meta)
    m0.pop("aem", None)
    lp0, b0 = R._logpost_and_bound(m0, pb.arrays, 0, theta, "generic")
    lp1, b1 = _fine(pb, theta)
    uc = np.full((nc, ns, J), 0.5) if u_c is None else np.array(u_c, dtype=np.float64)
    uf = np.full((nc, ns), 0.5) if u_f is None else np.array(u_f, dtype=np.float64)
    acc = np.zeros((nc, ns), dtype=np.uint8)
    cacc = np.zeros(nc, dtype=np.int64)
    fine_evals = 0
    out = dict(lp0=np.zeros((nc, ns), dtype=LD), b0=np.zeros((nc, ns)), lp1=np.zeros((nc, ns), dtype=LD),
               b1=np.zeros((nc, ns)), traj=np.zeros((nc, ns, d)),
               margin_c=np.full((nc, ns, J), np.inf), bound_c=np.zeros((nc, ns, J)),
               margin_f=np.full((nc, ns), np.inf), bound_f=np.zeros((nc, ns)), delta_f=np.full((nc, ns), np.nan, dtype=LD),
               aem_n_path=np.zeros((nc, ns + 1), dtype=np.int64), stale_decisions=0, eta_min=np.inf)
    out["lp0_init"], out["b0_init"], out["lp1_init"], out["b1_init"] = lp0.copy(), b0.copy(), lp1.copy(), b1.copy()
    allr = np.arange(nc)

    def decide(delta, bound, u, want):
        if force is None:
            return u, _accepts(delta, u)
        pattern_eta, eta, exact = force
        uu, dec, e = R._decide(delta, bound + EXP_SLACK, want, eta, exact)
        fin = np.isfinite(np.asarray(delta, dtype=np.float64))
        if fin.any():
            out["eta_min"] = min(out["eta_min"], float(e[fin].min()))
        return uu, dec

    for n in range(ns):
        s = theta.copy()
        lps_cur = None
        for j in range(J):
            p = R._propose(meta, arrays, s, z[:, n, j])
            live = allr[~R._equal(meta, p, s)]
            if live.size == 0:
                continue
            st = np.zeros(live.size, dtype=bool) if stale else None
            lpp, bp = ch.query(live, p[live], st)
            lps, bs = ch.query(live, s[live], st)
            delta = lpp - lps
            bound = bp + bs + U * np.abs(np.asarray(delta, dtype=np.float64))
            want = force[0]["coarse"][live, n, j] if force is not None else None
            u, dec = decide(delta, bound, uc[live, n, j], want)
            uc[live, n, j] = u
            out["margin_c"][live, n, j] = _margin(delta, u)
            out["bound_c"][live, n, j] = bound + EXP_SLACK
            if stale:
                out["stale_decisions"] += int(st.sum())
            mv = live[dec]
            s[mv] = p[mv]
            cacc[mv] += 1
        moved = allr[~R._equal(meta, s, theta)]
        if moved.size:
            lpf, bf = _fine(pb, s[moved])
            fine_evals += moved.size
            st = np.zeros(moved.size, dtype=bool) if stale else None
            lct, bct = ch.query(moved, theta[moved], st)
            lcs, bcs = ch.query(moved, s[moved], st)
            delta = ((lpf + lct) - lcs) - lp1[moved]
            mag = sum(np.abs(np.asarray(t, dtype=np.float64)) for t in (lpf, lct, lcs, lp1[moved]))
            bound = bf + bct + bcs + b1[moved] + 3.0 * U * mag
            want = force[0]["fine"][moved, n] if force is not None else None
            u, dec = decide(delta, bound, uf[moved, n], want)
            uf[moved, n] = u
            if accepted is not None and force is None:
                dec = np.asarray(accepted[moved, n], dtype=bool)
            out["margin_f"][moved, n] = _margin(delta, u)
            out["delta_f"][moved, n] = delta
            out["bound_f"][moved, n] = bound + EXP_SLACK
            if stale:
                out["stale_decisions"] += int(st.sum())
            a = moved[dec]
            ch.after_accept(a, s[a])
            theta[a] = s[a]
            lp0[a], b0[a] = lcs[dec], bcs[dec]
            lp1[a], b1[a] = lpf[dec], bf[dec]
            acc[a, n] = 1
        if accepted is not None and force is None:
            assert not np.asarray(accepted)[np.setdiff1d(allr, moved), n].any(), \
                f"step {n}: an accepted transition whose sub-chain did not move"
        out["lp0"][:, n], out["b0"][:, n], out["lp1"][:, n], out["b1"][:, n] = lp0, b0, lp1, b1
        out["traj"][:, n] = theta
        out["aem_n_path"][:, n + 1] = ch.en
    mb, m2b = ch.mean_bound(allr), ch.m2_bound(allr)
    out.update(u_c=uc, u_f=uf, accepted=acc, coarse_accepted=cacc, n_accept=acc.sum(axis=1, dtype=np.int64),
               theta=theta, aem_n=ch.en.copy(), aem_mean=ch.mu, aem_mean_bound=mb, aem_m2=ch.m2, aem_m2_bound=m2b,
               cache_keys=ch.keys, cache_val=ch.val, cache_bound=ch.vb, cache_n=ch.cn,
               coarse_evals=int(ch.model_evals.sum()), aem_model_evals=ch.model_evals.copy(), fine_evals=fine_evals,
               clamped=ch.clamped, unclamped=ch.unclamped, floored=ch.floored, lp0_final=lp0, b0_final=b0,
               lp1_final=lp1, b1_final=b1)
    return out


def aem_follow(meta, arrays, theta0, z, u_c, u_f, accepted, mistakes=()):
    """Follows a run's noise and its fine accept flags (e.g. a kernel's): coarse decisions are the reference's own
    (check that margin_c > bound_c wherever a sub-step was taken).  Returns a dict of
      lp0 / b0, lp1 / b1 [nc, ns]: the coarse value as last evaluated and the fine value after each step, with bounds;
      traj [nc, ns, d], theta: the states (exact);
      aem_n, aem_mean / aem_mean_bound, aem_m2 / aem_m2_bound: the error model at the end;
      cache_keys [nc, 3, d], cache_val / cache_bound [nc, 3], cache_n: the cache, oldest entry first;
      coarse_evals (coarse model evaluations), fine_evals, coarse_accepted [nc], n_accept [nc];
      margin_c / bound_c [nc, ns, J], margin_f / bound_f [nc, ns]: |delta - log u| of each decision against its
      bound (inf where no decision was taken); delta_f [nc, ns]: the fine screens' deltas (NaN where none)."""
    return _simulate(meta, arrays, theta0, z, u_c, u_f, accepted=np.asarray(accepted), mistakes=mistakes)


def aem_run(meta, arrays, theta0, z, u_c, u_f, mistakes=()):
    """The chain deciding every step by its own long-double deltas (a reference run playing a kernel)."""
    return _simulate(meta, arrays, theta0, z, u_c, u_f, mistakes=mistakes)


def aem_forced_schedule(meta, arrays, theta0, z, pattern, eta, exact_eta=False, mistakes=()):
    """forced_schedule for AEM: uniforms at max(eta, ETA_FACTOR x bound) from each threshold forcing `pattern`
    (logpost_reference.random_pattern's dict(coarse [nc, ns, J], fine [nc, ns])).  Returns _simulate's dict (u_c, u_f,
    the decisions as forced in accepted / coarse_accepted / n_accept, counters, aem_n and moments with bounds) plus:
      stale_decisions: decisions with a cached term more than 100x its bounds away from a fresh evaluation;
      aem_n_path [nc, ns + 1]: aem_n of every chain before the first and after every step;
      clamped / unclamped / floored: error-model refreshes whose heuristic clamped at 100, did not, or floored;
      eta_min: the smallest eta used at a decision that could go either way."""
    return _simulate(meta, arrays, theta0, z, force=(pattern, eta, exact_eta), mistakes=mistakes, stale=True)
