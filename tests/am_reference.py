"""Reference of per-chain adaptive Metropolis (AM, DESIGN.md section 5): am_update of generic_mh_kernel
(yagre_mcmc_b200/csrc/generic_kernel.cuh) and of the LV kernel (lv_kernel.cu), vectorised over chains, with absolute
bounds on the moments and the factor a double-precision kernel computes.

The recurrence.  Before every proposal of the MRW chain it drives (the chain itself, or the level-0 sub-chain of
two-level delayed acceptance and MLDA), update(x, t) runs with that chain's current state x and the index t: the
transition count since the last reset for one level, (am_t0 + n) J + j for sub-step j of transition n with J sub-steps.
From t = idle on the state is fed to a full-matrix Welford (n_am = t - idle + 1); once n_am >= max(collection, 2),
every refresh-th update ((n_am - collection) % refresh == 0, refresh 0 meaning 1) forms
C = s (sym(M2) / (n_am - 1) + eps I) and adopts its Cholesky factor if the factorisation succeeds, else keeps the
factor it had.  s is the given scale, or 2.4^2 / d.

Two tracks.
* Double track, in the kernel's order.  Every AM operation of both kernels is explicitly rounded (__dsub_rn,
  __dadd_rn, __dmul_rn, IEEE division and sqrt) and numpy float64 does not fuse, so this track restates them: the
  Welford step, sym(M2) as 0.5 (M2_ij + M2_ji), the division, eps and the scale, and the Cholesky factorisation in the
  kernel's order (chol_kernel: dot products accumulated left to right, the column below the diagonal scaled by the
  reciprocal 1 / l_jj).  The LV kernel's 2 x 2 form is the same sequence of operations.  This track gives the factor
  every proposal uses, hence the states: trajectories and forced decisions are exact expectations.
* Long-double track: the same Welford in long double (64-bit significand: its own error is 2^-11 of the bounds
  below), C_ld = s (sym(M2_ld) / (n_am - 1) + eps I) with the double values of s and eps, and these bounds
  (u = 2^-53, gamma_n = n u / (1 - n u)):

  - mu and M2: diag_reference.welford_tolerance of the states fed so far (the diagnostics' recurrence, the same
    derivation).
  - C: with |dM2| <= T, sym rounds once (0.5 is exact): dS <= (T + T') / 2 + u |S|; the division by n_am - 1:
    dcov <= dS / (n_am - 1) + u |cov|; eps on the diagonal: + u |cov_ii + eps|; the scale: s (...) + u |C|; all times
    (1 + 4u) for the compounding.
  - L: a residual bound that does not depend on conditioning (Higham, Accuracy and Stability, Thm 10.3): the computed
    factor satisfies L L' = C^ + dA, |dA| <= gamma_{d+1} |L||L'|; the reciprocal-then-multiply form rounds once more
    per entry below the diagonal (k = 2), and L L' is formed in long double (k = 3 covers it):
        |L L' - C_ld| <= gamma_{d+3} |L||L'| + dC,
    with exact zeros above the diagonal and a positive diagonal.

Adopt or keep.  Each refresh is classified before its outcome is looked at:
* PD for certain (Higham Thm 10.7): with H = D^-1/2 C D^-1/2, D = diag(C), Cholesky in floating point succeeds
  when lambda_min(H^) > d gamma_{d+2} / (1 - gamma_{d+2}); lambda_min(H^) >= lambda_min(H_ld) - 2 ||D^-1/2 dC D^-1/2||_F
  (the 2 covers the perturbation of D itself, whose relative change is required to stay below 1/4), and eigvalsh's own
  error is covered by 4 d^2 u.
* Not PD for certain, in structural cases only: eps = 0 and a coordinate k whose fed values are all equal -- a chain
  whose every proposal was rejected (every coordinate), or a frozen coordinate (the factor has an exactly-zero row k,
  so the proposal leaves coordinate k unchanged bit for bit).  Then M2's row and column k are exact zeros (the first
  update sets mu_k = x_k exactly, every later difference is 0), so are C's, every L_km (m < k) is 0 * rcp, and the
  pivot c_kk - sum L_km^2 = 0 fails the test s > 0.
* Anything else is undecidable (for example n_am <= d with eps = 0): a forced schedule raises
  logpost_reference.Undecidable rather than rely on it, a value run counts it.

Layouts: theta [nc, d], chain-major like cport.run_injected; device arrays are transposed by the tests.  numpy only.
"""
import numpy as np

import logpost_reference as R
from diag_reference import welford_tolerance
from logpost_reference import LD, U, gamma

# plausible mistakes of an AM update, each a flag of the reference (the negative controls of test_am_reference_cpu)
MISTAKES = ("update_after_proposal",       # the proposal uses the factor from before this update
            "idle_le",                     # idle compared with <=: the state of t = idle is not fed
            "refresh_phase_from_n",        # refresh when n_am % refresh == 0 instead of (n_am - collection) % refresh
            "m2_over_n",                   # covariance M2 / n_am instead of M2 / (n_am - 1)
            "eps_outside_scale",           # C = s cov + eps I instead of s (cov + eps I)
            "scale_from_capacity",         # default scale 2.4^2 / D (the kernel's capacity class) instead of / d
            "failed_reinstalls_problem",   # a failed refresh reinstalls the problem's factor
            "failed_keeps_partial",        # a failed refresh leaves the columns computed before the failing pivot
            "index_counts_transitions",    # two-level index am_t0 + n instead of (am_t0 + n) J + j
            "t0_restarts",                 # the AM index restarts at every launch
            "fed_theta",                   # two-level AM fed the chain state theta instead of the sub-chain state
            "raw_moments")                 # M2 as sum x x' - n mu mu' (cancels for states far from zero)


def cap(x):
    """Capacity class of a parameter dimension (the kernel instances D in {2, 4, 8})."""
    return 2 if x <= 2 else (4 if x <= 4 else 8)


def default_scale(d):
    """abi.cu make_args: 2.4 * 2.4 / d, in double."""
    return 2.4 * 2.4 / float(d)


def chol_kernel(C):
    """cholesky_lower of generic_kernel.cuh (and the LV kernel's 2 x 2 form) in float64 over chains: C [m, d, d] ->
    (L [m, d, d], ok [m], partial [m, d, d]).  A failing pivot stops its chain: partial holds the columns before it."""
    m, d, _ = C.shape
    L = np.zeros_like(C)
    ok = np.ones(m, dtype=bool)
    for j in range(d):
        dot = np.zeros(m)
        for k in range(j):
            dot = dot + L[:, j, k] * L[:, j, k]
        s = C[:, j, j] - dot
        ok &= s > 0.0
        ljj = np.sqrt(np.where(ok, s, 1.0))
        L[:, j, j] = np.where(ok, ljj, L[:, j, j])
        rcp = 1.0 / ljj
        for i in range(j + 1, d):
            dt = np.zeros(m)
            for k in range(j):
                dt = dt + L[:, i, k] * L[:, j, k]
            L[:, i, j] = np.where(ok, (C[:, i, j] - dt) * rcp, L[:, i, j])
    return np.where(ok[:, None, None], L, 0.0), ok, L


class AMTrack:
    """Per-chain AM state of both tracks, fed through update(); the counts a schedule reports."""

    def __init__(self, d, nc, L0, adaptive, mistakes=(), forced=True):
        self.d, self.nc = d, nc
        self.mistakes = frozenset(mistakes)
        assert self.mistakes <= set(MISTAKES), self.mistakes - set(MISTAKES)
        self.forced = forced
        self.idle = int(adaptive.get("idle", 0))
        self.collect = int(adaptive.get("collection", 100))
        self.refresh = max(1, int(adaptive.get("refresh", 1)))
        self.eps = float(adaptive.get("eps", 1e-4))
        sc = float(adaptive.get("scale") or 0.0)
        self.scale = sc if sc > 0 else default_scale(cap(d) if "scale_from_capacity" in self.mistakes else d)
        self.scale_true = sc if sc > 0 else default_scale(d)
        self.L0 = np.asarray(L0, dtype=np.float64)
        self.L = np.tile(self.L0, (nc, 1, 1))
        self.mu = np.zeros((nc, d))
        self.m2 = np.zeros((nc, d, d))
        self.s1 = np.zeros((nc, d))                      # raw_moments only
        self.s2 = np.zeros((nc, d, d))
        self.mu_ld = np.zeros((nc, d), dtype=LD)
        self.m2_ld = np.zeros((nc, d, d), dtype=LD)
        self.fed = []                                    # the states fed, [nc, d] each
        self.n_am = 0
        self.adopted = np.zeros(nc, dtype=np.int64)
        self.kept = np.zeros(nc, dtype=np.int64)
        self.C_ld = np.zeros((nc, d, d), dtype=LD)      # C_ld and its bound at each chain's last adoption
        self.dC = np.zeros((nc, d, d))
        self.refreshes = []                              # (n_am, launch) of every refresh
        self.first_update = None                         # (t, launch) of the first update that fed a state
        self.certain_pd = self.certain_fail = self.undecidable = 0
        self.structural_zero = set()                     # "rejected" / "frozen": kinds of certain failures seen

    # ---- the update --------------------------------------------------------------------------------------------
    def update(self, x, t, launch=0):
        skip = t <= self.idle if "idle_le" in self.mistakes else t < self.idle
        if skip:
            return
        if self.first_update is None:
            self.first_update = (t, launch)
        n_am = t - self.idle + 1
        self.n_am = n_am
        x = np.asarray(x, dtype=np.float64)
        self.fed.append(x.copy())
        # double track
        if "raw_moments" in self.mistakes:
            self.s1 = self.s1 + x
            self.s2 = self.s2 + x[:, :, None] * x[:, None, :]
            self.mu = self.s1 / float(n_am)
            self.m2 = self.s2 - float(n_am) * (self.mu[:, :, None] * self.mu[:, None, :])
        else:
            dl = x - self.mu
            self.mu = self.mu + dl / float(n_am)
            e = x - self.mu
            self.m2 = self.m2 + dl[:, :, None] * e[:, None, :]
        # long-double track
        xl = np.asarray(x, dtype=LD)
        dl = xl - self.mu_ld
        self.mu_ld = self.mu_ld + dl / LD(n_am)
        self.m2_ld = self.m2_ld + dl[:, :, None] * (xl - self.mu_ld)[:, None, :]
        phase = n_am if "refresh_phase_from_n" in self.mistakes else n_am - self.collect
        if n_am >= self.collect and n_am >= 2 and (self.refresh == 1 or phase % self.refresh == 0):
            self._refresh(n_am, launch)

    def _refresh(self, n_am, launch):
        d = self.d
        self.refreshes.append((n_am, launch))
        div = float(n_am if "m2_over_n" in self.mistakes else n_am - 1)
        cov = (0.5 * (self.m2 + self.m2.transpose(0, 2, 1))) / div
        eye = np.eye(d, dtype=bool)[None]
        if "eps_outside_scale" in self.mistakes:
            C = np.where(eye, self.scale * cov + self.eps, self.scale * cov)
        else:
            C = self.scale * np.where(eye, cov + self.eps, cov)
        Ln, ok, partial = chol_kernel(C)
        C_ld, dC = self._c_ld(n_am)
        kind = self._classify(C_ld, dC)
        if not self.mistakes:
            assert np.all(ok[kind == 1]) and not np.any(ok[kind == -1]), "the double track contradicts a certain outcome"
        if self.forced and np.any(kind == 0):
            raise R.Undecidable(f"AM refresh at n_am = {n_am}: chains {np.nonzero(kind == 0)[0][:8]} are near singular")
        self.certain_pd += int((kind == 1).sum())
        self.certain_fail += int((kind == -1).sum())
        self.undecidable += int((kind == 0).sum())
        fail = ~ok
        if "failed_reinstalls_problem" in self.mistakes:
            Lk = np.tile(self.L0, (self.nc, 1, 1))
        elif "failed_keeps_partial" in self.mistakes:
            Lk = partial
        else:
            Lk = self.L
        self.L = np.where(ok[:, None, None], Ln, Lk)
        self.adopted += ok
        self.kept += fail
        self.C_ld = np.where(ok[:, None, None], C_ld, self.C_ld)
        self.dC = np.where(ok[:, None, None], dC, self.dC)

    def _c_ld(self, n_am):
        """C_ld (long double) and the bound dC on |C^ - C_ld| of a correct double evaluation."""
        d = self.d
        s, eps = LD(self.scale_true), LD(self.eps)
        eye = np.eye(d, dtype=bool)[None]
        S = (self.m2_ld + self.m2_ld.transpose(0, 2, 1)) / 2
        cov = S / LD(n_am - 1)
        Cin = np.where(eye, cov + eps, cov)
        C_ld = s * Cin
        _, T = self.welford_bounds()
        f = lambda v: np.abs(np.asarray(v, dtype=np.float64))       # noqa: E731
        dS = 0.5 * (T + T.transpose(0, 2, 1)) + U * f(S)
        dcov = dS / float(n_am - 1) + U * f(cov)
        dCin = dcov + np.where(eye, U * f(Cin), 0.0)
        dC = (1.0 + 4.0 * U) * (float(s) * dCin + U * f(C_ld))
        return C_ld, dC

    def _classify(self, C_ld, dC):
        """+1 PD for certain, -1 not PD for certain (structural), 0 undecidable; per chain."""
        d = self.d
        kind = np.zeros(self.nc, dtype=np.int64)
        X = np.stack(self.fed, axis=1)                                  # [nc, n_am, d]
        const = (X == X[:, :1]).all(axis=1)                             # [nc, d]: coordinates never changed
        if self.eps == 0.0:
            zero = const.any(axis=1)
            kind[zero] = -1
            for c in np.nonzero(zero)[0]:
                self.structural_zero.add("rejected" if const[c].all() else "frozen")
        Cf = np.asarray(C_ld, dtype=np.float64)
        dg = np.einsum('cii->ci', Cf)
        pos = (dg > 0).all(axis=1) & (kind == 0)
        if pos.any():
            dd = np.einsum('cii->ci', dC)[pos]
            g = dg[pos]
            rel_ok = (dd < 0.25 * g).all(axis=1)
            sq = np.sqrt(g)
            H = Cf[pos] / (sq[:, :, None] * sq[:, None, :])
            E = dC[pos] / (sq[:, :, None] * sq[:, None, :])
            lam = np.linalg.eigvalsh(0.5 * (H + H.transpose(0, 2, 1)))[:, 0]
            pert = 2.0 * np.sqrt((E * E).sum(axis=(1, 2))) + 4.0 * d * d * U
            gd = float(gamma(d + 2))
            sure = rel_ok & (lam - pert > d * gd / (1.0 - gd))
            idx = np.nonzero(pos)[0]
            kind[idx[sure]] = 1
        return kind

    # ---- results --------------------------------------------------------------------------------------------
    def welford_bounds(self):
        """(mean [nc, d], M2 [nc, d, d]) bounds of welford_tolerance over the states fed so far."""
        if not self.fed:
            return np.zeros((self.nc, self.d)), np.zeros((self.nc, self.d, self.d))
        return welford_tolerance(np.stack(self.fed, axis=1), (self.mu_ld, self.m2_ld))

    def factor_residual(self, L):
        """(residual [nc, d, d], bound [nc, d, d]) of a factor L [nc, d, d] against each chain's last adopted C_ld
        (bound -1 where the chain never adopted: there L must be the problem's factor bit for bit)."""
        Ll = np.asarray(L, dtype=LD)
        res = np.asarray(np.abs(np.einsum('cik,cjk->cij', Ll, Ll) - self.C_ld), dtype=np.float64)
        A = np.abs(np.asarray(L, dtype=np.float64))
        b = float(gamma(self.d + 3)) * np.einsum('cik,cjk->cij', A, A) + self.dC
        return res, np.where((self.adopted > 0)[:, None, None], b, -1.0)


def check_factor(track, L, label=""):
    """L [nc, d, d] is a factor the track allows: the problem's bit for bit where no refresh was adopted, else lower
    triangular with a positive diagonal within the residual bound of the last adopted C_ld."""
    L = np.asarray(L, dtype=np.float64)
    never = track.adopted == 0
    assert np.array_equal(L[never], np.broadcast_to(track.L0, L[never].shape)), (label, "factor of a chain that never adopted")
    a = ~never
    assert np.all(np.triu(L[a], 1) == 0.0) and np.all(np.einsum('cii->ci', L[a]) > 0.0), (label, "factor shape")
    res, b = track.factor_residual(L)
    assert np.all(res[a] <= b[a]), (label, "factor residual", float(np.max(res[a] / np.maximum(b[a], 1e-300))))


def _index(n, j, J, launch_start, t0, mistakes):
    if "t0_restarts" in mistakes:
        n = n - launch_start
    else:
        n = n + t0
    return n if "index_counts_transitions" in mistakes else n * J + j


def am_schedule(meta, arrays, adaptive, theta0, z, pattern=None, eta=0.0, uniforms=None, launches=None, track=None,
                t0=0, mistakes=(), exact_eta=False):
    """logpost_reference.forced_schedule with the AM proposal-factor hook.  Forced (pattern, eta) or following given
    uniforms (dict(u_c, u_f): the run of a kernel on that noise, decided by the long-double deltas).

    launches: the transitions of each launch (default one launch); t0: am_steps before this schedule; track: an
    AMTrack to continue (set_state(keep_adaptation=True), or the next launches of the same handle).
    Returns forced_schedule's dict plus track (the AMTrack), am_steps, and what the schedule reached:
      adopted / kept [nc]: refreshes adopted and kept per chain; first_refresh: n_am of the first refresh;
      boundary_refreshes: refreshes in a later launch than the refresh (or first update) before them;
      first_update_launch: the launch of the first update that fed a state; certain_fail_kinds."""
    levels = int(meta["levels"])
    J = int(meta["J"]) if levels >= 2 else 1
    theta0 = np.asarray(theta0, dtype=np.float64)
    nc, d = theta0.shape
    ns = z.shape[1]
    if track is None:
        track = AMTrack(d, nc, arrays["prop_L"], adaptive, mistakes, forced=uniforms is None)
    launches = list(launches or [ns])
    assert sum(launches) == ns, (launches, ns)
    starts = np.repeat(np.cumsum([0] + launches[:-1]), launches)
    lidx = np.repeat(np.arange(len(launches)), launches)
    cur = dict(theta=theta0.copy(), n=-1)
    ms = track.mistakes

    def factor(n, j, s):
        if "fed_theta" in ms and levels >= 2:
            if j == 0:
                cur["theta"] = s.copy()
            x = cur["theta"]
        else:
            x = s
        t = _index(n, j, J, starts[n], t0, ms)
        before = track.L
        track.update(x, t, int(lidx[n]))
        return before if "update_after_proposal" in ms else track.L

    n_ref0 = len(track.refreshes)
    out = R.forced_schedule(meta, arrays, theta0, z, pattern, eta, exact_eta=exact_eta, factor=factor,
                            uniforms=uniforms)
    refs = track.refreshes[n_ref0:]
    prev = track.first_update[1] if track.first_update is not None else 0
    boundary = 0
    for _, lch in refs:
        boundary += lch > prev
        prev = lch
    out.update(track=track, am_steps=t0 + ns, adopted=track.adopted.copy(), kept=track.kept.copy(),
               first_refresh=track.refreshes[0][0] if track.refreshes else None, boundary_refreshes=boundary,
               first_update_launch=None if track.first_update is None else track.first_update[1],
               am_mean=track.mu.copy(), am_m2=track.m2.copy(), am_L=track.L.copy())
    return out
