"""CPU: the diagnostics reference (tests/diag_reference.py) the GPU tests hold the kernels to -- its pre-state convention
on the reference's own Welford fixtures, its agreement with the oracle's accumulator, its restart handling, and that its
bounds let a correct double-precision accumulator through while they stop the plausible wrong ones."""
import numpy as np
import pytest

from diag_reference import (check_welford, pre_states, welford_reference, welford_tolerance, U)
from golden_io import load

WELFORD_FIXTURES = ["mrw_gauss1d", "mrw_gauss2d_iid", "mrw_gauss2d_diag", "mrw_gauss2d_dense"]


def _welford_steps(x):
    """The step kernels' recurrence in float64, full co-moment, [nc, n, d] -> w_mean [d, nc], w_m2 [d, d, nc]."""
    nc, n, d = x.shape
    m, m2 = np.zeros((nc, d)), np.zeros((nc, d, d))
    for t in range(n):
        dl = x[:, t] - m
        m = m + dl / float(t + 1)
        e = x[:, t] - m
        m2 += dl[:, :, None] * e[:, None, :]
    return m.T.copy(), m2.transpose(1, 2, 0).copy()


def _welford_runs(pre):
    """The tensor path's run-length form (diagonal): the accumulators change only where the state does."""
    nc, n, d = pre.shape
    wm, wv = np.zeros((nc, d)), np.zeros((nc, d))
    for c in range(nc):
        wn, run = 0.0, 0.0
        for t in range(n):
            run += 1.0
            if t == n - 1 or np.any(pre[c, t + 1] != pre[c, t]):
                n1 = wn + run
                c1 = run / n1
                c2 = wn * c1
                dl = pre[c, t] - wm[c]
                wm[c] = dl * c1 + wm[c]
                wv[c] = dl * dl * c2 + wv[c]
                wn, run = n1, 0.0
    return wm.T.copy(), wv.T.copy()


def _random_walk(rng, nc, n, d, offset=0.0, p_move=0.4, stuck=()):
    """Metropolis-like sequences: a chain stays where it is with probability 1 - p_move."""
    x = np.empty((nc, n, d))
    x[:, 0] = offset + rng.standard_normal((nc, d))
    for t in range(1, n):
        move = rng.random(nc) < p_move
        move[list(stuck)] = False
        x[:, t] = np.where(move[:, None], x[:, t - 1] + 0.3 * rng.standard_normal((nc, d)), x[:, t - 1])
    return x


@pytest.mark.parametrize("name", WELFORD_FIXTURES)
def test_pre_state_convention_reproduces_the_reference_welford_fixtures(name):
    """The reference's FullDiagnostics (diagnostics.py:91-94) on its own runs: pre-states = traj[:, :ns]."""
    meta, a = load(name)
    ns = a["u_f"].shape[1]
    traj = a["traj"]                                          # [nc, ns + 1, d]
    samples = traj[:, 1:].transpose(1, 2, 0)                  # device layout [ns, d, nc]
    pre = pre_states(traj[:, 0], [samples])
    assert np.array_equal(pre, traj[:, :ns])
    mu, R = welford_reference(pre)
    tm, t2 = welford_tolerance(pre, (mu, R))
    var = np.einsum('cii->ci', R) / (ns - 1)
    assert np.all(np.abs(a["welford_mean"] - mu.astype(np.float64)) <= tm)
    assert np.all(np.abs(a["welford_var"] * (ns - 1) - np.einsum('cii->ci', R).astype(np.float64))
                  <= np.einsum('cii->ci', t2))
    np.testing.assert_allclose(a["welford_mean"], mu.astype(np.float64), rtol=1e-14)
    np.testing.assert_allclose(a["welford_var"], var.astype(np.float64), rtol=1e-14)


def test_reference_agrees_with_the_oracle_accumulator():
    """cport.welford (the oracle's diagonal Welford) inside the bounds, also for data far from zero."""
    from oracle import cport
    rng = np.random.default_rng(3)
    for offset in (0.0, 1e3, -1e6):
        pre = _random_walk(rng, 6, 700, 3, offset=offset)
        mu, R = welford_reference(pre)
        tm, t2 = welford_tolerance(pre, (mu, R))
        for c in range(pre.shape[0]):
            m, v = cport.welford(pre[c])
            assert np.all(np.abs(m - mu[c].astype(np.float64)) <= tm[c]), offset
            assert np.all(np.abs(v * (pre.shape[1] - 1) - np.diag(R[c]).astype(np.float64)) <= np.diag(t2[c])), offset


def test_pre_states_across_a_keep_diagnostics_restart():
    """run(3); set_state(y, keep_diagnostics=True); run(2); run(4) on 2 chains, by hand."""
    th0 = np.array([[0.0, 1.0], [5.0, 6.0]])
    r1 = np.arange(12, dtype=np.float64).reshape(3, 2, 2) + 100       # [ns, d, nc]
    r2 = np.arange(8, dtype=np.float64).reshape(2, 2, 2) + 200
    r3 = np.arange(16, dtype=np.float64).reshape(4, 2, 2) + 300
    y = np.array([[-1.0, -2.0], [-3.0, -4.0]])
    pre = pre_states(th0, [r1, r2, r3], [None, y, None])
    for c in range(2):
        want = [th0[c], r1[0, :, c], r1[1, :, c],             # r1's last sample is replaced by the restart state
                y[c], r2[0, :, c],
                r2[1, :, c], r3[0, :, c], r3[1, :, c], r3[2, :, c]]
        assert np.array_equal(pre[c], np.array(want))
    assert pre.shape == (2, 9, 2)
    # a run of zero transitions contributes nothing, and the restart state is the first pre-state of the next run
    assert np.array_equal(pre_states(th0, [r1, r1[:0], r2], [None, y, None]), pre_states(th0, [r1, r2], [None, y]))


def test_correct_accumulators_pass_and_wrong_ones_fail():
    """The bounds admit the kernels' double-precision recurrences (step form, full co-moment; run-length form,
    diagonal) and are exact for chains that never moved, while each of the mistakes the GPU tests look for fails."""
    rng = np.random.default_rng(11)
    nc, n, d = 40, 300, 2
    pre = _random_walk(rng, nc, n, d, offset=-0.7, stuck=(0, 7))
    wm, w2 = _welford_steps(pre)
    assert check_welford(wm, w2, n, pre, "steps") == 2
    rm, rv = _welford_runs(pre)
    assert check_welford(rm, rv, n, pre, "run length") == 2

    def fails(mean, m2, welford_n=n, p=pre):
        with pytest.raises(AssertionError):
            check_welford(mean, m2, welford_n, p)

    bad = w2.copy()                      # W01 from d0 * e0 instead of d0 * e1
    x = pre
    m = np.zeros((nc, d)); bad[0, 1] = 0.0
    for t in range(n):
        dl = x[:, t] - m
        m = m + dl / float(t + 1)
        bad[0, 1] += dl[:, 0] * (x[:, t, 0] - m[:, 0])
    fails(wm, bad)
    post = np.concatenate([pre[:, 1:], pre[:, -1:] + 0.5], axis=1)     # post-transition states
    fails(*_welford_steps(post))
    fails(wm, w2, welford_n=n + 1)                                      # one step counted twice
    fails(*_welford_runs(pre[:, :-3]), welford_n=n)                    # the last states never reach the accumulators
    wm1 = wm.copy(); wm1[0, 3] += 8 * n * U * abs(wm1[0, 3]) + 1e-12    # a mean off by more than its bound
    fails(wm1, w2)
    still = w2.copy(); still[0, 0, 0] = 1e-300                          # a stuck chain must have exactly zero M2
    fails(wm, still)
