"""CPU: tests/logpost_reference.py pinned before any GPU test relies on it.

* The oracle's yo_logpost stays within logpost_bound of the long-double reference on every model family, and a
  double-precision port of the tensor path's centred, folded formulation stays within the tensor-path bound.
* Plausible wrong evaluations exceed the bound on the same problems (each problem is chosen so that the mistake is
  visible: the dropped row / design point has a misfit far above the bound, the prior mean is far from zero, ...).
* C_RK4 covers a fresh measurement.
* forced_schedule's uniforms make the oracle's replay (cport.run_injected) take exactly the scheduled decisions.
"""
import numpy as np
import pytest

import bench_problems as bp
import logpost_reference as R
from support import (SCHEDULES, TENSOR, dense_noise_linear, dense_prior_tensor, fixture, lv_tempered,
                     qconst_tensor, schedule_noise)

from oracle import cport


def _oracle(meta, arrays, level, theta):
    pb = cport.Problem(meta, arrays)
    return np.array([cport.logpost(pb, level, t) for t in np.asarray(theta, dtype=np.float64)])


def _err(got, ref):
    return np.abs(np.asarray(got, dtype=np.longdouble) - ref).astype(np.float64)


def _theta(meta, n, seed, scale=0.3):
    if meta["model"] == "lv":
        return bp.lv_initial_states(n, seed=seed) + np.random.default_rng(seed).uniform(-1, 1, (n, 2)) * 0.5
    return scale * np.random.default_rng(seed).standard_normal((n, int(meta["dim"])))


GENERIC = {
    "gauss2d": bp.gauss2d_problem,
    "gauss1d_isclose": lambda: fixture("mrw_gauss1d"),
    "gauss3_levels": lambda: fixture("mlda3_gauss2d"),
    "linear_c3": lambda: bp.linear_problem(True),
    "linear_tempered": lambda: fixture("mlda_linear_tempered"),
    "linear_dense_noise_d5": dense_noise_linear,
    "linear_d8_dd8": lambda: bp.big_linear_problem(8, 8, 5, two_level=True, seed=4),
    "lv_two_level": lambda: bp.lv_problem(True),
    "lv_single_level": lambda: bp.lv_problem(False),
    "lv_tempered": lv_tempered,
    "lv_pcn": bp.lv_pcn_problem,
    "lv_one_design_point": lambda: bp.lv_problem(True, n_data=1),
    "lv_300_design_points": lambda: bp.lv_problem(True, n_data=300, Nc=16, Nf=48),
}


@pytest.mark.parametrize("name", sorted(GENERIC))
def test_oracle_within_bound(name):
    meta, arrays = GENERIC[name]()
    th = _theta(meta, 40, 3)
    for l in range(int(meta["levels"])):
        lp, b = R.logpost_bound(meta, arrays, l, th)
        assert np.all(np.isfinite(np.asarray(lp, dtype=np.float64))), name
        e = _err(_oracle(meta, arrays, l, th), lp)
        assert np.all(e <= b), (name, l, float((e / b).max()))
        assert np.all(b <= 1e-9 * (1.0 + np.abs(np.asarray(lp, dtype=np.float64)))), (name, l, float(b.max()))


def test_lv_nonfinite_region_is_minus_inf_or_undecidable():
    """theta = (6, 6): RK4 overflows in long double too; the reference says -inf with a zero bound, like the oracle."""
    meta, arrays = bp.lv_problem(True)
    th = np.array([[6.0, 6.0], [5.5, 6.5]])
    for l in range(2):
        lp, b = R.logpost_bound(meta, arrays, l, th)
        assert np.all(np.asarray(lp, dtype=np.float64) == -np.inf) and np.all(b == 0.0)
        assert np.all(_oracle(meta, arrays, l, th) == -np.inf)


def test_undecidable_points_raise():
    """A linear misfit whose square lands within 2^16 of DBL_MAX may or may not overflow in double."""
    meta, arrays = bp.linear_problem(False)
    th = np.array([[1.0, 1.0], [1e154, 0.0]])
    with pytest.raises(R.Undecidable):
        R.logpost_bound(meta, arrays, 0, th)


# ------------------------------------------------------------------------------------------------------------------
# the tensor path's centred, folded formulation (abi.cu's host side + linear_dmma_kernel.cu's logpost_tile)
# ------------------------------------------------------------------------------------------------------------------
def tensor_logpost_f64(arrays, theta, qc_f32=False, R_f32=False, qc_rel=0.0):
    data = np.asarray(arrays["L0_data"], dtype=np.float64)
    G, b = arrays["L0_G"], arrays["L0_b"]
    prec = np.diag(arrays["L0_noise_prec"])
    P0, m0 = arrays["L0_prior_prec"], arrays["L0_prior_mean"]
    nD, dd = data.shape
    d = G.shape[1]
    mean = data.sum(axis=0) / nD
    dq = data.astype(np.float32).astype(np.float64) if qc_f32 else data
    mq = dq.sum(axis=0) / nD
    q_const = float((prec * ((dq - mq) ** 2).sum(axis=0)).sum()) * (1.0 + qc_rel)
    sw = np.sqrt(nD * prec)
    Gw = sw[:, None] * G
    bdw = sw * (b - mean)
    dense = np.count_nonzero(P0 - np.diag(np.diag(P0))) > 0
    pprec = np.zeros(d) if dense else np.diag(P0)
    if dense:
        Ps = 0.5 * (P0 + P0.T)
        Lp = (np.linalg.cholesky(Ps.astype(np.float32)).astype(np.float64) if R_f32 else cport.cholesky(Ps))
        Rm = Lp.T
        Gw = np.vstack([Gw, Rm])
        bdw = np.concatenate([bdw, -(Rm @ m0)])
    th = np.asarray(theta, dtype=np.float64)
    e = th @ Gw.T + bdw
    q = (e * e).sum(axis=1)
    x = th - m0
    return -0.5 * (q + q_const) + (-0.5 * (pprec * x * x).sum(axis=1))


@pytest.mark.parametrize("name", sorted(TENSOR))
def test_tensor_path_formulation_within_its_bound(name):
    """The folded formulation in double (and the oracle's textbook one) within the tensor-path bound."""
    meta, arrays = TENSOR[name]()
    th = 0.05 * np.random.default_rng(1).standard_normal((30, int(meta["dim"])))
    lp, b = R.logpost_bound(meta, arrays, 0, th, path="tensor")
    assert R._default_path(meta, arrays) == "tensor"
    for got in (tensor_logpost_f64(arrays, th), _oracle(meta, arrays, 0, th)):
        e = _err(got, lp)
        assert np.all(e <= b), (name, float((e / b).max()))
    if name == "near_zero":
        assert np.abs(np.asarray(lp, dtype=np.float64)).max() < 1e-2
    if name == "q_const_dominated":
        assert np.all(b < 1e-12 * R._tensor_q_const(arrays))


# ------------------------------------------------------------------------------------------------------------------
# wrong evaluations fail the bound
# ------------------------------------------------------------------------------------------------------------------
def _lv_logpost_stage_point(arrays, level, theta, consts_f32=False):
    """The LV kernel's evaluation ported to numpy: stage-point RK4, misfit quad form, pairwise sum, prior."""
    pre = f"L{level}_"
    design, data = arrays[pre + "design"], arrays[pre + "data"]
    alpha, gamma_, T, N = arrays[pre + "lv"]
    out = []
    for t in np.asarray(theta, dtype=np.float64):
        x, y = R.lv_rk4_stage_point_f64(np.exp(t[0]), np.exp(t[1]), design[:, 0].copy(), design[:, 1].copy(),
                                        alpha, gamma_, T, int(N), consts_f32=consts_f32)
        r = np.stack([x - data[:, 0], y - data[:, 1]], axis=1)
        q = np.einsum('nk,kl,nl->n', r, arrays[pre + "noise_prec"], r)
        xm = t - arrays[pre + "prior_mean"]
        out.append(-0.5 * q.sum() + (-0.5 * xm @ arrays[pre + "prior_prec"] @ xm))
    return np.array(out)


def _wrong_cases():
    lin_meta, lin = bp.big_linear_problem(5, 4, 3, two_level=False, seed=12)
    lin = dict(lin, L0_prior_mean=np.full(5, 0.7))
    lv_meta, lv = bp.lv_problem(True)
    tmeta, tarr = fixture("mlda_linear_tempered")
    tl = [l for l in range(2) if f"L{l}_tempering" in tarr][0]
    other = 1 - tl
    moved = {k: v for k, v in tarr.items() if k != f"L{tl}_tempering"}
    moved[f"L{other}_tempering"] = tarr[f"L{tl}_tempering"]
    h_meta, h_arr = bp.lv_problem(False)
    a, g, T, N = h_arr["L0_lv"]
    h_wrong = dict(h_arr, L0_lv=np.array([a, g, T * N / (N + 1), N]))
    qc_meta, qc = qconst_tensor()
    dp_meta, dp = dense_prior_tensor()
    return {
        # name: (meta, arrays, level, wrong evaluation (theta -> lp), path)
        "last_data_row_dropped": (lin_meta, lin, 0, lambda th: _oracle(
            lin_meta, dict(lin, L0_data=lin["L0_data"][:-1]), 0, th), "generic"),
        "last_design_point_dropped": (lv_meta, lv, 0, lambda th: _oracle(
            lv_meta, dict(lv, L0_data=lv["L0_data"][:-1], L0_design=lv["L0_design"][:-1]), 0, th), "lv"),
        "prior_mean_ignored": (lin_meta, lin, 0, lambda th: _oracle(
            lin_meta, dict(lin, L0_prior_mean=np.zeros(5)), 0, th), "generic"),
        "tempering_on_the_wrong_level": (tmeta, tarr, other, lambda th: _oracle(tmeta, moved, other, th), "generic"),
        "lv_rate_constants_float32": (lv_meta, lv, 1, lambda th: _lv_logpost_stage_point(lv, 1, th, True), "lv"),
        "h_is_T_over_N_plus_1": (h_meta, h_arr, 0, lambda th: _oracle(h_meta, h_wrong, 0, th), "lv"),
        "q_const_from_float32_data": (qc_meta, qc, 0, lambda th: tensor_logpost_f64(qc, th, qc_f32=True), "tensor"),
        "R_from_float32_cholesky": (dp_meta, dp, 0, lambda th: tensor_logpost_f64(dp, th, R_f32=True), "tensor"),
    }


WRONG = sorted(_wrong_cases())


@pytest.mark.parametrize("name", WRONG)
def test_wrong_evaluation_exceeds_the_bound(name):
    meta, arrays, level, wrong, path = _wrong_cases()[name]
    th = _theta(meta, 12, 5, scale=0.05)
    lp, b = R.logpost_bound(meta, arrays, level, th, path=path)
    e = _err(wrong(th), lp)
    assert np.all(e > b), (name, float((e / b).min()))


def test_lv_stage_point_port_within_bound():
    """The right version of the port used above stays within the LV bound (so the float32 case fails for its
    constants, not for the port)."""
    meta, arrays = bp.lv_problem(True)
    th = _theta(meta, 12, 5, scale=0.05)
    lp, b = R.logpost_bound(meta, arrays, 1, th)
    assert np.all(_err(_lv_logpost_stage_point(arrays, 1, th), lp) <= b)


def test_c_rk4_covers_a_fresh_measurement():
    got = R.measure_c_rk4(2000, (16, 64, 512), seed=99)
    assert max(got.values()) <= R.C_RK4, got
    assert max(got.values()) >= R.C_RK4 / 40, got        # the constant is not vacuous either


# ------------------------------------------------------------------------------------------------------------------
# the schedules force the chosen decisions in the oracle
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("eta", [0.0, 1e-7, 1e-3])
@pytest.mark.parametrize("name", sorted(SCHEDULES))
def test_forced_schedule_reproduced_by_the_oracle(name, eta):
    make, nc, ns, init = SCHEDULES[name]
    meta, arrays = make()
    th0 = init(nc)
    z = schedule_noise(meta, nc, ns, 17)
    J = z.shape[2]
    pat = R.random_pattern(nc, ns, J, seed=23)
    sch = R.forced_schedule(meta, arrays, th0, z, pat, eta)
    ref = cport.run_injected(cport.Problem(meta, arrays), th0, z, sch["u_c"], sch["u_f"])
    assert np.array_equal(ref["accepted"], sch["accepted"]), name
    assert np.array_equal(ref["coarse_accepted"], sch["coarse_accepted"]), name
    assert np.array_equal(ref["accepted"].sum(axis=1), sch["n_accept"]), name
    assert np.array_equal(ref["n_evals"] - nc * (np.arange(3) < int(meta["levels"])), sch["evals"]), name
    assert np.array_equal(ref["traj"][:, -1], sch["theta"]), name
    # about half of the decisions that could go either way follow the pattern's accepts
    rate = sch["accepted"].mean()
    assert 0.15 < rate < 0.85, (name, rate)
    assert sch["eta_min"] >= eta
