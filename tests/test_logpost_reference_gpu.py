"""GPU: every kernel's log-posteriors against the long-double reference (tests/logpost_reference.py) within derived
absolute bounds, and its accept decisions on uniforms placed at known distances from the threshold.

a. Values: Philox runs without a record (the production instances: the warp-specialised kernel, FREE_NOISE on the
   tensor path); state()["logpost"], every stored step of run(logpost=True) and ens.logpost() at the same points
   must be within logpost_bound of the reference.
b. Forced decisions: z and forced_schedule's uniforms injected, all steps in one call; the accept flags,
   coarse_accepted, n_accept and the counters must equal the schedule exactly, at eta = the smallest allowed
   (ETA_FACTOR x the bound of each delta), 1e-7 and 1e-3.
c. Exact semantics of accept_rule: u = 0 accepts everything (lp = -inf proposals too), delta == 0 with u = 1 accepts,
   a NaN delta accepts; below the bound, early rejection on and off give bit-identical results."""
import numpy as np
import pytest
import torch

import bench_problems as bp
import logpost_reference as R
from support import SCHEDULES, TENSOR, dense_noise_linear, ensemble, fixture, lv_tempered, schedule_noise, value_case

pytestmark = pytest.mark.gpu


# ------------------------------------------------------------------------------------------------------------------
# a. values
# ------------------------------------------------------------------------------------------------------------------
LV_VALUES = {
    # name: (problem, chains, sample, stored, kw)
    "headline": (lambda: bp.lv_problem(True), 65536, 2048, 256, {}),
    "single_level": (lambda: bp.lv_problem(False), 3000, 512, 128, {}),
    "pcn": (bp.lv_pcn_problem, 1000, 512, 128, {}),
    "tempered_level0": (lv_tempered, 500, None, 128, {}),
    "one_design_point": (lambda: bp.lv_problem(True, n_data=1), 700, None, None, {}),
    "300_design_points": (lambda: bp.lv_problem(True, n_data=300, Nc=16, Nf=48, prop_var=2e-4), 97, None, None, {}),
    "fine_one_segment": (lambda: bp.lv_problem(True), 1024, 256, 64, dict(rk4_segment=512)),
    "fine_several_segments": (lambda: bp.lv_problem(True), 1024, 256, 64, dict(rk4_segment=96)),
    "proposals_reach_minus_inf": (lambda: bp.lv_problem(False, prop_var=4.0), 2000, 512, 128, {}),
}


@pytest.mark.parametrize("name", sorted(LV_VALUES))
def test_lv_kernel_logpost_values(name):
    make, nc, sample, stored, kw = LV_VALUES[name]
    meta, arrays = make()
    value_case(meta, arrays, bp.lv_initial_states(nc), sample=sample, stored=stored, **kw)


SMALL = [(d, dd) for d in (1, 2, 3, 5, 8) for dd in (1, 2, 4, 5, 8)]


@pytest.mark.parametrize("k", range(len(SMALL)))
def test_one_chain_per_thread_logpost_values(k):
    """d x data_dim, one and two levels in turn, a dense noise precision every third shape."""
    d, dd = SMALL[k]
    meta, arrays = bp.big_linear_problem(d, dd, 3, two_level=k % 2 == 1, J=2, seed=60 + k)
    if k % 3 == 0:
        A = np.random.default_rng(k).standard_normal((dd, dd))
        P = A @ A.T / dd + 10.0 * np.eye(dd)
        arrays = dict(arrays, **{f"L{l}_noise_prec": P for l in range(meta["levels"])})
    value_case(meta, arrays, 0.1 * np.random.default_rng(k).standard_normal((257, d)))


GENERIC_VALUES = {
    "three_level_gauss": (lambda: fixture("mlda3_gauss2d"), lambda n: np.tile([0.5, 1.0], (n, 1)), 33),
    "isclose_1d": (lambda: fixture("mrw_gauss1d"), lambda n: np.full((n, 1), -1.0), 100),
    "one_chain": (lambda: bp.linear_problem(True), lambda n: np.zeros((n, 2)), 1),
    "40001_chains": (lambda: bp.linear_problem(True), lambda n: np.zeros((n, 2)), 40001),
    "dense_noise_d5": (dense_noise_linear, lambda n: 0.1 * np.random.default_rng(1).standard_normal((n, 5)), 999),
    "tempered_surrogate": (lambda: fixture("mlda_linear_tempered"), lambda n: np.zeros((n, 2)), 500),
    "adaptive_metropolis": (bp.gauss2d_problem, lambda n: np.tile([-1.0, 2.0], (n, 1)), 300),
}


@pytest.mark.parametrize("name", sorted(GENERIC_VALUES))
def test_generic_logpost_values(name):
    make, init, nc = GENERIC_VALUES[name]
    meta, arrays = make()
    kw = dict(adaptive=dict(idle=1, collection=3, refresh=1)) if name == "adaptive_metropolis" else {}
    value_case(meta, arrays, init(nc), sample=2048, **kw)


@pytest.mark.parametrize("name", sorted(TENSOR))
def test_tensor_path_logpost_values(name):
    meta, arrays = TENSOR[name]()
    d = int(meta["dim"])
    value_case(meta, arrays, 0.01 * np.random.default_rng(4).standard_normal((2500, d)), sample=512)


# ------------------------------------------------------------------------------------------------------------------
# b. forced decisions
# ------------------------------------------------------------------------------------------------------------------
def _inject(z, sch):
    return dict(z=np.ascontiguousarray(z.transpose(1, 2, 3, 0)),
                u_c=np.ascontiguousarray(sch["u_c"].transpose(1, 2, 0)),
                u_f=np.ascontiguousarray(sch["u_f"].transpose(1, 0)))


def run_forced(meta, arrays, th0, z, sch, **kw):
    ens = ensemble(meta, arrays, th0.shape[0], seed=5, **kw)
    ens.set_state(th0)
    out = ens.run(z.shape[1], samples=True, accepted=True, logpost=True, inject=_inject(z, sch))
    torch.cuda.synchronize()
    res = dict(out={k: out[k].clone() for k in ("samples", "accepted", "logpost")},
               state={k: v.clone() for k, v in ens.state().items() if torch.is_tensor(v)},
               counters=ens.counters(), skipped=ens.skipped_evals())
    ens.close()
    return res


def check_forced(meta, sch, res, label):
    nc = sch["accepted"].shape[0]
    acc = res["out"]["accepted"].cpu().numpy().T
    assert np.array_equal(acc, sch["accepted"]), (label, np.argwhere(acc != sch["accepted"])[:5])
    c = res["counters"]
    assert np.array_equal(res["state"]["n_accept"].cpu().numpy(), sch["n_accept"]), label
    assert c["coarse_accepted"] == int(sch["coarse_accepted"].sum()), label
    assert c["transitions"] == acc.size and c["accepted"] == int(acc.sum()), label
    lv = int(meta["levels"])
    ev = sch["evals"]
    want = {1: dict(fine_evals=ev[0]), 2: dict(coarse_evals=ev[0], fine_evals=ev[1]),
            3: dict(coarse_evals=ev[0], mid_evals=ev[1], fine_evals=ev[2])}[lv]
    assert {k: c[k] for k in want} == {k: int(v) for k, v in want.items()}, (label, c, want)
    assert 0.05 < acc.mean() < 0.95, label           # at eta = 1e-3 many screens can only accept
    return nc


FORCED_ETAS = [0.0, 1e-7, 1e-3]
FORCED_SIZES = {"lv_two_level": (256, 4), "lv_single_level": (256, 4), "lv_pcn": (256, 4),
                "tensor_single_level": (128, 6), "tensor_two_level": (128, 5)}


def _forced_on_off(meta, arrays, th0, ns, label, seed=100, **kw):
    """Forced runs at every eta with early rejection on and off; returns the integrations skipped by the on-runs."""
    nc = th0.shape[0]
    skipped = 0
    for i, eta in enumerate(FORCED_ETAS):
        z = schedule_noise(meta, nc, ns, seed + i)
        sch = R.forced_schedule(meta, arrays, th0, z, R.random_pattern(nc, ns, z.shape[2], seed=seed + 100 + i), eta)
        print(f"{label} eta={eta}: smallest eta used {sch['eta_min']:.3g}")
        if meta["model"] == "lv" and meta["levels"] == 2:
            on = run_forced(meta, arrays, th0, z, sch, early_reject=True, **kw)
            off = run_forced(meta, arrays, th0, z, sch, early_reject=False, **kw)
            check_forced(meta, sch, on, f"{label} eta={eta} on")
            check_forced(meta, sch, off, f"{label} eta={eta} off")
            skipped += on["skipped"]
            print(f"{label} eta={eta}: {on['skipped']} integrations skipped")
        else:
            check_forced(meta, sch, run_forced(meta, arrays, th0, z, sch), f"{label} eta={eta}")
    return skipped


@pytest.mark.parametrize("name", sorted(SCHEDULES))
def test_forced_decisions(name):
    """Every case family of the CPU schedule test, on its kernel; the LV two-level case with early rejection on and
    off."""
    make, nc, ns, init = SCHEDULES[name]
    nc, ns = FORCED_SIZES.get(name, (max(nc, 512), ns))
    meta, arrays = make()
    _forced_on_off(meta, arrays, init(nc), ns, name)


def test_forced_decisions_with_early_rejection_certifying():
    """Units still queued when the first misfits of a phase arrive (8,192 chains: about 550 level-0 units per CTA and
    phase, taken 128 at a time by 128-thread CTAs), so early rejection certifies some of the forced rejections: the
    certify path ran with uniforms next to the threshold and must decide exactly as the full evaluation does.  With
    the default launch geometry a CTA takes all units of a phase in its first grab at this size, and nothing is skipped.
    Nc = 16, Nf = 48 keep the long-double schedule affordable."""
    meta, arrays = bp.lv_problem(True, Nc=16, Nf=48)
    skipped = _forced_on_off(meta, arrays, bp.lv_initial_states(8192), 2, "lv_two_level_8192", seed=500,
                             threads_per_block=128)
    assert skipped > 0


# ------------------------------------------------------------------------------------------------------------------
# c. exact semantics
# ------------------------------------------------------------------------------------------------------------------
def _dyadic_gauss():
    arrays = dict(prop_L=np.eye(2), L0_g_mean=np.zeros(2), L0_g_prec=np.diag([2.0, 0.5]), L0_g_logconst=np.array(-1.5))
    return dict(model="gauss", dim=2, levels=1, J=1, eq="exact"), arrays


def _dyadic_linear(d, dd, two_level, nd=1):
    """b = data = 0, dyadic G, power-of-two precisions: every log-posterior is exact, and lp(-theta) == lp(theta)."""
    rng = np.random.default_rng(d * 100 + dd)
    meta = dict(model="linear", dim=d, levels=2 if two_level else 1, J=3 if two_level else 1, eq="exact")
    arrays = dict(prop_L=np.eye(d))
    for l in range(meta["levels"]):
        G = rng.integers(-4, 5, (dd, d)) / 4.0
        arrays.update({f"L{l}_G": G, f"L{l}_b": np.zeros(dd), f"L{l}_data": np.zeros((nd, dd)),
                       f"L{l}_noise_prec": 4.0 * np.eye(dd), f"L{l}_prior_mean": np.zeros(d),
                       f"L{l}_prior_prec": 0.5 * np.eye(d)})
    return meta, arrays


EXACT = {
    # name: problem with a zero-mean target, dyadic theta0
    "gauss": _dyadic_gauss,
    "linear_single_level": lambda: _dyadic_linear(3, 4, False),
    "linear_two_level": lambda: _dyadic_linear(3, 4, True),
    "tensor_single_level": lambda: _dyadic_linear(12, 20, False),
    "tensor_two_level": lambda: _dyadic_linear(20, 33, True),
}


def _reflect_noise(meta, th0, ns):
    """z that proposes theta' = -theta at every (sub-)step with prop_L = I."""
    nc, d = th0.shape
    J = int(meta["J"])
    z = np.empty((nc, ns, J, d))
    s = th0.copy()
    for n in range(ns):
        for j in range(J):
            z[:, n, j] = -2.0 * s
            s = -s
    return z


@pytest.mark.parametrize("name", sorted(EXACT))
def test_delta_exactly_zero_with_u_one_accepts(name):
    meta, arrays = EXACT[name]()
    nc, ns, d, J = 300, 5, int(meta["dim"]), int(meta["J"])
    th0 = np.random.default_rng(1).integers(-8, 9, (nc, d)) / 8.0
    th0[th0.sum(axis=1) == 0, 0] = 0.5                               # theta != -theta
    th0[(th0 == 0).all(axis=1)] = 0.5
    z = _reflect_noise(meta, th0, ns)
    lp0 = [np.asarray(R.logpost_ld(meta, arrays, l, th0), dtype=np.float64) for l in range(meta["levels"])]
    for l in range(meta["levels"]):
        assert np.array_equal(lp0[l], np.asarray(R.logpost_ld(meta, arrays, l, -th0), dtype=np.float64))
    sch = dict(u_c=np.ones((nc, ns, J)), u_f=np.ones((nc, ns)))
    res = run_forced(meta, arrays, th0, z, sch)
    assert res["out"]["accepted"].cpu().numpy().all(), name
    assert res["counters"]["coarse_accepted"] == (nc * ns * J if meta["levels"] == 2 else 0)
    want = th0 * (-1.0) ** (ns * J)
    assert np.array_equal(res["state"]["theta"].cpu().numpy().T, want)
    for l in range(meta["levels"]):                                  # dyadic problems: the kernels are exact too
        assert np.array_equal(res["state"]["logpost"][l].cpu().numpy(), lp0[l]), (name, l)


U_ZERO = {
    # name: (problem, initial states, noise scale, kw)
    "lv_two_level_early_rejection": (lambda: bp.lv_problem(True), bp.lv_initial_states, 20.0, {}),
    "lv_single_level": (lambda: bp.lv_problem(False), bp.lv_initial_states, 20.0, {}),
    "gauss": (bp.gauss2d_problem, lambda n: np.zeros((n, 2)), 1e3, {}),
    "linear_two_level": (lambda: bp.linear_problem(True), lambda n: np.zeros((n, 2)), 1e3, {}),
    "tensor_two_level": (lambda: bp.big_linear_problem(32, 96, 2, two_level=True, J=3),
                         lambda n: np.zeros((n, 32)), 1e3, {}),
}


@pytest.mark.parametrize("name", sorted(U_ZERO))
def test_u_zero_accepts_everything(name):
    """Proposals far out (LV: into the overflow region, lp = -inf) are all accepted at u = 0."""
    make, init, scale, kw = U_ZERO[name]
    meta, arrays = make()
    nc, ns = 512, 4
    J = int(meta["J"])
    th0 = init(nc)
    z = scale * np.random.default_rng(3).standard_normal((nc, ns, J, int(meta["dim"])))
    sch = dict(u_c=np.zeros((nc, ns, J)), u_f=np.zeros((nc, ns)))
    res = run_forced(meta, arrays, th0, z, sch, **kw)
    assert res["out"]["accepted"].cpu().numpy().all(), name
    assert res["counters"]["coarse_accepted"] == (nc * ns * J if meta["levels"] == 2 else 0)
    if meta["model"] == "lv":
        assert np.any(res["state"]["logpost"].cpu().numpy() == -np.inf)   # the -inf region was reached


NAN_DELTA = {
    # name: (problem, initial state inside the overflow region, proposal step relative to it)
    "lv_two_level": (lambda: bp.lv_problem(True), np.array([6.0, 6.0]), 0.01),
    "lv_single_level": (lambda: bp.lv_problem(False), np.array([6.0, 6.0]), 0.01),
    "gauss": (bp.gauss2d_problem, np.array([1e200, -1e200]), 1e-5),
    "linear_two_level": (lambda: bp.linear_problem(True), np.array([1e200, 1e200]), 1e-5),
    "tensor_single_level": (lambda: bp.big_linear_problem(23, 45, 3), np.full(23, 1e200), 1e-5),
}


@pytest.mark.parametrize("name", sorted(NAN_DELTA))
def test_nan_delta_accepts(name):
    """Both log-posteriors -inf (or NaN): delta is NaN, a = 1, every u accepts (here u = 1 - 2^-53)."""
    make, start, step = NAN_DELTA[name]
    meta, arrays = make()
    nc, ns, J, d = 64, 3, int(meta["J"]), int(meta["dim"])
    th0 = np.tile(start, (nc, 1))
    z = step * np.abs(start) / np.diag(arrays["prop_L"]) * np.random.default_rng(5).standard_normal((nc, ns, J, d))
    u = 1.0 - 2.0 ** -53
    res = run_forced(meta, arrays, th0, z, dict(u_c=np.full((nc, ns, J), u), u_f=np.full((nc, ns), u)))
    assert res["out"]["accepted"].cpu().numpy().all(), name


def test_lv_start_at_minus_inf_proposal_finite_accepts_at_u_one():
    """theta = (6, 6) has lp = -inf; a proposal at a finite point has delta = +inf and accepts at u = 1.  In two
    levels the coarse step accepts (+inf), the remaining sub-steps propose the same point (skipped), and the fine
    screen's delta is NaN (-inf terms of the old state): accepted as well."""
    for two in (False, True):
        meta, arrays = bp.lv_problem(two)
        nc, J = 128, int(meta["J"])
        th0 = np.tile([6.0, 6.0], (nc, 1))
        target = bp.lv_initial_states(nc)
        z = np.zeros((nc, 1, J, 2))
        z[:, 0, 0] = (target - th0) / np.diag(arrays["prop_L"])
        res = run_forced(meta, arrays, th0, z, dict(u_c=np.ones((nc, 1, J)), u_f=np.ones((nc, 1))))
        assert res["out"]["accepted"].cpu().numpy().all(), two
        assert np.all(np.isfinite(res["state"]["logpost"].cpu().numpy()))


def test_below_the_bound_early_rejection_on_and_off_identical():
    """Uniforms 1e-12 from the long-double threshold (below what any bound certifies): no reference decision is
    asserted, but skipping must not change a single bit."""
    meta, arrays = bp.lv_problem(True)
    nc, ns = 512, 4
    th0 = bp.lv_initial_states(nc)
    for i, eta in enumerate((1e-13, 1e-12, 1e-10)):
        z = schedule_noise(meta, nc, ns, 300 + i)
        sch = R.forced_schedule(meta, arrays, th0, z, R.random_pattern(nc, ns, 3, seed=400 + i), eta, exact_eta=True)
        on = run_forced(meta, arrays, th0, z, sch, early_reject=True)
        off = run_forced(meta, arrays, th0, z, sch, early_reject=False)
        for part in ("out", "state"):
            for k in on[part]:
                assert torch.equal(on[part][k], off[part][k]), (eta, part, k)
        assert on["counters"] == off["counters"]
