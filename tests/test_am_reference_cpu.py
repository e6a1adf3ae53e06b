"""CPU: the reference of per-chain adaptive Metropolis (am_reference.py) against the C oracle, before the GPU tests rely
on it, and the configuration rules around it.

* On every forced case of the GPU file (support.AM_FORCED), the oracle replaying the uniforms of am_schedule takes
  exactly the scheduled decisions and reaches the same states; its am_mean, am_m2 and am_L equal the double track bit
  for bit and lie within the long-double bounds, which stay below BOUND_RATIO of the values' own scale.
* Negative controls: each plausible mistake of an AM update, applied to the reference run that plays the kernel on the
  schedule's uniforms, breaks a forced decision, a refresh count or a bound on at least one forced case.  A failed
  refresh that reinstalls the problem's factor is equivalent to the correct one on every decidable schedule (pinned).
* Every edge the schedules are meant to reach is reached.
* refresh = 0 replays through the oracle as refresh = 1, as the device runs it; yg_create refuses a negative or
  non-finite eps and a non-finite scale.
"""
import ctypes as C
import functools

import numpy as np
import pytest

import am_reference as A
import logpost_reference as R
from support import AM_FORCED, AM_SWEEP, am_forced_inputs, am_problem, am_start, schedule_noise

BOUND_RATIO = 1e-6      # every bound <= BOUND_RATIO x (|value| + the scale of its row and column)


@functools.lru_cache(maxsize=None)
def _schedule(name):
    meta, arrays, ad, th0, z, pattern, launches = am_forced_inputs(name)
    sch = A.am_schedule(meta, arrays, ad, th0, z, pattern, 0.0, launches=launches)
    return meta, arrays, ad, th0, z, launches, sch


def test_sweep_covers_every_instance():
    caps = {(A.cap(kw["d"]), A.cap(kw["dd"])) for kw, *_ in AM_SWEEP.values()}
    assert caps == {(D, DD) for D in (2, 4, 8) for DD in (2, 4, 8)}
    assert {A.cap(kw["d"]) for kw, *_ in AM_SWEEP.values() if kw["d"] < A.cap(kw["d"])} == {4, 8}   # padding d < D


def _ratio(bound, value, scale):
    return float(np.max(bound / (np.abs(np.asarray(value, dtype=np.float64)) + scale + 1e-300)))


@pytest.mark.parametrize("name", list(AM_FORCED))
def test_oracle_replay_reproduces_the_schedule(name):
    from oracle import cport
    meta, arrays, ad, th0, z, _, sch = _schedule(name)
    tr = sch["track"]
    ref = cport.run_injected(cport.Problem(meta, arrays, adaptive=ad), th0, z, sch["u_c"], sch["u_f"])
    assert np.array_equal(ref["accepted"], sch["accepted"]), name
    assert np.array_equal(ref["coarse_accepted"], sch["coarse_accepted"]), name
    assert np.array_equal(ref["traj"][:, 1:], sch["traj"]), name
    # the double track is the oracle's arithmetic, bit for bit
    for k in ("am_mean", "am_m2", "am_L"):
        assert np.array_equal(ref[k], sch[k]), (name, k)
    # the long-double track and its bounds
    tm, t2 = tr.welford_bounds()
    em = np.abs(ref["am_mean"] - tr.mu_ld).astype(np.float64)
    e2 = np.abs(ref["am_m2"] - tr.m2_ld).astype(np.float64)
    assert np.all(em <= tm) and np.all(e2 <= t2), (name, float(np.max(em - tm)), float(np.max(e2 - t2)))
    A.check_factor(tr, ref["am_L"], name)
    # the bounds are far below the values: mean against |mu| + sd, M2 against |M2| + max(M2_ii, M2_jj), the residual
    # against |C| + max(C_ii, C_jj) (the larger diagonal: a frozen coordinate's row of M2 is zero, its bound is not)
    R2 = np.asarray(tr.m2_ld, dtype=np.float64)
    dg = np.sqrt(np.maximum(np.einsum('cii->ci', R2), 0.0))
    n = max(tr.n_am - 1, 1)
    assert _ratio(tm, tr.mu_ld, dg / np.sqrt(n)) <= BOUND_RATIO, name
    assert _ratio(t2, R2, np.maximum(dg[:, :, None], dg[:, None, :]) ** 2) <= BOUND_RATIO, name
    res, b = tr.factor_residual(ref["am_L"])
    a = tr.adopted > 0
    if a.any():
        Cf = np.asarray(tr.C_ld[a], dtype=np.float64)
        cd = np.einsum('cii->ci', Cf)
        assert _ratio(b[a], Cf, np.maximum(cd[:, :, None], cd[:, None, :])) <= BOUND_RATIO, name
    assert sch["eta_min"] >= R.ETA_FACTOR * 8 * R.U, name


def _follow(name, mistakes=()):
    meta, arrays, ad, th0, z, launches, sch = _schedule(name)
    return A.am_schedule(meta, arrays, ad, th0, z, uniforms=dict(u_c=sch["u_c"], u_f=sch["u_f"]), launches=launches,
                         mistakes=mistakes)


def _detected(name, run):
    """Which of a forced decision, a refresh count or a bound the run breaks against the correct schedule."""
    sch = _schedule(name)[-1]
    tr = sch["track"]
    tm, t2 = tr.welford_bounds()
    try:
        A.check_factor(tr, run["am_L"])
        factor_ok = True
    except AssertionError:
        factor_ok = False
    return dict(
        decision=not np.array_equal(run["accepted"], sch["accepted"])
        or not np.array_equal(run["coarse_accepted"], sch["coarse_accepted"]),
        count=not np.array_equal(run["adopted"], sch["adopted"]) or not np.array_equal(run["kept"], sch["kept"]),
        bound=bool(np.any(np.abs(run["am_mean"] - tr.mu_ld).astype(np.float64) > tm)
                   or np.any(np.abs(run["am_m2"] - tr.m2_ld).astype(np.float64) > t2) or not factor_ok))


# the cheap cases first: a negative control stops at the first case that sees it
_BY_COST = sorted(AM_FORCED, key=lambda n: n.startswith("lv"))


def test_correct_run_breaks_nothing():
    for name in AM_FORCED:
        run = _follow(name)
        assert run["margin_min"] > 0, name
        assert not any(_detected(name, run).values()), name


@pytest.mark.parametrize("mistake", [m for m in A.MISTAKES if m != "failed_reinstalls_problem"])
def test_negative_control_is_seen_by_a_forced_case(mistake):
    seen = {}
    for name in _BY_COST:
        seen[name] = [k for k, v in _detected(name, _follow(name, (mistake,))).items() if v]
        if seen[name]:
            return
    pytest.fail(f"{mistake} is seen by no forced case: {seen}")


def test_failed_refresh_reinstalling_the_problem_factor_is_equivalent():
    """A refresh fails for certain only on a structural zero (eps = 0 and a coordinate whose fed values are all
    equal), and such a chain has never adopted a factor: one with a zero row would not be positive definite, and an
    adopted factor would have moved that coordinate.  So its factor still is the problem's, and reinstalling it
    changes nothing on any schedule whose refreshes are all decidable; this pins that it changes nothing here."""
    for name in AM_FORCED:
        sch = _schedule(name)[-1]
        run = _follow(name, ("failed_reinstalls_problem",))
        assert not any(_detected(name, run).values()), name
        assert np.array_equal(run["am_L"], sch["am_L"]), name
    assert any(_schedule(n)[-1]["kept"].any() for n in AM_FORCED)


def test_forced_cases_reach_every_edge():
    reach = dict(idle0=False, idle_past_first_launch=False, collection=set(), refresh=set(), default_scale=False,
                 given_scale=False, rejected_eps0=False, rejected_eps=False, frozen_eps0=False, frozen_eps=False,
                 offset=False, boundary=False, two_level=False, three_level=False, lv=False)
    for name in AM_FORCED:
        meta, arrays, ad, th0, z, launches, sch = _schedule(name)
        tr = sch["track"]
        idle = ad.get("idle", 0)
        reach["idle0"] |= idle == 0
        reach["idle_past_first_launch"] |= sch["first_update_launch"] > 0
        reach["collection"].add(min(ad["collection"], 3))
        reach["refresh"].add(ad["refresh"])
        reach["default_scale"] |= not ad.get("scale")
        reach["given_scale"] |= bool(ad.get("scale"))
        assert sch["first_refresh"] == max(ad["collection"], 2), name
        still = (np.stack(tr.fed, axis=1) == np.stack(tr.fed, axis=1)[:, :1]).all(axis=1)      # [nc, d]
        rejected, frozen = still.all(axis=1), still.any(axis=1) & ~still.all(axis=1)
        eps0 = ad["eps"] == 0.0
        if rejected.any():
            reach["rejected_eps0" if eps0 else "rejected_eps"] = True
            assert np.all(sch["kept"][rejected] > 0) if eps0 else np.all(sch["adopted"][rejected] > 0), name
        if np.any(np.all(np.asarray(arrays["prop_L"]) == 0.0, axis=1)):
            reach["frozen_eps0" if eps0 else "frozen_eps"] = True
            assert (frozen.any() or rejected.any()) if eps0 else np.all(sch["adopted"] > 0), name
        reach["offset"] |= float(np.abs(th0).min()) > 1e3
        reach["boundary"] |= sch["boundary_refreshes"] > 0
        reach["two_level"] |= meta["levels"] == 2 and meta["model"] == "linear"
        reach["three_level"] |= meta["levels"] == 3
        reach["lv"] |= meta["model"] == "lv"
    assert reach.pop("collection") == {0, 1, 2, 3} and reach.pop("refresh") >= {0, 1, 3}
    assert all(reach.values()), reach


def test_refresh_zero_replays_as_refresh_one():
    """The device maps refresh = 0 to 1 (abi.cu make_args); the oracle's problem does the same, where it used to
    divide by zero."""
    from oracle import cport
    meta, arrays = am_problem(3, dd=2, seed=61)
    nc, ns = 16, 12
    th0 = am_start(meta, arrays, nc, 62)
    z = schedule_noise(meta, nc, ns, 63)
    u_c, u_f = np.full((nc, ns, 1), 0.5), np.random.default_rng(64).random((nc, ns))
    out = [cport.run_injected(cport.Problem(meta, arrays, adaptive=dict(idle=0, collection=2, refresh=r, eps=1e-4)),
                              th0, z, u_c, u_f) for r in (0, 1)]
    for k in ("accepted", "traj", "am_mean", "am_m2", "am_L"):
        assert np.array_equal(out[0][k], out[1][k]), k
    assert not np.array_equal(out[1]["am_L"], np.broadcast_to(arrays["prop_L"], out[1]["am_L"].shape))


def test_create_refuses_bad_eps_and_scale_without_touching_the_gpu():
    """yg_create applies the builder's rule (AMBuilder.regularisationParameter: eps >= 0) and refuses a non-finite eps
    or scale: a NaN would make every refresh fail, and the chain would never adapt.  A scale <= 0 selects the default."""
    from yagre_mcmc_b200 import _lib
    lib = _lib.load()
    h = C.c_void_p()
    for eps, scale in ((-1e-8, 0.0), (float("nan"), 0.0), (float("inf"), 0.0), (1e-4, float("nan")),
                       (1e-4, float("inf")), (0.0, float("-inf"))):
        cfg = _lib.YgConfig()
        cfg.abi_version = _lib.YG_ABI_VERSION
        cfg.n_chains, cfg.dim, cfg.n_levels, cfg.model = 4, 3, 1, _lib.MODEL_GAUSS
        cfg.adaptive, cfg.am_collection_steps, cfg.am_refresh = 1, 10, 1
        cfg.am_eps, cfg.am_scale = eps, scale
        assert lib.yg_create(C.byref(cfg), C.byref(h)) == _lib.YG_ERR_INVALID, (eps, scale)
        assert b"eps" in lib.yg_last_error() and not h.value, (eps, scale)
