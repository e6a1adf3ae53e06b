"""CPU: the long-double reference of the adaptive-error-model chain (aem_reference.py) against the C oracle, before the
GPU tests rely on it.

* On every shape of the GPU file (support.AEM_SWEEP, support.AEM_FORCED), the oracle replaying the uniforms of
  aem_forced_schedule takes exactly the scheduled decisions, reaches the same aem_n and coarse model-evaluation counts,
  and its error-model moments and log-posteriors lie within the reference's bounds; those bounds stay below
  1e-9 (1 + |value|).
* Negative controls: each plausible mistake of an AEM step, applied to the reference run that plays the kernel, breaks
  a forced decision, a count or a bound on at least one forced case of the GPU file.
"""
import functools

import numpy as np
import pytest

import aem_reference as A
import logpost_reference as R
from support import AEM_FORCED, AEM_SWEEP, aem_forced_inputs, aem_problem, aem_start, schedule_noise

BOUND_RTOL = 1e-9


def _sweep_inputs(name):
    kw, nc, ns, _ = AEM_SWEEP[name]
    meta, arrays = aem_problem(**kw)
    return meta, arrays, aem_start(arrays, nc, kw["seed"] + 100), schedule_noise(meta, nc, ns, kw["seed"] + 200), \
        R.random_pattern(nc, ns, meta["J"], kw["seed"] + 300)


@functools.lru_cache(maxsize=None)
def _schedule(kind, name):
    meta, arrays, th0, z, pattern = (_sweep_inputs if kind == "sweep" else aem_forced_inputs)(name)
    return meta, arrays, th0, z, A.aem_forced_schedule(meta, arrays, th0, z, pattern, 0.0)


def _within(got, ref, bound):
    e = np.abs(np.asarray(got, dtype=np.longdouble) - np.asarray(ref, dtype=np.longdouble)).astype(np.float64)
    return e <= bound


def _small(value, bound):
    return np.all(bound <= BOUND_RTOL * (1.0 + np.abs(np.asarray(value, dtype=np.float64))))


def test_sweep_covers_every_capacity_pair():
    pairs = {(A.cap(kw["d"]), A.cap(kw["dd"])) for kw, *_ in AEM_SWEEP.values()}
    assert pairs == {(D, DD) for D in (2, 4, 8) for DD in (2, 4, 8)}
    assert {A.cap(kw["d"]) for kw, *_ in AEM_FORCED.values()} == {2, 4, 8}


@pytest.mark.parametrize("kind,name", [("sweep", n) for n in AEM_SWEEP] + [("forced", n) for n in AEM_FORCED])
def test_oracle_replay_reproduces_the_schedule(kind, name):
    from oracle import cport
    meta, arrays, th0, z, sch = _schedule(kind, name)
    ref = cport.run_injected(cport.Problem(meta, arrays), th0, z, sch["u_c"], sch["u_f"])
    assert np.array_equal(ref["accepted"], sch["accepted"]), name
    assert np.array_equal(ref["coarse_accepted"], sch["coarse_accepted"]), name
    assert np.array_equal(ref["aem_n"], sch["aem_n"]), name
    assert np.array_equal(ref["aem_model_evals"], sch["aem_model_evals"]), name
    assert int(ref["n_evals"][1]) - th0.shape[0] == sch["fine_evals"], name
    assert np.array_equal(ref["traj"][:, 1:], sch["traj"]), name
    # error model
    assert np.all(_within(ref["aem_mean"], sch["aem_mean"], sch["aem_mean_bound"])), name
    n = sch["aem_n"][:, None]
    many = np.broadcast_to(n > 1, sch["aem_m2"].shape)
    var = sch["aem_m2"][many] / np.broadcast_to(n - 1, many.shape)[many]
    vb = sch["aem_m2_bound"][many] / np.broadcast_to(n - 1, many.shape)[many] + R.U * np.abs(var.astype(np.float64))
    assert np.all(_within(ref["aem_var"][many], var, vb)), name
    # log-posteriors: the oracle tracks the fine level; level 0 keeps the value chain_init computed
    assert np.all(_within(ref["logpost_L1"][:, 1:], sch["lp1"], sch["b1"])), name
    assert np.all(_within(ref["logpost_L1"][:, 0], sch["lp1_init"], sch["b1_init"])), name
    assert np.all(_within(ref["logpost_L0"][:, 0], sch["lp0_init"], sch["b0_init"])), name
    # the bounds are tight enough to mean something
    for v, b in (("lp0", "b0"), ("lp1", "b1"), ("cache_val", "cache_bound"), ("aem_mean", "aem_mean_bound"),
                 ("aem_m2", "aem_m2_bound")):
        assert _small(sch[v], sch[b]), (name, v, float(np.max(sch[b] / (1 + np.abs(np.asarray(sch[v], dtype=float))))))
    assert sch["eta_min"] >= R.ETA_FACTOR * 8 * R.U, name


def test_coarse_value_before_any_error_sample_is_the_plain_level_0_log_posterior():
    """With no error sample yet, the AEM coarse log-posterior is logpost_reference's level 0: same value, and the AEM
    bound is within a small factor of the plain one."""
    meta, arrays = aem_problem(d=3, dd=5, n_data=9, J=2, min_data=2, heuristic=True, seed=21)
    th = aem_start(arrays, 50, 22)
    ch = A._Chains(A._Problem(meta, arrays, ()), 50)
    lp, b = ch.coarse(np.arange(50), th)
    m0 = {k: v for k, v in meta.items() if k != "aem"}
    ref, rb = R.logpost_bound(m0, arrays, 0, th, path="generic")
    assert np.all(np.abs((lp - ref).astype(np.float64)) <= 1e-3 * rb)
    assert np.all(b <= 8.0 * rb) and np.all(b >= rb / 8.0)


def _detected(sch, run):
    """Which of a forced decision, a count or a bound the run breaks (a cache of another size is compared by its
    consequences only: decisions, evaluation counts and moments)."""
    same_cache = run["cache_keys"].shape == sch["cache_keys"].shape
    return dict(
        decision=not np.array_equal(run["accepted"], sch["accepted"])
        or not np.array_equal(run["coarse_accepted"], sch["coarse_accepted"]),
        count=run["coarse_evals"] != sch["coarse_evals"] or not np.array_equal(run["aem_n"], sch["aem_n"])
        or (same_cache and not np.array_equal(run["cache_n"], sch["cache_n"])),
        bound=bool(np.any(~_within(run["aem_mean"], sch["aem_mean"], sch["aem_mean_bound"]))
                   or np.any(~_within(run["aem_m2"], sch["aem_m2"], sch["aem_m2_bound"]))
                   or np.any(~_within(run["lp0"], sch["lp0"], sch["b0"]))
                   or (same_cache and np.any(~_within(run["cache_val"], sch["cache_val"], sch["cache_bound"])))))


def test_correct_run_breaks_nothing():
    for name in AEM_FORCED:
        meta, arrays, th0, z, sch = _schedule("forced", name)
        run = A.aem_run(meta, arrays, th0, z, sch["u_c"], sch["u_f"])
        assert not any(_detected(sch, run).values()), name


@pytest.mark.parametrize("mistake", [m for m in A.MISTAKES if m != "update_no_touch"])
def test_negative_control_is_seen_by_a_forced_case(mistake):
    seen = {}
    for name in AEM_FORCED:
        meta, arrays, th0, z, sch = _schedule("forced", name)
        run = A.aem_run(meta, arrays, th0, z, sch["u_c"], sch["u_f"], mistakes=(mistake,))
        seen[name] = [k for k, v in _detected(sch, run).items() if v]
    assert any(seen.values()), (mistake, seen)


def test_update_without_cache_touch_is_equivalent():
    """The error-model update's cache lookup (query_model_evaluation) always finds P as the newest entry, because
    the fine screen has just queried pi_c(P): moving it back is a no-op and no model evaluation is ever counted
    there.  So leaving the touch out is not a mistake any test can see; this pins that it changes nothing."""
    for name in AEM_FORCED:
        meta, arrays, th0, z, sch = _schedule("forced", name)
        run = A.aem_run(meta, arrays, th0, z, sch["u_c"], sch["u_f"], mistakes=("update_no_touch",))
        assert np.array_equal(run["cache_keys"], sch["cache_keys"]) and np.array_equal(run["cache_n"], sch["cache_n"])
        assert not any(_detected(sch, run).values()), name


def test_forced_cases_exercise_staleness_crossings_and_the_heuristic():
    clamped = unclamped = floored = 0
    for name in AEM_FORCED:
        meta, arrays, th0, z, sch = _schedule("forced", name)
        md = meta["aem"]["min_data"]
        path = sch["aem_n_path"]
        ns = path.shape[1] - 1
        for k in (md - 1, md, md + 1):          # reached strictly inside the run by some chain
            assert np.any(path[:, 1:ns] == k), (name, k)
        assert sch["stale_decisions"] > 0, name
        clamped, unclamped, floored = clamped + sch["clamped"], unclamped + sch["unclamped"], floored + sch["floored"]
    assert clamped > 0 and unclamped > 0 and floored > 0
