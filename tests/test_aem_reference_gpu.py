"""GPU: aem_mh_kernel (the adaptive-error-model step) against the long-double reference of aem_reference.py, at every
capacity class of the kernel.

* Values (support.AEM_SWEEP: all nine aem_mh_kernel<D, DD> instances): a Philox run and a recorded run are bitwise
  equal; following the recorded noise and the kernel's own accept flags, the reference then bounds every stored and
  final log-posterior, the error-model moments and the cache values, and matches aem_n, the cache keys, the counters
  and the states exactly; every decision whose margin exceeds its bound agrees.
* Forced decisions (support.AEM_FORCED, one per parameter capacity and more) at three distances from the thresholds.
* u = 0, a scalar chain under isclose equality, more chains than one grid sweep, and state round trips.
"""
import numpy as np
import pytest
import torch

import aem_reference as A
import logpost_reference as R
from support import (AEM_FORCED, AEM_SWEEP, aem_forced_inputs, aem_problem, aem_start, ensemble, replay,
                     schedule_noise)

pytestmark = pytest.mark.gpu


def _inject(z, u_c, u_f):
    """Chain-major noise to the device layouts of ChainEnsemble.run(inject=...)."""
    return dict(z=np.ascontiguousarray(np.transpose(z, (1, 2, 3, 0))),
                u_c=np.ascontiguousarray(np.transpose(u_c, (1, 2, 0))),
                u_f=np.ascontiguousarray(np.transpose(u_f, (1, 0))))


def _recorded(out):
    z = out["z"].cpu().numpy().transpose(3, 0, 1, 2)
    u_c = np.nan_to_num(out["u_c"].cpu().numpy().transpose(2, 0, 1), nan=0.5)
    u_f = np.nan_to_num(out["u_f"].cpu().numpy().transpose(1, 0), nan=0.5)
    return z, u_c, u_f


def _np(st):
    return {k: (v.cpu().numpy() if torch.is_tensor(v) else v) for k, v in st.items()}


def _within(got, ref, bound, label):
    e = np.abs(np.asarray(got, dtype=np.longdouble) - np.asarray(ref, dtype=np.longdouble)).astype(np.float64)
    ok = e <= bound
    assert np.all(ok), (label, float(np.max(e / np.maximum(bound, 1e-300))), np.argwhere(~ok)[:4])


def _check_state(meta, st, ref, label):
    """The kernel's final per-chain state against the reference: exact aem_n and cache keys / n, moments and cache
    values within bound."""
    d = int(meta["dim"])
    assert np.array_equal(st["aem_n"], ref["aem_n"]), label
    _within(st["aem_mean"].T, ref["aem_mean"], ref["aem_mean_bound"], (label, "aem_mean"))
    _within(st["aem_m2"].T, ref["aem_m2"], ref["aem_m2_bound"], (label, "aem_m2"))
    cache = st["aem_cache"]                                               # [3 (d + 1) + 1, nc]
    n = cache[3 * (d + 1)].astype(np.int64)
    assert np.array_equal(n, ref["cache_n"]), label
    for i in range(3):
        used = i < n
        keys = cache[i * (d + 1):i * (d + 1) + d].T
        assert np.array_equal(keys[used], ref["cache_keys"][used, i]), (label, "cache key", i)
        _within(cache[i * (d + 1) + d][used], ref["cache_val"][used, i], ref["cache_bound"][used, i],
                (label, "cache value", i))
    _within(st["logpost"][0], ref["lp0_final"], ref["b0_final"], (label, "final lp0"))
    _within(st["logpost"][1], ref["lp1_final"], ref["b1_final"], (label, "final lp1"))
    assert np.array_equal(st["theta"].T, ref["theta"]), label
    assert np.array_equal(st["n_accept"], ref["n_accept"]), label


def _check_counters(c, ref, label):
    got = {k: c[k] for k in ("transitions", "accepted", "coarse_evals", "fine_evals", "coarse_accepted")}
    want = dict(transitions=ref["accepted"].size, accepted=int(ref["accepted"].sum()), coarse_evals=ref["coarse_evals"],
                fine_evals=ref["fine_evals"], coarse_accepted=int(ref["coarse_accepted"].sum()))
    assert got == want, (label, got, want)


def _check_stored(out, ref, thin, label):
    samples = out["samples"].cpu().numpy().transpose(2, 0, 1)            # [nc, ns / thin, d]
    assert np.array_equal(samples, ref["traj"][:, thin - 1::thin]), label
    lp = out["logpost"].cpu().numpy()                                     # [ns / thin, 2, nc]
    _within(lp[:, 0].T, ref["lp0"][:, thin - 1::thin], ref["b0"][:, thin - 1::thin], (label, "stored lp0"))
    _within(lp[:, 1].T, ref["lp1"][:, thin - 1::thin], ref["b1"][:, thin - 1::thin], (label, "stored lp1"))


@pytest.mark.parametrize("name", list(AEM_SWEEP))
def test_values_at_every_capacity_class(name):
    kw, nc, ns, thin = AEM_SWEEP[name]
    meta, arrays = aem_problem(**kw)
    th0 = aem_start(arrays, nc, kw["seed"] + 100)
    label = f"{name} (aem_mh_kernel<{A.cap(kw['d'])}, {A.cap(kw['dd'])}>)"
    runs = []
    for record in (False, True):
        ens = ensemble(meta, arrays, nc, seed=kw["seed"] + 7, aem=meta["aem"])
        ens.set_state(th0)
        out = ens.run(ns, thin=thin, samples=True, accepted=True, logpost=True, record=record)
        torch.cuda.synchronize()
        launch = ens.last_launch()
        assert launch["block"] == 128 and launch["launches"] >= 1, (label, launch)
        runs.append((out, _np(ens.state()), ens.counters()))
        ens.close()
    (free, st_free, c_free), (rec, st, c) = runs
    for k in ("samples", "accepted", "logpost"):
        assert torch.equal(free[k], rec[k]), (label, k)
    for k, v in st.items():
        assert (np.array_equal(v, st_free[k]) if isinstance(v, np.ndarray) else v == st_free[k]), (label, k)
    assert c == c_free, label
    z, u_c, u_f = _recorded(rec)
    acc = rec["accepted"].cpu().numpy().T
    ref = A.aem_follow(meta, arrays, th0, z, u_c, u_f, acc)
    taken = np.isfinite(ref["margin_c"])
    assert np.all(ref["margin_c"][taken] > ref["bound_c"][taken]), (label, "a coarse decision within its bound")
    certain = np.isfinite(ref["margin_f"]) & (ref["margin_f"] > ref["bound_f"])
    own = A._accepts(ref["delta_f"][certain], u_f[certain])
    assert np.array_equal(own, acc[certain].astype(bool)), (label, "fine decisions")
    _check_stored(rec, ref, thin, label)
    _check_state(meta, st, ref, label)
    _check_counters(c, ref, label)


@pytest.mark.parametrize("eta", [0.0, 1e-7, 1e-3])
@pytest.mark.parametrize("name", list(AEM_FORCED))
def test_forced_decisions(name, eta):
    meta, arrays, th0, z, pattern = aem_forced_inputs(name)
    sch = A.aem_forced_schedule(meta, arrays, th0, z, pattern, eta)
    nc, ns = sch["u_f"].shape
    ens = ensemble(meta, arrays, nc, seed=5, aem=meta["aem"])
    ens.set_state(th0)
    out = ens.run(ns, samples=True, accepted=True, logpost=True, inject=_inject(z, sch["u_c"], sch["u_f"]))
    torch.cuda.synchronize()
    label = f"{name} eta={eta}"
    assert np.array_equal(out["accepted"].cpu().numpy().T, sch["accepted"]), label
    st = _np(ens.state())
    _check_stored(out, sch, 1, label)
    _check_state(meta, st, sch, label)
    _check_counters(ens.counters(), sch, label)
    # what the schedule exercised
    md = meta["aem"]["min_data"]
    for k in (md - 1, md, md + 1):
        assert np.any(sch["aem_n_path"][:, 1:ns] == k), (label, k)
    assert sch["stale_decisions"] > 0, label
    heur = {"d2_floor": ("floored", "unclamped"), "d4_clamp": ("clamped",), "d8_one_component": ("unclamped",)}
    for k in heur.get(name, ()):
        assert sch[k] > 0, (label, k)
    ens.close()


def test_zero_uniforms_accept_every_sub_step_and_screen():
    """u = 0 passes u <= min(exp(delta), 1) for every delta: every moved sub-step and every screen is accepted, and
    aem_n counts the moved fine steps."""
    meta, arrays = aem_problem(d=3, dd=5, n_data=9, J=3, min_data=2, heuristic=True, seed=31)
    nc, ns = 33, 30
    th0 = aem_start(arrays, nc, 32)
    z = schedule_noise(meta, nc, ns, 33)
    u_c, u_f = np.zeros((nc, ns, 3)), np.zeros((nc, ns))
    ens = ensemble(meta, arrays, nc, seed=1, aem=meta["aem"])
    ens.set_state(th0)
    out = ens.run(ns, samples=True, accepted=True, logpost=True, inject=_inject(z, u_c, u_f))
    torch.cuda.synchronize()
    acc = out["accepted"].cpu().numpy().T
    ref = A.aem_follow(meta, arrays, th0, z, u_c, u_f, acc)
    assert np.all(acc == 1)
    c, st = ens.counters(), _np(ens.state())
    assert c["coarse_accepted"] == nc * ns * 3 and c["accepted"] == nc * ns
    assert np.array_equal(st["aem_n"], np.full(nc, ns)) and np.array_equal(st["aem_n"], ref["aem_n"])
    _check_state(meta, st, ref, "u = 0")
    _check_counters(c, ref, "u = 0")


def _isclose_noise(meta, arrays, th0, ns, seed):
    """z for a scalar chain driven by u = 0 (every proposal that is not isclose-equal to its state is accepted, so
    the path is known in advance): per sub-step a normal draw, or a step of a few 1e-10 relative (isclose-equal: the
    sub-step is skipped), or at the last sub-step a return to within 5e-10 relative of the transition's start (the
    sub-chain moved, yet the screen sees an isclose-equal state and is skipped).  Returns z and the counts of both."""
    rng = np.random.default_rng(seed)
    nc, J = th0.shape[0], int(meta["J"])
    L = float(np.asarray(arrays["prop_L"])[0, 0])
    z = rng.standard_normal((nc, ns, J, 1))
    theta = th0.copy()
    tiny = back = 0
    for n in range(ns):
        s = theta.copy()
        kind = rng.random((nc, J))
        for j in range(J):
            t = kind[:, j] < 0.3
            z[t, n, j, 0] = rng.uniform(1.0, 6.0, t.sum()) * 1e-10 * s[t, 0] / L
            if j == J - 1:
                b = (kind[:, j] > 0.8) & (s[:, 0] != theta[:, 0])
                z[b, n, j, 0] = (theta[b, 0] * (1.0 + 5e-10) - s[b, 0]) / L
            p = R._propose(meta, arrays, s, z[:, n, j])
            eq = R._equal(meta, p, s)
            tiny += int(eq.sum())
            s = np.where(eq[:, None], s, p)
        same = R._equal(meta, s, theta)
        back += int((same & (s[:, 0] != theta[:, 0])).sum())
        theta = np.where(same[:, None], theta, s)
    return z, tiny, back


def test_scalar_isclose_equality():
    """d = 1 with eq='isclose' (parameter/scalar.py:38-43, math.isclose at rel_tol 1e-9): a proposal within 1e-9
    relative of the sub-chain state skips the sub-step, and a sub-chain ending within 1e-9 relative of the chain
    state skips the screen, in the kernel as in the oracle.  The cache lookup stays exact, as in the oracle; whether
    the reference library's memoisation compares ScalarParameter keys with isclose is not verified here."""
    from oracle import cport
    meta, arrays = aem_problem(d=1, dd=2, n_data=9, J=3, min_data=3, heuristic=True, seed=41, eq="isclose")
    nc, ns = 64, 40
    th0 = 1.0 + 0.1 * np.abs(aem_start(arrays, nc, 42))
    z, tiny, back = _isclose_noise(meta, arrays, th0, ns, 43)
    assert tiny > 100 and back > 20, (tiny, back)
    u_c, u_f = np.zeros((nc, ns, 3)), np.zeros((nc, ns))
    ens = ensemble(meta, arrays, nc, seed=1, aem=meta["aem"])
    ens.set_state(th0)
    out = ens.run(ns, samples=True, accepted=True, logpost=True, inject=_inject(z, u_c, u_f))
    torch.cuda.synchronize()
    acc = out["accepted"].cpu().numpy().T
    orc = cport.run_injected(cport.Problem(meta, arrays), th0, z, u_c, u_f)
    c, st = ens.counters(), _np(ens.state())
    assert np.array_equal(acc, orc["accepted"])
    assert np.array_equal(out["samples"].cpu().numpy().transpose(2, 0, 1), orc["traj"][:, 1:])
    assert np.array_equal(st["aem_n"], orc["aem_n"])
    assert c["coarse_evals"] == int(orc["aem_model_evals"].sum())
    assert c["coarse_accepted"] == int(orc["coarse_accepted"].sum())
    assert c["fine_evals"] == int(orc["n_evals"][1]) - nc
    ref = A.aem_follow(meta, arrays, th0, z, u_c, u_f, acc)
    _check_stored(out, ref, 1, "isclose")
    _check_state(meta, st, ref, "isclose")
    _check_counters(c, ref, "isclose")


def test_more_chains_than_one_grid_sweep():
    """310,001 chains: more than the launch's grid x block (148 SMs x 16 x 128 = 303,104 on a B200), so threads take a
    second chain.  One handle equals two handles over the halves (chain_offset) bit for bit, and a row sample that
    includes chains of the second sweep replays through the oracle."""
    meta, arrays = aem_problem(d=2, dd=2, n_data=2, J=2, min_data=2, heuristic=True, seed=51)
    nc, ns, seed = 310_001, 6, 52
    th0 = aem_start(arrays, nc, 53)
    ens = ensemble(meta, arrays, nc, seed=seed, aem=meta["aem"])
    ens.set_state(th0)
    out = ens.run(ns, samples=True, accepted=True, record=True)
    torch.cuda.synchronize()
    launch = ens.last_launch()
    assert nc > launch["grid"] * launch["block"], launch
    st = _np(ens.state())
    h = 155_001
    parts = []
    for lo, hi in ((0, h), (h, nc)):
        e = ensemble(meta, arrays, hi - lo, seed=seed, chain_offset=lo, aem=meta["aem"])
        e.set_state(th0[lo:hi])
        parts.append((e.run(ns, samples=True, accepted=True), _np(e.state())))
        e.close()
    for k in ("samples", "accepted"):
        assert torch.equal(torch.cat([p[0][k] for p in parts], dim=-1), out[k]), k
    for k in ("theta", "logpost", "aem_n", "aem_mean", "aem_m2", "aem_cache", "n_accept"):
        assert np.array_equal(np.concatenate([p[1][k] for p in parts], axis=-1), st[k]), k
    sweep = launch["grid"] * launch["block"]
    rows = np.sort(np.concatenate([np.random.default_rng(54).choice(sweep, 200, replace=False),
                                   sweep + np.random.default_rng(55).choice(nc - sweep, 200, replace=False)]))
    assert np.any(rows >= sweep)
    ref = replay(meta, arrays, th0, out, rows=rows)
    assert np.array_equal(out["accepted"].cpu().numpy().T[rows], ref["accepted"])
    assert np.array_equal(out["samples"].cpu().numpy().transpose(2, 0, 1)[rows], ref["traj"][:, 1:])
    assert np.array_equal(st["aem_n"][rows], ref["aem_n"])
    ens.close()


def test_state_round_trips():
    """d = 5, data_dim = 3: the cache stride d + 1 = 6 is not the capacity 8.  load_state resumes bitwise;
    set_state(keep_adaptation) continues bitwise; set_state without it clears aem_n, the moments and the cache, and
    the next run equals a fresh handle's from the same state at the same Philox step."""
    meta, arrays = aem_problem(d=5, dd=3, n_data=9, J=2, min_data=3, heuristic=True, error_scale=0.1, prop_scale=0.5,
                               seed=61)
    nc, k, seed = 257, 20, 62
    th0 = aem_start(arrays, nc, 63)
    a = ensemble(meta, arrays, nc, seed=seed, aem=meta["aem"])
    a.set_state(th0)
    a.run(k, samples=False)
    mid = a.state()
    assert int(mid["aem_n"].max()) > meta["aem"]["min_data"]          # the mean shift and the inflation are on
    second = a.run(k, samples=True, accepted=True, logpost=True)
    end = _np(a.state())
    # load_state into a fresh handle
    b = ensemble(meta, arrays, nc, seed=seed, aem=meta["aem"])
    b.load_state(mid)
    out = b.run(k, samples=True, accepted=True, logpost=True)
    for key in ("samples", "accepted", "logpost"):
        assert torch.equal(out[key], second[key]), key
    for key, v in _np(b.state()).items():
        assert (np.array_equal(v, end[key]) if isinstance(v, np.ndarray) else v == end[key]), key
    # set_state(keep_adaptation): same error model and cache, same stream position
    c = ensemble(meta, arrays, nc, seed=seed, aem=meta["aem"])
    c.load_state(mid)
    c.set_state(mid["theta"].t(), keep_diagnostics=True, keep_adaptation=True)
    st_c = _np(c.state())
    for key in ("aem_n", "aem_mean", "aem_m2", "aem_cache"):
        assert np.array_equal(st_c[key], _np(mid)[key]), key
    out = c.run(k, samples=True, accepted=True)
    for key in ("samples", "accepted"):
        assert torch.equal(out[key], second[key]), key
    for key in ("theta", "aem_n", "aem_mean", "aem_m2", "aem_cache", "w_mean", "w_m2"):
        assert np.array_equal(_np(c.state())[key], end[key]), key
    # set_state without it: a fresh error model and an empty cache, then a fresh handle's run at that step
    c.load_state(mid)
    c.set_state(mid["theta"].t())
    st_c = _np(c.state())
    assert not st_c["aem_n"].any() and not st_c["aem_mean"].any() and not st_c["aem_m2"].any()
    assert not st_c["aem_cache"][-1].any()
    out = c.run(k, samples=True, accepted=True, logpost=True)
    f = ensemble(meta, arrays, nc, seed=seed, aem=meta["aem"])
    f.set_state(mid["theta"].t(), step_index=mid["step_index"])
    want = f.run(k, samples=True, accepted=True, logpost=True)
    for key in ("samples", "accepted", "logpost"):
        assert torch.equal(out[key], want[key]), key
    st_f = _np(f.state())
    for key, v in _np(c.state()).items():
        if key not in ("welford_n", "w_mean", "w_m2"):
            assert (np.array_equal(v, st_f[key]) if isinstance(v, np.ndarray) else v == st_f[key]), key
    for e in (a, b, c, f):
        e.close()


def test_tempered_level_0_is_refused():
    """The error model's coarse log-posterior has no tempering factor, so a tempered level 0 would run untempered:
    yg_set_problem refuses it.  A tempering of exactly 1 is the untempered model and is accepted."""
    meta, arrays = aem_problem(d=2, dd=2, n_data=2, J=2, min_data=2, heuristic=True, seed=71)
    with pytest.raises(NotImplementedError, match="tempered level 0"):
        ensemble(meta, dict(arrays, L0_tempering=np.array(0.5)), 8, aem=meta["aem"])
    ensemble(meta, dict(arrays, L0_tempering=np.array(1.0)), 8, aem=meta["aem"]).close()
    ensemble({k: v for k, v in meta.items() if k != "aem"}, dict(arrays, L0_tempering=np.array(0.5)), 8).close()
