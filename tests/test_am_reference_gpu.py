"""GPU: per-chain adaptive Metropolis in generic_mh_kernel (every AM-carrying <D, DD, TWO_LEVEL> instance and the
warp-specialised one) and in the LV kernel, against the reference of am_reference.py.

* Values: a Philox run and a recorded run are bitwise equal (for d = 2 the Philox run is the warp-specialised instance,
  so WS equals plain).  Following the recorded noise, the reference decides every step by its long-double deltas (each
  decision beyond its bound), and matches the kernel's accept flags, trajectory and am_steps exactly; the final mean,
  M2 and factor equal the double track bit for bit and lie within the long-double bounds.
* Forced decisions (support.AM_FORCED) at three eta on injected noise, each run as launches of 1, 2, 5 and the rest.
* One transition per launch, with the AM state compared after every launch; splits, restarts and reloads; more chains
  than one grid sweep.
"""
import numpy as np
import pytest
import torch

import am_reference as A
import bench_problems as bp
from support import AM_FORCED, AM_SWEEP, _am_lv, am_forced_inputs, am_problem, am_start, ensemble, three_level_gauss

pytestmark = pytest.mark.gpu


def _inject(z, u_c, u_f):
    return dict(z=np.ascontiguousarray(np.transpose(z, (1, 2, 3, 0))),
                u_c=np.ascontiguousarray(np.transpose(u_c, (1, 2, 0))),
                u_f=np.ascontiguousarray(np.transpose(u_f, (1, 0))))


def _recorded(out):
    z = out["z"].cpu().numpy().transpose(3, 0, 1, 2)
    u_c = np.nan_to_num(out["u_c"].cpu().numpy().transpose(2, 0, 1), nan=0.5)
    u_f = np.nan_to_num(out["u_f"].cpu().numpy().transpose(1, 0), nan=0.5)
    return z, u_c, u_f


def _am_state(ens):
    st = ens.state()
    return dict(am_mean=st["am_mean"].cpu().numpy().T, am_m2=st["am_m2"].cpu().numpy().transpose(2, 0, 1),
                am_L=st["prop_L"].cpu().numpy().transpose(2, 0, 1), theta=st["theta"].cpu().numpy().T,
                am_steps=st["am_steps"])


def _check_am(got, track, label):
    """The kernel's AM state (chain-major) within the long-double bounds, and equal to the double track bit for bit."""
    if track.fed:
        tm, t2 = track.welford_bounds()
        assert np.all(np.abs(got["am_mean"] - track.mu_ld).astype(np.float64) <= tm), (label, "mean bound")
        assert np.all(np.abs(got["am_m2"] - track.m2_ld).astype(np.float64) <= t2), (label, "M2 bound")
    A.check_factor(track, got["am_L"], label)
    assert np.array_equal(got["am_mean"], track.mu), (label, "am_mean")
    assert np.array_equal(got["am_m2"], track.m2), (label, "am_m2")
    assert np.array_equal(got["am_L"], track.L), (label, "am_L")


def _value_case(name):
    if name == "gauss_three_level":
        meta, arrays = three_level_gauss()
        return meta, arrays, dict(idle=2, collection=3, refresh=1, eps=1e-5), \
            np.tile([0.5, 1.0], (64, 1)) + 0.01 * np.random.default_rng(1).standard_normal((64, 2)), 12
    if name.startswith("lv"):
        meta, arrays = _am_lv(2 if name == "lv_two_level" else 1)
        return meta, arrays, dict(idle=1, collection=2, refresh=1, eps=1e-6), bp.lv_initial_states(32), 10
    base, lv = name.rsplit("_L", 1)
    kw, ad, nc, ns = AM_SWEEP[base]
    meta, arrays = am_problem(levels=int(lv), **kw)
    return meta, arrays, ad, am_start(meta, arrays, nc, kw["seed"] + 100), ns


VALUE_CASES = [f"{n}_L{lv}" for n in AM_SWEEP for lv in (1, 2)] + ["gauss_three_level", "lv_one_level", "lv_two_level"]


@pytest.mark.parametrize("name", VALUE_CASES)
def test_values(name):
    meta, arrays, ad, th0, ns = _value_case(name)
    nc, d = th0.shape
    runs = []
    for record in (False, True):
        ens = ensemble(meta, arrays, nc, seed=17, adaptive=ad)
        ens.set_state(th0)
        out = ens.run(ns, samples=True, accepted=True, logpost=True, record=record)
        torch.cuda.synchronize()
        runs.append((out, {k: (v.cpu().numpy() if torch.is_tensor(v) else v) for k, v in ens.state().items()},
                     ens.last_launch(), _am_state(ens)))
        ens.close()
    (free, st_free, l_free, _), (rec, st, l_rec, am) = runs
    if meta["model"] != "lv":
        assert (l_free["block"] == 64) == (d <= 2) and l_rec["block"] != 64, (name, l_free, l_rec)
    for k in ("samples", "accepted", "logpost"):
        assert torch.equal(free[k], rec[k]), (name, k)
    for k, v in st.items():
        assert (np.array_equal(v, st_free[k]) if isinstance(v, np.ndarray) else v == st_free[k]), (name, k)
    z, u_c, u_f = _recorded(rec)
    ref = A.am_schedule(meta, arrays, ad, th0, z, uniforms=dict(u_c=u_c, u_f=u_f))
    assert ref["margin_min"] > 0, (name, "a decision within its bound")
    assert ref["track"].undecidable == 0, name
    assert np.array_equal(rec["accepted"].cpu().numpy().T, ref["accepted"]), name
    assert np.array_equal(rec["samples"].cpu().numpy().transpose(2, 0, 1), ref["traj"]), name
    assert am["am_steps"] == ns, name
    assert ref["adopted"].sum() > 0, name
    _check_am(am, ref["track"], name)


def _run_launches(ens, z, u_c, u_f, launches):
    acc, lo = [], 0
    for k in launches:
        out = ens.run(k, samples=True, accepted=True, inject=_inject(z[:, lo:lo + k], u_c[:, lo:lo + k], u_f[:, lo:lo + k]))
        acc.append(out["accepted"].cpu().numpy().T)
        lo += k
    torch.cuda.synchronize()
    return np.concatenate(acc, axis=1)


@pytest.mark.parametrize("eta", [0.0, 1e-7, 1e-3])
@pytest.mark.parametrize("name", list(AM_FORCED))
def test_forced_decisions(name, eta):
    meta, arrays, ad, th0, z, pattern, launches = am_forced_inputs(name)
    sch = A.am_schedule(meta, arrays, ad, th0, z, pattern, eta, launches=launches)
    nc, ns = sch["u_f"].shape
    ens = ensemble(meta, arrays, nc, seed=5, adaptive=ad)
    ens.set_state(th0)
    acc = _run_launches(ens, z, sch["u_c"], sch["u_f"], launches)
    label = f"{name} eta={eta}"
    assert np.array_equal(acc, sch["accepted"]), label
    am = _am_state(ens)
    assert np.array_equal(am["theta"], sch["theta"]) and am["am_steps"] == ns, label
    assert ens.counters()["coarse_accepted"] == int(sch["coarse_accepted"].sum()), label
    _check_am(am, sch["track"], label)
    ens.close()


def test_one_transition_per_launch():
    """The AM state after every launch of one transition equals the reference's after that transition: no transient
    error, and am_t0 carries the index across launches (idle, collection and refresh phases included)."""
    name = "d3_two_level_refresh3"
    meta, arrays, ad, th0, z, pattern, launches = am_forced_inputs(name)
    sch = A.am_schedule(meta, arrays, ad, th0, z, pattern, 0.0, launches=launches)
    nc, ns = sch["u_f"].shape
    ens = ensemble(meta, arrays, nc, seed=5, adaptive=ad)
    ens.set_state(th0)
    track, x = None, th0
    for n in range(ns):
        sl = slice(n, n + 1)
        ref = A.am_schedule(meta, arrays, ad, x, z[:, sl], uniforms=dict(u_c=sch["u_c"][:, sl], u_f=sch["u_f"][:, sl]),
                            track=track, t0=n)
        track, x = ref["track"], ref["theta"]
        acc = _run_launches(ens, z[:, sl], sch["u_c"][:, sl], sch["u_f"][:, sl], [1])
        assert np.array_equal(acc, sch["accepted"][:, sl]), n
        am = _am_state(ens)
        assert am["am_steps"] == n + 1 and np.array_equal(am["theta"], x), n
        _check_am(am, track, f"after launch {n}")
    assert track.adopted.sum() > 0 and len(track.refreshes) > 1
    ens.close()


def test_splits_restarts_and_reloads():
    """One Philox schedule: launches of 1, 2, 5 and the rest equal one launch bit for bit; set_state(keep_adaptation)
    continues the reference's schedule; set_state without it restarts from the problem's factor with am_steps = 0;
    state() -> load_state() resumes bit for bit."""
    kw, ad, nc, ns = AM_SWEEP["4x4"]
    meta, arrays = am_problem(levels=2, **kw)
    th0 = am_start(meta, arrays, nc, 71)
    outs = []
    for plan in ([ns], [1, 2, 5, ns - 8]):
        ens = ensemble(meta, arrays, nc, seed=72, adaptive=ad)
        ens.set_state(th0)
        parts = [ens.run(k, samples=True, accepted=True) for k in plan]
        torch.cuda.synchronize()
        outs.append(({k: torch.cat([p[k] for p in parts]) for k in ("samples", "accepted")},
                     {k: (v.cpu().numpy() if torch.is_tensor(v) else v) for k, v in ens.state().items()}))
        if len(plan) == 1:
            keep = ens
        else:
            ens.close()
    (a, sa), (b, sb) = outs
    for k in ("samples", "accepted"):
        assert torch.equal(a[k], b[k]), k
    for k, v in sa.items():
        assert (np.array_equal(v, sb[k]) if isinstance(v, np.ndarray) else v == sb[k]), k
    # reload into a fresh handle, then both run on
    mid = keep.state()
    other = ensemble(meta, arrays, nc, seed=72, adaptive=ad)
    other.load_state(mid)
    x1 = am_start(meta, arrays, nc, 73)
    results = []
    for e in (keep, other):
        e.set_state(x1, keep_diagnostics=True, keep_adaptation=True)
        results.append((e.run(8, samples=True, accepted=True, record=True), _am_state(e)))
    torch.cuda.synchronize()
    (r1, am1), (r2, am2) = results
    for k in ("samples", "accepted"):
        assert torch.equal(r1[k], r2[k]), k
    for k in ("am_mean", "am_m2", "am_L"):
        assert np.array_equal(am1[k], am2[k]), k
    assert am1["am_steps"] == ns + 8
    # the reference: the first schedule, then the restart from x1 with the same adaptation state
    z0, uc0, uf0 = _recorded(_rerun_recorded(meta, arrays, ad, th0, nc, ns))
    first = A.am_schedule(meta, arrays, ad, th0, z0, uniforms=dict(u_c=uc0, u_f=uf0))
    z1, uc1, uf1 = _recorded(r1)
    ref = A.am_schedule(meta, arrays, ad, x1, z1, uniforms=dict(u_c=uc1, u_f=uf1), track=first["track"], t0=ns)
    assert ref["margin_min"] > 0
    assert np.array_equal(r1["accepted"].cpu().numpy().T, ref["accepted"])
    _check_am(am1, ref["track"], "keep_adaptation")
    # set_state without the flag: the problem's factor, zero moments, am_steps 0
    keep.set_state(x1)
    am = _am_state(keep)
    assert am["am_steps"] == 0 and not am["am_mean"].any() and not am["am_m2"].any()
    assert np.array_equal(am["am_L"], np.broadcast_to(arrays["prop_L"], am["am_L"].shape))
    for e in (keep, other):
        e.close()


def _rerun_recorded(meta, arrays, ad, th0, nc, ns):
    ens = ensemble(meta, arrays, nc, seed=72, adaptive=ad)
    ens.set_state(th0)
    out = ens.run(ns, samples=True, accepted=True, record=True)
    torch.cuda.synchronize()
    ens.close()
    return out


def test_more_chains_than_one_grid_sweep():
    """310,001 chains: more than the generic launch's grid x block (148 SMs x 16 x 128 = 303,104 on a B200).  One
    handle equals two handles over the halves (chain_offset) bit for bit, and a row sample that includes chains of the
    second sweep follows the reference."""
    meta, arrays = am_problem(3, dd=2, seed=81)
    ad = dict(idle=0, collection=2, refresh=1, eps=1e-4)
    nc, ns, seed = 310_001, 6, 82
    th0 = am_start(meta, arrays, nc, 83)
    ens = ensemble(meta, arrays, nc, seed=seed, adaptive=ad)
    ens.set_state(th0)
    out = ens.run(ns, samples=True, accepted=True, record=True)
    torch.cuda.synchronize()
    launch = ens.last_launch()
    sweep = launch["grid"] * launch["block"]
    assert nc > sweep, launch
    st = {k: v.cpu().numpy() for k, v in ens.state().items() if torch.is_tensor(v)}
    h = 155_001
    parts = []
    for lo, hi in ((0, h), (h, nc)):
        e = ensemble(meta, arrays, hi - lo, seed=seed, chain_offset=lo, adaptive=ad)
        e.set_state(th0[lo:hi])
        parts.append((e.run(ns, samples=True, accepted=True), {k: v.cpu().numpy() for k, v in e.state().items()
                                                                if torch.is_tensor(v)}))
        e.close()
    for k in ("samples", "accepted"):
        assert torch.equal(torch.cat([p[0][k] for p in parts], dim=-1), out[k]), k
    for k in ("theta", "prop_L", "am_mean", "am_m2", "n_accept"):
        assert np.array_equal(np.concatenate([p[1][k] for p in parts], axis=-1), st[k]), k
    rows = np.sort(np.concatenate([np.random.default_rng(84).choice(sweep, 200, replace=False),
                                   sweep + np.random.default_rng(85).choice(nc - sweep, 200, replace=False)]))
    z, u_c, u_f = _recorded(out)
    ref = A.am_schedule(meta, arrays, ad, th0[rows], z[rows], uniforms=dict(u_c=u_c[rows], u_f=u_f[rows]))
    assert ref["margin_min"] > 0
    assert np.array_equal(out["accepted"].cpu().numpy().T[rows], ref["accepted"])
    got = dict(am_mean=st["am_mean"].T[rows], am_m2=st["am_m2"].transpose(2, 0, 1)[rows],
               am_L=st["prop_L"].transpose(2, 0, 1)[rows])
    _check_am(got, ref["track"], "second sweep")
    ens.close()
