"""GPU: the C-ABI backend beyond the fixture trajectories -- device-generated (Philox) noise
replayed through the C oracle, sharding / resume / thinning invariances, the diagnostics
kernels against the reference's post-processing fixtures, adaptive Metropolis, and
size-independent properties at BASELINE.json's full ensemble sizes."""
import numpy as np
import pytest
import torch

import bench_problems as bp
from diag_reference import check_replay_diagnostics, pre_states
from golden_io import load, rel_err

pytestmark = pytest.mark.gpu

LOGPOST_RTOL = 1e-10      # north_star: 1e-10 relative on log-posterior


def _ens(meta, arrays, nc, **kw):
    from yagre_mcmc_b200.ensemble import ChainEnsemble, LoweredProblem
    return ChainEnsemble(LoweredProblem(meta, arrays), nc, **kw)


def _replay(meta, arrays, th0, out, adaptive=None):
    """Runs the oracle on the noise the device recorded (chain-major layout)."""
    from oracle import cport
    z = out["z"].cpu().numpy().transpose(3, 0, 1, 2)
    u_c = np.nan_to_num(out["u_c"].cpu().numpy().transpose(2, 0, 1), nan=0.5)
    u_f = np.nan_to_num(out["u_f"].cpu().numpy().transpose(1, 0), nan=0.5)
    return cport.run_injected(cport.Problem(meta, arrays, adaptive=adaptive), th0, z, u_c, u_f)     # meta['aem'] is honoured


CASES = {
    "lv_two_level": lambda: (bp.lv_problem(True), lambda n: bp.lv_initial_states(n), 300, 30),
    "lv_single_level": lambda: (bp.lv_problem(False), lambda n: bp.lv_initial_states(n), 300, 30),
    "lv_two_level_ragged": lambda: (bp.lv_problem(True, Nc=37, Nf=203, J=2, n_data=7), lambda n: bp.lv_initial_states(n), 211, 17),
    "linear_two_level": lambda: (bp.linear_problem(True), lambda n: np.zeros((n, 2)), 1000, 200),
    "linear_single_level": lambda: (bp.linear_problem(False), lambda n: np.zeros((n, 2)), 1000, 200),
    "gauss2d": lambda: (bp.gauss2d_problem(), lambda n: np.tile([-8.0, -7.0], (n, 1)), 1000, 300),
    "lv_pcn": lambda: (bp.lv_pcn_problem(), lambda n: bp.lv_initial_states(n), 300, 30),
    # large linear model on the FP64 tensor path (DMMA): full size, ragged sizes, two level
    "big_linear_64x256": lambda: (bp.big_linear_problem(64, 256, 1), lambda n: np.zeros((n, 64)), 200, 25),
    "big_linear_ragged": lambda: (bp.big_linear_problem(23, 45, 3), lambda n: np.zeros((n, 23)), 77, 25),
    "big_linear_two_level": lambda: (bp.big_linear_problem(32, 96, 2, two_level=True, J=3), lambda n: np.zeros((n, 32)), 150, 20),
}


@pytest.mark.parametrize("name", sorted(CASES))
def test_philox_run_replayed_through_oracle(name):
    """Device draws the noise (Philox + Box-Muller), records it; the oracle replays the same noise:
    identical decisions and trajectories, log-posterior within tolerance."""
    (meta, arrays), init, nc, ns = CASES[name]()
    th0 = init(nc)
    ens = _ens(meta, arrays, nc, seed=99)
    ens.set_state(th0)
    lp_init = ens.state()["logpost"].cpu().numpy()
    out = ens.run(ns, samples=True, accepted=True, logpost=True, record=True)
    torch.cuda.synchronize()
    ref = _replay(meta, arrays, th0, out)
    acc = out["accepted"].cpu().numpy().T
    assert int((acc != ref["accepted"]).sum()) == 0
    traj = out["samples"].cpu().numpy().transpose(2, 0, 1)
    assert rel_err(traj, ref["traj"][:, 1:]).max() <= 1e-12
    lp = out["logpost"].cpu().numpy().transpose(2, 0, 1)
    assert rel_err(lp_init[0], ref["logpost_L0"][:, 0]).max() <= LOGPOST_RTOL
    assert rel_err(lp[:, :, 0], ref["logpost_L0"][:, 1:]).max() <= LOGPOST_RTOL
    if meta["levels"] == 2:
        assert rel_err(lp[:, :, 1], ref["logpost_L1"][:, 1:]).max() <= LOGPOST_RTOL
    c = ens.counters()
    assert c["transitions"] == nc * ns and c["accepted"] == int(acc.sum())
    ev = ref["n_evals"]
    if meta["levels"] == 2:
        # nc evaluations per level belong to the initial state in the oracle's count
        assert (c["coarse_evals"], c["fine_evals"]) == (int(ev[0]) - nc, int(ev[1]) - nc)
    check_replay_diagnostics(ens.state(), c, ref, pre_states(th0, [out["samples"].cpu().numpy()]), name)
    z = out["z"].cpu().numpy()
    assert abs(z.mean()) < 0.02 and abs(z.var() - 1.0) < 0.03          # the recorded draws are N(0,1)


def test_device_philox_matches_host_philox_bitwise():
    """Uniforms are pure integer arithmetic + one exact scaling: the device stream must equal the
    oracle's Philox restatement bit for bit, keyed by (seed, global chain id, step, sub-step)."""
    from oracle import cport
    meta, arrays = bp.linear_problem(True)
    nc, ns, off = 64, 8, 1000
    ens = _ens(meta, arrays, nc, seed=4242, chain_offset=off)
    ens.set_state(np.zeros((nc, 2)))
    out = ens.run(ns, record=True, samples=False)
    u_c = out["u_c"].cpu().numpy()      # [ns, J, nc]
    u_f = out["u_f"].cpu().numpy()      # [ns, nc]
    z = out["z"].cpu().numpy()          # [ns, J, d, nc]
    checked = 0
    for n in range(ns):
        for c in range(0, nc, 7):
            for j in range(meta["J"]):
                if not np.isnan(u_c[n, j, c]):
                    assert u_c[n, j, c] == cport.philox_uniform(4242, off + c, n, j)
                    checked += 1
                zz = cport.philox_normals(4242, off + c, n, j, 2)
                np.testing.assert_allclose(z[n, j, :, c], zz, rtol=1e-13, atol=1e-15)   # libm vs libdevice log/sincos
            if not np.isnan(u_f[n, c]):
                assert u_f[n, c] == cport.philox_uniform(4242, off + c, n, 0xFFFF)
    assert checked > 50


@pytest.mark.parametrize("two_level", [True, False])
def test_sharding_invariance(two_level):
    """One handle over n chains == two handles over the halves with chain_offset (what two GPUs do):
    bitwise equal samples, whatever the launch geometry."""
    meta, arrays = bp.lv_problem(two_level, Nc=32, Nf=96)
    nc, ns = 512, 12
    th0 = bp.lv_initial_states(nc)
    full = _ens(meta, arrays, nc, seed=5)
    full.set_state(th0)
    a = full.run(ns, samples=True)["samples"].cpu().numpy()
    parts = []
    for (lo, hi, geo) in [(0, 200, dict(blocks_per_sm=2, threads_per_block=256)), (200, nc, dict(rk4_segment=16))]:
        e = _ens(meta, arrays, hi - lo, seed=5, chain_offset=lo, **geo)
        e.set_state(th0[lo:hi])
        parts.append(e.run(ns, samples=True)["samples"].cpu().numpy())
    assert np.array_equal(a, np.concatenate(parts, axis=2))


@pytest.mark.parametrize("case", ["lv", "linear", "gauss_am"])
def test_resume_is_bit_exact(case):
    """get_state / load_state (the reference's restart-from-trajectory[-1] idiom, made exact):
    20 transitions == 8 + save + load into a fresh handle + 12."""
    adaptive = None
    if case == "lv":
        (meta, arrays), th0 = bp.lv_problem(True, Nc=16, Nf=64), bp.lv_initial_states(300)
    elif case == "linear":
        (meta, arrays), th0 = bp.linear_problem(True), np.zeros((300, 2))
    else:
        (meta, arrays), th0 = bp.gauss2d_problem(), np.tile([-8.0, -7.0], (300, 1))
        adaptive = dict(idle=2, collection=5, eps=1e-4)
    nc = th0.shape[0]
    a = _ens(meta, arrays, nc, seed=8, adaptive=adaptive)
    a.set_state(th0)
    ref = a.run(20, samples=True)["samples"].cpu().numpy()
    ref_state = a.state()
    b = _ens(meta, arrays, nc, seed=8, adaptive=adaptive)
    b.set_state(th0)
    first = b.run(8, samples=True)["samples"].cpu().numpy()
    saved = b.state()
    c = _ens(meta, arrays, nc, seed=8, adaptive=adaptive)
    c.load_state(saved)
    second = c.run(12, samples=True)["samples"].cpu().numpy()
    assert np.array_equal(ref, np.concatenate([first, second], axis=0))
    end = c.state()
    for k in ("theta", "logpost", "n_accept", "w_mean", "w_m2"):
        assert torch.equal(end[k], ref_state[k]), k
    assert end["step_index"] == 20 and end["welford_n"] == ref_state["welford_n"]


def test_checkpoint_files_and_trajectory_dump(tmp_path):
    """io.py: a run resumed from a checkpoint FILE continues bit-exactly; the trajectory dump round-trips."""
    from yagre_mcmc_b200 import io
    meta, arrays = bp.lv_problem(True, Nc=16, Nf=64)
    nc = 200
    th0 = bp.lv_initial_states(nc)
    a = _ens(meta, arrays, nc, seed=3, chain_offset=1000)
    a.set_state(th0)
    ref = a.run(30, samples=True)["samples"]
    b = _ens(meta, arrays, nc, seed=3, chain_offset=1000)
    b.set_state(th0)
    first = b.run(10, samples=True)["samples"]
    ck = io.save_checkpoint(str(tmp_path / "ck"), b, extra=dict(note="after 10"))
    c = _ens(meta, arrays, nc, seed=3, chain_offset=1000)
    head = io.load_checkpoint(ck, c)
    assert head["step_index"] == 10 and head["extra"]["note"] == "after 10"
    second = c.run(20, samples=True)["samples"]
    assert torch.equal(torch.cat([first, second]), ref)
    wrong = _ens(meta, arrays, nc, seed=4, chain_offset=1000)
    with pytest.raises(ValueError, match="seed"):
        io.load_checkpoint(ck, wrong)
    f = io.save_trajectory(str(tmp_path / "traj"), ref, thin=1, chain_offset=1000, meta=dict(model="lv"))
    back, side = io.load_trajectory(f)
    assert np.array_equal(back, ref.cpu().numpy()) and side["n_chains"] == nc and side["chain_offset"] == 1000
    assert io.as_reference_layout(back).shape == (30, nc, 2)
    mm, _ = io.load_trajectory(f, mmap=True)
    assert np.array_equal(mm[-1], back[-1])


def test_load_state_rejects_misshapen_arrays():
    """load_state checks every array against the ensemble's layout before yg_load_state copies from it (each array
    here is at least as large as that copy, so nothing reads out of bounds whatever the check does)."""
    meta, arrays = bp.linear_problem(True)
    nc = 64
    a = _ens(meta, arrays, nc, seed=8)
    a.set_state(np.zeros((nc, 2)))
    a.run(5, samples=False)
    st = a.state()
    b = _ens(meta, arrays, nc, seed=8)
    for theta in (st["theta"].t().contiguous(), torch.zeros(3, nc, dtype=torch.float64, device=st["theta"].device)):
        with pytest.raises(ValueError, match="theta"):
            b.load_state(dict(st, theta=theta))
    with pytest.raises(ValueError, match="logpost"):
        b.load_state({k: v for k, v in st.items() if k != "logpost"})
    b.load_state(st)
    assert torch.equal(b.state()["theta"], st["theta"])


def test_failed_set_problem_leaves_the_handle_unchanged():
    """A tensor-path handle (data_dim 16) given a one-chain-per-thread problem that fails validation keeps its problem:
    the same log-posteriors, and it still runs."""
    import ctypes as C
    from yagre_mcmc_b200 import _lib
    from yagre_mcmc_b200.ensemble import LoweredProblem
    meta, arrays = bp.big_linear_problem(2, 16, 1)
    nc = 64
    ens = _ens(meta, arrays, nc, seed=12)
    pts = np.random.default_rng(0).standard_normal((8, 2))
    before = ens.logpost(0, pts)
    small_meta, small_arrays = bp.linear_problem(False)
    small = LoweredProblem(dict(small_meta, proposal="pcn", pcn_step=0.7), small_arrays)
    pb = small.c_struct()
    assert ens.lib.yg_set_problem(ens._h, C.byref(pb)) == _lib.YG_ERR_INVALID
    assert torch.equal(ens.logpost(0, pts), before)
    ens.set_state(np.zeros((nc, 2)))
    ens.run(10, samples=False)
    assert ens.counters()["transitions"] == nc * 10


def test_thinning_and_outputs():
    meta, arrays = bp.lv_problem(True, Nc=16, Nf=64)
    nc = 200
    th0 = bp.lv_initial_states(nc)
    a = _ens(meta, arrays, nc, seed=3)
    a.set_state(th0)
    full = a.run(20, samples=True, logpost=True)
    b = _ens(meta, arrays, nc, seed=3)
    b.set_state(th0)
    thin = b.run(20, thin=5, samples=True, logpost=True)
    assert torch.equal(full["samples"][4::5], thin["samples"])
    assert torch.equal(full["logpost"][4::5], thin["logpost"])
    assert tuple(thin["samples"].shape) == (4, 2, nc)
    with pytest.raises(ValueError):
        b.run(7, thin=5, samples=True)


def test_error_paths_follow_reference_exception_types():
    from yagre_mcmc_b200.ensemble import ChainEnsemble, LoweredProblem
    meta, arrays = bp.linear_problem(True)
    e = ChainEnsemble(LoweredProblem(meta, arrays), 16)
    with pytest.raises(RuntimeError):                      # run before set_state
        e.run(3)
    with pytest.raises(ValueError):
        e.set_state(np.zeros((5, 2)))
    with pytest.raises(NotImplementedError):
        LoweredProblem(dict(meta, model="pde"), arrays)
    bad = dict(arrays)
    bad["prop_L"] = np.eye(9)
    with pytest.raises((ValueError, NotImplementedError)):
        ChainEnsemble(LoweredProblem(dict(meta, dim=9), bad), 16)


def test_pcn_posterior_moments_match_mrw():
    """pCN (likelihood-ratio acceptance, prior-preserving proposal) and MRW (posterior-ratio acceptance)
    target the same posterior: 8,192 chains each on the C4 problem must agree in mean and covariance."""
    nc = 8192
    out = []
    for meta, arrays in (bp.lv_pcn_problem(), bp.lv_problem(False)):
        ens = _ens(meta, arrays, nc, seed=31)
        ens.set_state(bp.lv_initial_states(nc))
        ens.run(300, samples=False)
        th = ens.state()["theta"].cpu().numpy()
        out.append((th.mean(1), np.cov(th)))
        c = ens.counters()
        assert 0.05 < c["accepted"] / c["transitions"] < 0.8
    se = np.sqrt(np.diag(out[1][1]) / nc)
    assert np.all(np.abs(out[0][0] - out[1][0]) < 6 * se)
    np.testing.assert_allclose(out[0][1], out[1][1], rtol=0.1, atol=2e-5)


def test_big_linear_posterior_moments_and_diagnostics():
    """d = 64, dataDim = 256 on the DMMA kernel: the posterior is Gaussian in closed form."""
    nc, d = 4096, 64
    meta, arrays = bp.big_linear_problem(d, 256, 1)
    mean, cov = bp.linear_gaussian_posterior(arrays, 0)
    ens = _ens(meta, arrays, nc, seed=41)
    ens.set_state(np.tile(mean, (nc, 1)))
    ens.run(1500, samples=False)
    out = ens.run(40, thin=40, samples=True, accepted=True)
    th = out["samples"][-1].cpu().numpy()                       # [d, nc]
    se = np.sqrt(np.diag(cov) / nc)
    assert np.all(np.abs(th.mean(1) - mean) < 5 * se)
    np.testing.assert_allclose(th.var(1, ddof=1), np.diag(cov), rtol=0.15)
    c = ens.counters()
    assert 0.1 < c["accepted"] / c["transitions"] < 0.5 and c["transitions"] == nc * 1540
    st = ens.state()
    assert tuple(st["w_m2"].shape) == (d, nc) and tuple(st["w_mean"].shape) == (d, nc)
    assert torch.equal(st["theta"], out["samples"][-1])
    assert st["welford_n"] == 1540 and torch.isfinite(st["w_m2"]).all()
    with pytest.raises(NotImplementedError):
        ens.pooled_stats()
    # sizes beyond the kernel, or features it does not have, are refused loudly
    with pytest.raises(NotImplementedError):
        _ens(*bp.big_linear_problem(65, 64, 1), 16)
    dense = dict(arrays)                            # round 2: a dense proposal factor runs (4 warps per SM at this size)
    dense["prop_L"] = 0.02 * np.linalg.cholesky(np.eye(d) + 0.01)
    e2 = _ens(meta, dense, 64, seed=1)
    e2.set_state(np.tile(mean, (64, 1)))
    e2.run(20, samples=False)
    assert e2.counters()["transitions"] == 64 * 20 and e2.last_launch()["block"] == 4 * 32
    with pytest.raises(NotImplementedError):        # per-chain adaptation would need a d x d factor per chain
        _ens(meta, arrays, 16, adaptive=dict(idle=1, collection=2))


def test_logpost_matches_oracle():
    from oracle import cport
    rng = np.random.default_rng(0)
    for (meta, arrays), pts in [(bp.lv_problem(True), bp.LV_TRUTH + 0.3 * rng.standard_normal((64, 2))),
                                (bp.linear_problem(True), rng.standard_normal((64, 2)) * 2),
                                (bp.big_linear_problem(32, 96, 2, two_level=True), rng.standard_normal((64, 32))),
                                (bp.gauss2d_problem(), rng.standard_normal((64, 2)) * 3)]:
        ens = _ens(meta, arrays, 4)
        pb = cport.Problem(meta, arrays)
        for lvl in range(meta["levels"]):
            got = ens.logpost(lvl, pts).cpu().numpy()
            want = np.array([cport.logpost(pb, lvl, p) for p in pts])
            assert rel_err(got, want).max() <= LOGPOST_RTOL


def test_nonfinite_forward_output_is_rejected():
    """RK4 blows up for extreme parameters: forward output -> +inf, logL -> -inf, proposal rejected
    by the unchanged acceptance rule (policy of the oracle's solver plugin)."""
    meta, arrays = bp.lv_problem(True, Nc=8, Nf=16)
    ens = _ens(meta, arrays, 32)
    lp = ens.logpost(0, np.tile([6.0, 6.0], (32, 1))).cpu().numpy()
    assert np.all(np.isneginf(lp))


# ------------------------------------------------------------------------------------------
# adaptive error model (chain/method/aem.py)
# ------------------------------------------------------------------------------------------

def _aem_run(meta, a, **kw):
    nc, ns = a["u_f"].shape
    ens = _ens(meta, a, nc, aem=meta["aem"], **kw)
    ens.set_state(a["theta0"])
    inj = dict(z=np.ascontiguousarray(np.transpose(a["z"], (1, 2, 3, 0))),
               u_c=np.ascontiguousarray(np.transpose(a["u_c"], (1, 2, 0))),
               u_f=np.ascontiguousarray(np.transpose(a["u_f"], (1, 0))))
    out = ens.run(ns, samples=True, accepted=True, inject=inj)
    return ens, out


@pytest.mark.parametrize("name", ["aem_linear", "aem_linear_noheuristic"])
def test_adaptive_error_model_matches_reference_fixture(name):
    """Same noise as the unmodified reference's AEM run: identical decisions and trajectory, the same
    error-model state, and the same number of coarse model evaluations (= the LRU(3) cache of the
    coarse likelihood, stale entries included, behaves like the reference's)."""
    meta, a = load(name)
    ens, out = _aem_run(meta, a)
    acc = out["accepted"].cpu().numpy().T
    assert int((acc != a["accepted"]).sum()) == 0
    traj = out["samples"].cpu().numpy().transpose(2, 0, 1)
    assert rel_err(traj, a["traj"][:, 1:]).max() <= 1e-12
    st = ens.state()
    n = st["aem_n"].cpu().numpy()
    assert np.array_equal(n, a["aem_n"])
    np.testing.assert_allclose(st["aem_mean"].cpu().numpy().T, a["aem_mean"], rtol=1e-10, atol=1e-14)
    np.testing.assert_allclose(st["aem_m2"].cpu().numpy().T / (n[:, None] - 1), a["aem_var"], rtol=1e-10, atol=1e-14)
    c = ens.counters()
    assert c["coarse_evals"] == int(a["n_model_evals"][:, 0].sum())
    assert c["accepted"] == int(a["accepted"].sum())


def test_adaptive_error_model_philox_replay_and_resume():
    from oracle import cport
    meta, arrays = bp.linear_problem(True)
    meta = dict(meta, aem=dict(min_data=8, heuristic=True))
    nc, ns = 500, 300
    th0 = np.zeros((nc, 2))
    ens = _ens(meta, arrays, nc, seed=77, aem=meta["aem"])
    ens.set_state(th0)
    out = ens.run(ns, samples=True, accepted=True, record=True)
    ref = _replay(meta, arrays, th0, out)
    acc = out["accepted"].cpu().numpy().T
    assert int((acc != ref["accepted"]).sum()) == 0
    assert rel_err(out["samples"].cpu().numpy().transpose(2, 0, 1), ref["traj"][:, 1:]).max() <= 1e-12
    st = ens.state()
    assert np.array_equal(st["aem_n"].cpu().numpy(), ref["aem_n"])
    np.testing.assert_allclose(st["aem_mean"].cpu().numpy().T, ref["aem_mean"], rtol=1e-9, atol=1e-13)
    assert ens.counters()["coarse_evals"] == int(ref["aem_model_evals"].sum())
    # the error model lifts the fine acceptance rate well above the plain two-level chain's (SURVEY 8f: 0.04 -> 0.35)
    plain = _ens(bp.linear_problem(True)[0], arrays, nc, seed=77)
    plain.set_state(th0)
    plain.run(ns, samples=False)
    assert acc[:, 150:].mean() > 2.0 * plain.counters()["accepted"] / (nc * ns)
    # resume: 300 = 120 + save/load + 180, bit exact (cache and error model are part of the state)
    b = _ens(meta, arrays, nc, seed=77, aem=meta["aem"])
    b.set_state(th0)
    first = b.run(120, samples=True)["samples"]
    c = _ens(meta, arrays, nc, seed=77, aem=meta["aem"])
    c.load_state(b.state())
    second = c.run(180, samples=True)["samples"]
    assert torch.equal(torch.cat([first, second]), out["samples"])
    with pytest.raises(ValueError):
        _ens(meta, arrays, 8, aem=dict(min_data=1))
    with pytest.raises(NotImplementedError):
        _ens(bp.lv_problem(True)[0], bp.lv_problem(True)[1], 8, aem=dict(min_data=5))


# ------------------------------------------------------------------------------------------
# diagnostics kernels
# ------------------------------------------------------------------------------------------

def test_iat_kernel_matches_reference_fixture():
    """integrated_autocorrelation of the reference (postprocessing/autocorrelation.py) on its own
    outputs: tests/golden/postprocessing.npz."""
    from yagre_mcmc_b200.ensemble import iat_ess
    _, a = load("postprocessing")
    for i in range(5):
        s = torch.as_tensor(a[f"seq{i}"], device="cuda").unsqueeze(2).contiguous()       # [N, d, 1]
        for method, key in (("max", "iat_max"), ("mean", "iat_mean")):
            iat, ess = iat_ess(s, method)
            assert int(iat[0]) == int(a[key][i]), (i, method)
            assert int(ess[0]) == s.shape[0] // max(int(a[key][i]), 1)


def test_iat_kernel_many_chains_matches_oracle():
    from oracle import cport
    from yagre_mcmc_b200.ensemble import iat_ess
    rng = np.random.default_rng(1)
    N, d, nc = 1500, 2, 96
    x = np.zeros((N, d, nc))
    rho = rng.uniform(0.0, 0.97, size=(d, nc))
    e = rng.standard_normal((N, d, nc))
    for t in range(1, N):
        x[t] = rho * x[t - 1] + e[t]
    iat, ess = iat_ess(torch.as_tensor(x, device="cuda"), "max")
    want = np.array([cport.iat(x[:, :, c], "max") for c in range(nc)])
    assert np.array_equal(iat.cpu().numpy(), want)
    assert np.array_equal(ess.cpu().numpy(), N // np.maximum(want, 1))


def test_iat_kernel_long_series():
    """Series longer than the shared-memory capacity (C2 / C3 run 100,000 / 50,000 steps per chain) go through
    the stream-ordered scratch path: same numbers as the oracle's restatement of the reference."""
    from oracle import cport
    from yagre_mcmc_b200.ensemble import iat_ess
    rng = np.random.default_rng(4)
    N, d, nc = 30000, 2, 5
    rho = np.array([[0.0, 0.5, 0.9, 0.97, 0.99], [0.3, 0.2, 0.95, 0.5, 0.9]])
    e = rng.standard_normal((N, d, nc))
    x = np.zeros((N, d, nc))
    for t in range(1, N):
        x[t] = rho * x[t - 1] + e[t]
    for method in ("max", "mean"):
        iat, ess = iat_ess(torch.as_tensor(x, device="cuda"), method)
        want = np.array([cport.iat(x[:, :, c], method) for c in range(nc)])
        assert np.array_equal(iat.cpu().numpy(), want), (method, iat, want)
        assert np.array_equal(ess.cpu().numpy(), N // np.maximum(want, 1))
    assert want.max() > 20


def test_split_moments_and_pooled_stats_match_numpy():
    from yagre_mcmc_b200.ensemble import split_moments
    from yagre_mcmc_b200.parallel import moments_from_stats, split_rhat
    meta, arrays = bp.gauss2d_problem()
    nc, ns = 1000, 400
    ens = _ens(meta, arrays, nc, seed=2)
    ens.set_state(np.tile(bp.GAUSS2D_MEAN, (nc, 1)))
    out = ens.run(ns, samples=True, accepted=True)
    s = out["samples"]
    x = s.cpu().numpy()
    hm, hv = split_moments(s)
    half = ns // 2
    np.testing.assert_allclose(hm[0].cpu().numpy(), x[:half].mean(0), rtol=1e-12, atol=1e-14)
    np.testing.assert_allclose(hm[1].cpu().numpy(), x[half:].mean(0), rtol=1e-12, atol=1e-14)
    np.testing.assert_allclose(hv[0].cpu().numpy(), x[:half].var(0, ddof=1), rtol=1e-11)
    np.testing.assert_allclose(hv[1].cpu().numpy(), x[half:].var(0, ddof=1), rtol=1e-11)
    rh = split_rhat(s)
    assert np.all(rh > 0.99) and np.all(rh < 1.1)
    # pooled statistics: Welford of the pre-transition states = theta0 followed by samples[:-1]
    pre = np.concatenate([np.tile(bp.GAUSS2D_MEAN[None, :, None], (1, 1, nc)), x[:-1]], axis=0)   # [ns, d, nc]
    pooled = moments_from_stats(ens.pooled_stats(), 2)
    flat = pre.transpose(0, 2, 1).reshape(-1, 2)
    np.testing.assert_allclose(pooled["mean"], flat.mean(0), rtol=1e-10, atol=1e-12)
    np.testing.assert_allclose(pooled["covariance"], np.cov(flat.T), rtol=1e-9)
    assert pooled["n_chains"] == nc and pooled["samples_per_chain"] == ns
    assert abs(pooled["acceptance_rate"] - out["accepted"].double().mean().item()) < 1e-12
    # deterministic two-stage reduction: bitwise reproducible
    assert torch.equal(ens.pooled_stats(), ens.pooled_stats())


# ------------------------------------------------------------------------------------------
# adaptive Metropolis (parity unpinned vs the reference; pinned vs the oracle's restatement)
# ------------------------------------------------------------------------------------------

AM_MEAN = np.array([1.0, 1.5])
AM_COV = np.array([[3.2, -0.4], [-0.4, 0.2]])      # test/test_adaptive.py target


def _am_problem():
    prec = np.linalg.inv(AM_COV)
    prec = 0.5 * (prec + prec.T)
    arrays = dict(prop_L=np.eye(2), L0_g_mean=AM_MEAN, L0_g_prec=prec, L0_g_logconst=0.0)
    return dict(model="gauss", dim=2, levels=1, J=1, eq="exact"), arrays


def test_adaptive_metropolis_matches_oracle_recurrence():
    meta, arrays = _am_problem()
    ad = dict(idle=10, collection=30, eps=1e-4, refresh=3)
    nc, ns = 256, 150
    th0 = np.tile([-3.0, 4.0], (nc, 1))
    ens = _ens(meta, arrays, nc, seed=21, adaptive=ad)
    ens.set_state(th0)
    out = ens.run(ns, samples=True, accepted=True, logpost=True, record=True)
    ref = _replay(meta, arrays, th0, out, adaptive=ad)
    acc = out["accepted"].cpu().numpy().T
    # the adapted factor goes through sqrt / divisions whose rounding may differ in the last ulp
    # between nvcc and gcc: decisions may flip only at ties; trajectories agree to 1e-9 otherwise
    flips = int((acc != ref["accepted"]).sum())
    assert flips == 0
    traj = out["samples"].cpu().numpy().transpose(2, 0, 1)
    assert rel_err(traj, ref["traj"][:, 1:]).max() <= 1e-9
    L = ens.state()["prop_L"].cpu().numpy()
    assert np.all(L[0, 1] == 0.0) and np.all(L[0, 0] > 0) and not np.allclose(L[0, 0], 1.0)


def test_adaptive_metropolis_moments_and_acceptance():
    """Thresholds of the reference's (skipped) test/test_adaptive.py:24-27,51,72,90."""
    from yagre_mcmc_b200.parallel import moments_from_stats
    meta, arrays = _am_problem()
    nc, ns = 2048, 6000
    ens = _ens(meta, arrays, nc, seed=19, adaptive=dict(idle=100, collection=500, eps=1e-4))
    ens.set_state(np.tile([-3.0, 4.0], (nc, 1)))
    ens.run(1500, samples=False)                          # burn-in + adaptation
    s = ens.run(ns, samples=True, accepted=True)
    x = s["samples"].cpu().numpy()                        # [ns, d, nc]
    flat = x.transpose(0, 2, 1).reshape(-1, 2)
    np.testing.assert_allclose(flat.mean(0), AM_MEAN, atol=0.03)
    np.testing.assert_allclose(np.cov(flat.T), AM_COV, atol=0.05)
    rate = s["accepted"].double().mean().item()
    assert 0.1 <= rate <= 0.8
    # the adapted proposal is close to s * target covariance, s = 2.4^2 / d
    L = ens.state()["prop_L"].cpu().numpy()               # [d, d, nc]
    C = np.einsum('ikc,jkc->ijc', L, L).mean(axis=2)
    np.testing.assert_allclose(C, 2.4 ** 2 / 2 * AM_COV, rtol=0.15, atol=0.05)


# ------------------------------------------------------------------------------------------
# full-size properties (BASELINE.json configs)
# ------------------------------------------------------------------------------------------

def test_c5_full_size_properties():
    """C5 at 65,536 chains per GPU: every chain advances, counters are consistent, the ensemble mean
    sits at the posterior mode region, and a perfect surrogate (coarse == fine) is never rejected at
    the fine screen (reference test/test_mlda.py:94-130)."""
    nc, ns = 65536, 40
    meta, arrays = bp.lv_problem(True)
    ens = _ens(meta, arrays, nc, seed=11)
    th0 = bp.lv_initial_states(nc)
    ens.set_state(th0)
    out = ens.run(ns, samples=True, accepted=True)
    acc = out["accepted"]
    c = ens.counters()
    assert c["transitions"] == nc * ns
    assert c["accepted"] == int(acc.sum().item())
    assert c["coarse_evals"] <= 3 * nc * ns and c["coarse_evals"] >= 3 * nc * ns - 10
    assert c["accepted"] <= c["fine_evals"] <= nc * ns
    rate = c["accepted"] / (nc * ns)
    assert 0.25 < rate < 0.5
    st = ens.state()
    assert torch.equal(st["n_accept"], acc.sum(dim=0).to(torch.int64))
    assert torch.equal(st["theta"], out["samples"][-1])
    assert torch.isfinite(st["logpost"]).all()
    m = out["samples"][-1].mean(dim=1).cpu().numpy()
    assert np.all(np.abs(m - bp.LV_TRUTH) < 0.1)
    # accepted <=> state changed
    prev = torch.cat([torch.as_tensor(th0.T, device="cuda").unsqueeze(0), out["samples"][:-1]])
    moved = (out["samples"] != prev).any(dim=1)
    assert torch.equal(moved, acc.bool())

    meta2, arrays2 = bp.lv_problem(True, Nc=96, Nf=96)
    ens2 = _ens(meta2, arrays2, 8192, seed=12)
    ens2.set_state(bp.lv_initial_states(8192))
    ens2.run(30, samples=False)
    c2 = ens2.counters()
    assert c2["fine_evals"] > 0
    assert abs(c2["accepted"] / c2["fine_evals"] - 1.0) < 1e-3


@pytest.mark.parametrize("two_level", [True, False])
def test_lv_posterior_moments_match_long_reference_runs(two_level):
    """north_star: posterior mean and covariance match long runs of the reference within Monte-Carlo
    error.  Fixture: 8 seeded chains x 9,000 steps of the UNMODIFIED reference chain stack (its own
    numpy RNG, no injection) on C5 / C4, written by oracle/make_golden.py case_lv_long.  The ensemble
    (65,536 chains) has a negligible error of its own, so the tolerance is the reference run's:
    5 standard errors of its mean (from the spread of the 8 chain means), 4 sqrt(2/ESS) on variances."""
    meta_r, ref = load("lv_long_twoLevel" if two_level else "lv_long_singleLevel")
    nc = 65536
    meta, arrays = bp.lv_problem(two_level)
    ens = _ens(meta, arrays, nc, seed=2024)
    ens.set_state(bp.lv_initial_states(nc))
    ens.run(150 if two_level else 400, samples=False)          # burn-in (IAT 4.3 / 17)
    out = ens.run(60, samples=True, thin=20)
    x = out["samples"].cpu().numpy().transpose(1, 0, 2).reshape(2, -1)     # 3 snapshots x 65,536 chains
    se = ref["chain_means"].std(axis=0, ddof=1) / np.sqrt(ref["chain_means"].shape[0])
    assert np.all(np.abs(x.mean(axis=1) - ref["mean"]) < 5.0 * se + 1e-3), (x.mean(axis=1), ref["mean"], se)
    cov = np.cov(x)
    rel = 4.0 * np.sqrt(2.0 / float(ref["ess"]))
    np.testing.assert_allclose(np.diag(cov), np.diag(ref["cov"]), rtol=rel)
    assert abs(cov[0, 1] - ref["cov"][0, 1]) < rel * np.sqrt(ref["cov"][0, 0] * ref["cov"][1, 1])
    c = ens.counters()
    rate = c["accepted"] / c["transitions"]
    assert abs(rate - ref["acceptance"].mean()) < 5.0 * ref["acceptance"].std(ddof=1) / np.sqrt(8) + 2e-3


def test_lv_forward_through_logpost_matches_reference_solver():
    """log-posterior of the device RK4 model at the fixture's parameter points against the value
    computed from the reference solver's forward output (DOP853, tests/golden/lv_forward.npz)."""
    _, a = load("lv_forward")
    meta, arrays = bp.lv_problem(True)
    ens = _ens(meta, arrays, len(a["thetas"]), seed=1)
    lp = ens.logpost(1, a["thetas"]).cpu().numpy()
    for i, th in enumerate(a["thetas"]):
        r = a["ref_forward"][i] - arrays["L1_data"]
        want = -0.5 * np.sum(r * (r @ arrays["L1_noise_prec"].T)) - 0.5 * th @ arrays["L1_prior_prec"] @ th
        assert abs(lp[i] - want) < 2e-3 * abs(want) + 2e-3, (i, lp[i], want)


@pytest.mark.parametrize("case", ["gauss2d", "gauss2d_adaptive", "linear_single_level", "linear_two_level", "gauss1d_isclose"])
def test_warp_specialised_small_ensemble_kernel_is_bit_identical(case):
    """Ensembles of <= 32,768 chains with d <= 2 and Philox noise run the warp-specialised variant of the
    one-chain-per-thread kernel (producer warp draws the noise into a shared-memory ring, consumer warp runs
    the state-dependent half).  Record mode always runs the plain kernel, which the Philox-replay tests pin to
    the oracle: samples, decisions, counters and the whole chain state must agree bit for bit, including a
    ragged last warp, one chain, thinning and a continued run."""
    am = None
    if case == "gauss2d":
        (meta, arrays), init = bp.gauss2d_problem(), lambda n: np.tile([-8.0, -7.0], (n, 1))
    elif case == "gauss2d_adaptive":
        (meta, arrays), init = bp.gauss2d_problem(), lambda n: np.tile([-8.0, -7.0], (n, 1))
        am = dict(idle=20, collection=30, refresh=3, eps=1e-4)
    elif case == "gauss1d_isclose":
        meta, a = load("mrw_gauss1d")
        arrays = {k: v for k, v in a.items() if k.startswith("L0_") or k == "prop_L"}
        init = lambda n: np.full((n, 1), -3.0)
    else:
        (meta, arrays), init = bp.linear_problem(case == "linear_two_level"), lambda n: np.zeros((n, 2))
    for nc in (1, 333):
        res = []
        for record in (False, True):
            ens = _ens(meta, arrays, nc, seed=77, adaptive=am)
            ens.set_state(init(nc))
            o1 = ens.run(120, samples=True, accepted=True, logpost=True, thin=3, record=record)
            o2 = ens.run(37, samples=True, accepted=True, record=record)          # continues (step index, Welford)
            launch = ens.last_launch()
            res.append((o1, o2, ens.counters(), ens.state(), launch))
        assert res[0][4]["block"] == 64 and res[1][4]["block"] == 128          # specialised vs plain kernel
        for k in ("samples", "accepted", "logpost"):
            assert torch.equal(res[0][0][k], res[1][0][k]), k
        assert torch.equal(res[0][1]["samples"], res[1][1]["samples"])
        assert res[0][2] == res[1][2]
        for k, v in res[0][3].items():
            if torch.is_tensor(v):
                assert torch.equal(v, res[1][3][k]), k


def test_pooled_proposal_covariance():
    """Optional pooled proposal covariance (north_star): after a burn-in with the example's poor proposal
    (1.0 I on a target with variances 2.4 / 0.7) the covariance pooled over all chains replaces it; the factor
    is chol(2.4^2/d Sigma_target) within Monte-Carlo error, the chains keep sampling the same target, and the
    C-ABI refuses factors that are not lower triangular / positive, and pCN ensembles."""
    from yagre_mcmc_b200.parallel import pooled_proposal_covariance
    nc = 4096
    meta, arrays = bp.gauss2d_problem()
    ens = _ens(meta, arrays, nc, seed=31)
    ens.set_state(np.tile([1.0, 1.5], (nc, 1)))
    ens.run(3000, samples=False)
    c0 = ens.counters()
    out = pooled_proposal_covariance(ens)
    want = np.linalg.cholesky(2.4 * 2.4 / 2 * bp.GAUSS2D_COV)
    np.testing.assert_allclose(out["prop_L"], want, rtol=0.05, atol=0.02)
    ens.run(2000, samples=False)
    c1 = ens.counters()
    th = ens.state()["theta"].cpu().numpy()
    se = np.sqrt(np.diag(bp.GAUSS2D_COV) / nc)
    assert np.all(np.abs(th.mean(1) - bp.GAUSS2D_MEAN) < 4.5 * se)
    np.testing.assert_allclose(np.cov(th), bp.GAUSS2D_COV, rtol=0.12, atol=0.03)
    rate0 = c0["accepted"] / c0["transitions"]
    rate1 = (c1["accepted"] - c0["accepted"]) / (c1["transitions"] - c0["transitions"])
    assert 0.28 < rate1 < 0.42 and abs(rate1 - 0.35) < abs(rate0 - 0.35) + 0.02     # 2-D optimal scaling: ~0.35
    # the same call on an adaptive ensemble restarts every chain's factor from the pooled one
    ens_a = _ens(meta, arrays, 256, seed=32, adaptive=dict(idle=10 ** 9, collection=10 ** 9, refresh=1, eps=1e-4))
    ens_a.set_state(np.tile([1.0, 1.5], (256, 1)))
    ens_a.run(10, samples=False)
    ens_a.set_proposal_factor(want)
    ens_a.run(1, samples=False)
    L = ens_a.state()["prop_L"].cpu().numpy()                      # [d, d, n]
    np.testing.assert_array_equal(L, np.broadcast_to(want[:, :, None], L.shape))
    with pytest.raises((ValueError, RuntimeError)):
        ens.set_proposal_factor(np.array([[1.0, 0.5], [0.0, 1.0]]))
    with pytest.raises((ValueError, RuntimeError)):
        ens.set_proposal_factor(np.array([[1.0, 0.0], [0.0, -1.0]]))
    metap, arraysp = bp.lv_pcn_problem()
    ens_p = _ens(metap, arraysp, 64, seed=33)
    ens_p.set_state(bp.lv_initial_states(64))
    with pytest.raises((NotImplementedError, RuntimeError)):
        ens_p.set_proposal_factor(np.eye(2))


def test_c4_single_level_full_size():
    nc, ns = 65536, 10
    meta, arrays = bp.lv_problem(False)
    ens = _ens(meta, arrays, nc, seed=13)
    ens.set_state(bp.lv_initial_states(nc))
    out = ens.run(ns, samples=True, accepted=True)
    c = ens.counters()
    assert c["fine_evals"] == nc * ns and c["coarse_evals"] == 0
    assert 0.04 < c["accepted"] / (nc * ns) < 0.6       # measured 0.087 with proposal variance 0.15
    assert torch.isfinite(out["samples"]).all()


def test_c3_linear_posterior_moments():
    """Linear-Gaussian model: the posterior is Gaussian in closed form; 16,384 chains (C3) must
    reproduce its mean and covariance.  Single level: within Monte-Carlo error (4.5 standard errors of
    one ensemble snapshot).  Two level: this coarse/fine pair mixes very slowly (fine acceptance 0.10,
    relaxation time of the ensemble variance ~5e4 steps measured on the device), so the two-level
    check is a looser one; exactness of the two-level step is pinned by the trajectory fixtures."""
    nc = 16384
    mean, cov = bp.linear_posterior('f')
    se = np.sqrt(np.diag(cov) / nc)
    meta, arrays = bp.linear_problem(False)
    ens = _ens(meta, arrays, nc, seed=17)
    ens.set_state(np.zeros((nc, 2)))
    ens.run(5000, samples=False)
    th = ens.state()["theta"].cpu().numpy()
    assert np.all(np.abs(th.mean(1) - mean) < 4.5 * se)
    np.testing.assert_allclose(np.cov(th), cov, rtol=0.06, atol=2e-3)

    meta, arrays = bp.linear_problem(True)
    ens = _ens(meta, arrays, nc, seed=17)
    ens.set_state(np.zeros((nc, 2)))
    ens.run(30000, samples=False)
    s = ens.run(2000, thin=500, samples=True)["samples"].cpu().numpy()    # [4, d, nc]
    flat = s.transpose(0, 2, 1).reshape(-1, 2)
    np.testing.assert_allclose(flat.mean(0), mean, atol=0.03)
    np.testing.assert_allclose(np.cov(flat.T), cov, rtol=0.15, atol=5e-3)
    c = ens.counters()
    assert 0.05 < c["accepted"] / c["transitions"] < 0.2


def test_c2_gaussian_target_moments():
    nc = 4096
    meta, arrays = bp.gauss2d_problem()
    ens = _ens(meta, arrays, nc, seed=23)
    ens.set_state(np.tile([-8.0, -7.0], (nc, 1)))
    ens.run(1000, samples=False)
    s = ens.run(500, thin=10, samples=True)["samples"].cpu().numpy()
    flat = s.transpose(0, 2, 1).reshape(-1, 2)
    np.testing.assert_allclose(flat.mean(0), bp.GAUSS2D_MEAN, atol=0.02)
    np.testing.assert_allclose(np.cov(flat.T), bp.GAUSS2D_COV, atol=0.05)


# ------------------------------------------------------------------------------------------
# edge cases: smallest / largest / ragged sizes
# ------------------------------------------------------------------------------------------

@pytest.mark.parametrize("shape", ["one_chain", "one_design_point", "one_rk4_step", "j1", "many_design_points",
                                   "long_observation_grid"])
def test_lv_edge_shapes_against_oracle(shape):
    kw = dict(one_chain=dict(), one_design_point=dict(n_data=1), one_rk4_step=dict(Nc=1, Nf=3),
              j1=dict(J=1), many_design_points=dict(n_data=37, Nc=8, Nf=24),
              # > 128 design points: numpy's pairwise summation blocks (np_pairwise_sum), 8 chains per CTA chunk
              long_observation_grid=dict(n_data=300, Nc=4, Nf=12, prop_var=2e-4))[shape]
    nc = 1 if shape == "one_chain" else 97
    meta, arrays = bp.lv_problem(True, **({"Nc": 16, "Nf": 48} | kw))
    th0 = bp.lv_initial_states(nc)
    ens = _ens(meta, arrays, nc, seed=3)
    ens.set_state(th0)
    out = ens.run(15, samples=True, accepted=True, logpost=True, record=True)
    ref = _replay(meta, arrays, th0, out)
    assert int((out["accepted"].cpu().numpy().T != ref["accepted"]).sum()) == 0
    assert rel_err(out["samples"].cpu().numpy().transpose(2, 0, 1), ref["traj"][:, 1:]).max() <= 1e-12
    lp = out["logpost"].cpu().numpy().transpose(2, 0, 1)
    assert rel_err(lp[:, :, 1], ref["logpost_L1"][:, 1:]).max() <= LOGPOST_RTOL


def test_zero_steps_and_repeated_short_runs():
    """n_steps = 0 is a no-op; 12 runs of 1 transition equal one run of 12 (step index carries over)."""
    meta, arrays = bp.lv_problem(True, Nc=16, Nf=48)
    nc = 130
    th0 = bp.lv_initial_states(nc)
    a = _ens(meta, arrays, nc, seed=9)
    a.set_state(th0)
    ref = a.run(12, samples=True)["samples"]
    b = _ens(meta, arrays, nc, seed=9)
    b.set_state(th0)
    assert b.run(0, samples=True)["samples"].shape[0] == 0
    parts = [b.run(1, samples=True)["samples"] for _ in range(12)]
    assert torch.equal(torch.cat(parts), ref)
    assert b.counters()["step_index"] == 12


def test_c5_full_ensemble_on_one_gpu():
    """524,288 chains (the whole C5 ensemble) on one device: every chain advances, no chain is lost at the
    CTA chunk boundaries (each CTA walks its 3,543 chains in chunks of <= 1,024)."""
    nc = 524288
    meta, arrays = bp.lv_problem(True)
    ens = _ens(meta, arrays, nc, seed=21)
    th0 = bp.lv_initial_states(nc)
    ens.set_state(th0)
    out = ens.run(4, samples=True, accepted=True)
    c = ens.counters()
    assert c["transitions"] == 4 * nc and c["coarse_evals"] >= 3 * 4 * nc - 8
    acc = out["accepted"]
    assert torch.equal(ens.state()["n_accept"], acc.sum(dim=0).to(torch.int64))
    moved = (out["samples"][0] != torch.as_tensor(th0.T, device="cuda")).any(dim=0)
    assert torch.equal(moved, acc[0].bool())
    # chain-offset keying: chains [1000, 1100) of the big run equal a 100-chain handle with chain_offset 1000
    sub = _ens(meta, arrays, 100, seed=21, chain_offset=1000)
    sub.set_state(th0[1000:1100])
    assert torch.equal(sub.run(4, samples=True)["samples"], out["samples"][:, :, 1000:1100])
