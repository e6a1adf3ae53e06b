"""Helpers the test modules share: the north-star tolerance, the ensemble constructor and the oracle replay of recorded
noise, host programs built with nvcc, a free port for the gloo tests, the problem builders several suites run, and the
GPU drivers of the diagnostics, log-posterior and pooled-sample suites.

A plain module, not a conftest.  yagre_mcmc_b200.ensemble and oracle are imported inside the functions that use them,
so CPU-only test modules can import this one."""
import os
import shutil
import socket
import subprocess

import numpy as np
import pytest
import torch

import bench_problems as bp
import logpost_reference as R
from diag_reference import check_pooled, check_welford, pre_states
from golden_io import load

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

LOGPOST_RTOL = 1e-10      # north_star: 1e-10 relative on log-posterior


def ensemble(meta, arrays, nc, **kw):
    from yagre_mcmc_b200.ensemble import ChainEnsemble, LoweredProblem
    return ChainEnsemble(LoweredProblem(meta, arrays), nc, **kw)


def replay(meta, arrays, th0, out, rows=None, adaptive=None):
    """Runs the oracle on the noise the device recorded (chain-major layout), on the chains `rows` if given;
    meta['aem'] is honoured."""
    from oracle import cport
    z = out["z"].cpu().numpy().transpose(3, 0, 1, 2)
    u_c = np.nan_to_num(out["u_c"].cpu().numpy().transpose(2, 0, 1), nan=0.5)
    u_f = np.nan_to_num(out["u_f"].cpu().numpy().transpose(1, 0), nan=0.5)
    if rows is not None:
        z, u_c, u_f, th0 = z[rows], u_c[rows], u_f[rows], th0[rows]
    return cport.run_injected(cport.Problem(meta, arrays, adaptive=adaptive), th0, z, u_c, u_f)


def host_program(tmp_path, name, source):
    """Compiles `source` with nvcc (-std=c++17 -O2, the repository root on the include path), runs it and returns its
    stdout.  nvcc is taken from PATH, else from the CUDA toolkit under CUDA_HOME (default /usr/local/cuda); the test is
    skipped where there is none."""
    nvcc = shutil.which("nvcc") or os.path.join(os.environ.get("CUDA_HOME") or "/usr/local/cuda", "bin", "nvcc")
    if not os.path.exists(nvcc):
        pytest.skip("nvcc not found")
    src = tmp_path / f"{name}.cu"
    src.write_text(source)
    exe = tmp_path / name
    subprocess.run([nvcc, "-std=c++17", "-O2", "-I", ROOT, str(src), "-o", str(exe)], check=True, capture_output=True)
    return subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout


def free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


# ------------------------------------------------------------------------------------------------------------------
# problems
# ------------------------------------------------------------------------------------------------------------------
def fixture(name):
    meta, a = load(name)
    return meta, {k: v for k, v in a.items() if k.startswith(("L0_", "L1_", "L2_")) or k in ("prop_L", "pcn_mean")}


def three_level_gauss():
    _, a = load("mlda3_gauss2d")
    arrays = {k: a[k] for k in a if k.startswith(("L0_", "L1_", "L2_")) or k == "prop_L"}
    return dict(model="gauss", dim=2, levels=3, J=6, eq="exact"), arrays


def lv_tempered():
    meta, arrays = bp.lv_problem(True)
    return meta, dict(arrays, L0_tempering=np.array(0.4))


def dense_noise_linear():
    meta, arrays = bp.big_linear_problem(5, 4, 3, two_level=False, seed=12)
    A = np.random.default_rng(3).standard_normal((4, 4))
    return meta, dict(arrays, L0_noise_prec=A @ A.T + 4 * np.eye(4), L0_prior_mean=np.full(5, 0.7))


def dense_prior_tensor():
    rng = np.random.default_rng(11)
    d, dd = 24, 40
    meta, arrays = bp.big_linear_problem(d, dd, 2)
    A = rng.standard_normal((d, d))
    prec = np.linalg.inv(1.5 * (A @ A.T / d + 0.5 * np.eye(d)))
    return meta, dict(arrays, L0_prior_prec=0.5 * (prec + prec.T), L0_prior_mean=0.1 * rng.standard_normal(d))


def qconst_tensor():
    """Misfit dominated by q_const: 2,000 data rows scattered (sd 30) about the model, far beyond the noise (0.05)."""
    meta, arrays = bp.big_linear_problem(23, 45, 1, seed=5)
    rng = np.random.default_rng(6)
    data = arrays["L0_data"][0] + 30.0 * rng.standard_normal((2000, 45))
    return meta, dict(arrays, L0_data=data)


def _near_zero_tensor():
    """|lp| about 1e-4: noise and prior precisions of 1e-6."""
    meta, arrays = bp.big_linear_problem(9, 1, 3, seed=8)
    return meta, dict(arrays, L0_noise_prec=np.full((1, 1), 1e-6), L0_prior_prec=1e-6 * np.eye(9))


def _tensor_4_warps():
    """d = 64, two levels of 176 and 192 rows: the blob (206,208 bytes) and four warps' tiles take 232,320 bytes, within
    the 227 KiB of one block."""
    meta, arrays = bp.big_linear_problem(64, 192, 1, two_level=True, J=2, seed=9)
    r = slice(0, 176)
    return meta, dict(arrays, L0_data=arrays["L0_data"][:, r], L0_G=arrays["L0_G"][r], L0_b=arrays["L0_b"][r],
                      L0_noise_prec=arrays["L0_noise_prec"][r, r])


TENSOR = {
    "9x1": lambda: bp.big_linear_problem(9, 1, 3, seed=2),
    "23x45": lambda: bp.big_linear_problem(23, 45, 3),
    "32x96_two_level": lambda: bp.big_linear_problem(32, 96, 2, two_level=True, J=3),
    "64x256": lambda: bp.big_linear_problem(64, 256, 1),
    "dense_prior": dense_prior_tensor,
    "q_const_dominated": qconst_tensor,
    "near_zero": _near_zero_tensor,
    "64x176_192_four_warps": _tensor_4_warps,
}


def _pcn_linear():
    meta, arrays = bp.linear_problem(False)
    return dict(meta, proposal="pcn", pcn_step=0.05), dict(arrays, pcn_mean=np.array([0.3, -0.2]))


SCHEDULES = {
    # name: (problem, chains, steps, initial states)
    "lv_two_level": (lambda: bp.lv_problem(True), 24, 4, lambda n: bp.lv_initial_states(n)),
    "lv_single_level": (lambda: bp.lv_problem(False), 24, 5, lambda n: bp.lv_initial_states(n)),
    "lv_pcn": (bp.lv_pcn_problem, 24, 5, lambda n: bp.lv_initial_states(n)),
    "gauss_single_level": (bp.gauss2d_problem, 64, 10, lambda n: np.tile([-1.0, 2.0], (n, 1))),
    "gauss_isclose_1d": (lambda: fixture("mrw_gauss1d"), 64, 10, lambda n: np.full((n, 1), -1.0)),
    "linear_pcn": (_pcn_linear, 64, 10, lambda n: np.zeros((n, 2))),
    "linear_two_level": (lambda: bp.linear_problem(True), 64, 8, lambda n: np.zeros((n, 2))),
    "linear_tempered_surrogate": (lambda: fixture("mlda_linear_tempered"), 64, 8, lambda n: np.zeros((n, 2))),
    "gauss_three_level": (lambda: fixture("mlda3_gauss2d"), 64, 8, lambda n: np.tile([0.5, 1.0], (n, 1))),
    "tensor_single_level": (lambda: bp.big_linear_problem(23, 45, 3), 32, 6,
                            lambda n: 0.01 * np.random.default_rng(2).standard_normal((n, 23))),
    "tensor_two_level": (lambda: bp.big_linear_problem(32, 96, 2, two_level=True, J=3), 32, 5,
                         lambda n: 0.01 * np.random.default_rng(3).standard_normal((n, 32))),
}


def aem_problem(d, dd, n_data, J, min_data, heuristic, dense_prop=False, dense_prior=False, zero_error_rows=0,
                seed=0, error_scale=1.0, spread=1.5, prop_scale=2.4, eq="exact"):
    """Two-level linear model for the adaptive error model, d parameters and dd data components, diagonal noise.
    The coarse model is the fine one with row k of G and b perturbed at a scale error_scale x noise sd x 10^(spread
    (k / (dd - 1) - 1)) (so the error variances span 2 spread decades: the heuristic clamps when that ratio passes 50);
    the last zero_error_rows rows are left identical to the fine level's, so those error components are exactly 0.
    The proposal is prop_scale / sqrt(d) times the fine posterior's Cholesky factor (dense_prop) or its marginal sds."""
    rng = np.random.default_rng(seed)
    truth = rng.standard_normal(d)
    G_f = rng.standard_normal((dd, d)) / np.sqrt(d)
    b_f = 0.1 * rng.standard_normal(dd)
    sd = 0.1 * (1.0 + 0.5 * np.arange(dd) / dd)
    scale = error_scale * sd * 10.0 ** (spread * (np.arange(dd) / max(dd - 1, 1) - 1.0))
    G_c = G_f + scale[:, None] * rng.standard_normal((dd, d))
    b_c = b_f + scale * rng.standard_normal(dd)
    if zero_error_rows:
        G_c[dd - zero_error_rows:], b_c[dd - zero_error_rows:] = G_f[dd - zero_error_rows:], b_f[dd - zero_error_rows:]
    data = truth @ G_f.T + b_f + sd * rng.standard_normal((n_data, dd))
    prior_prec = np.eye(d) / 4.0
    if dense_prior:
        A = rng.standard_normal((d, d))
        prior_prec = np.linalg.inv(A @ A.T / d + np.eye(d))
        prior_prec = 0.5 * (prior_prec + prior_prec.T)
    prior_mean = truth + 0.3 * rng.standard_normal(d)
    arrays = {}
    for l, (G, b) in enumerate(((G_c, b_c), (G_f, b_f))):
        arrays.update({f"L{l}_G": G, f"L{l}_b": b, f"L{l}_data": data, f"L{l}_noise_prec": np.diag(1.0 / sd ** 2),
                       f"L{l}_prior_mean": prior_mean, f"L{l}_prior_prec": prior_prec})
    _, cov = bp.linear_gaussian_posterior(arrays, 1)
    arrays["prop_L"] = prop_scale / np.sqrt(d) * (np.linalg.cholesky(cov) if dense_prop else np.diag(np.sqrt(np.diag(cov))))
    meta = dict(model="linear", dim=d, levels=2, J=J, eq=eq, aem=dict(min_data=min_data, heuristic=bool(heuristic)))
    return meta, arrays


def aem_start(arrays, nc, seed):
    """nc initial states drawn from the fine level's posterior."""
    mean, cov = bp.linear_gaussian_posterior(arrays, 1)
    return mean + np.random.default_rng(seed).standard_normal((nc, mean.size)) @ np.linalg.cholesky(cov).T


# The AEM value sweep: every (capacity(d), capacity(data_dim)) pair of aem_mh_kernel<D, DD> once.
# name: (aem_problem kwargs, chains, steps, thin)
AEM_SWEEP = {
    "1x1": (dict(d=1, dd=1, n_data=129, J=1, min_data=8, heuristic=True, seed=1), 1, 60, 1),
    "1x3": (dict(d=1, dd=3, n_data=9, J=5, min_data=2, heuristic=True, seed=2), 33, 40, 1),
    "2x8": (dict(d=2, dd=8, n_data=2, J=2, min_data=3, heuristic=False, zero_error_rows=2, error_scale=0.3, seed=3),
            4097, 24, 1),
    "3x2": (dict(d=3, dd=2, n_data=1, J=5, min_data=3, heuristic=True, dense_prop=True, seed=4), 33, 42, 3),
    "3x3": (dict(d=3, dd=3, n_data=129, J=1, min_data=8, heuristic=False, error_scale=0.1, prop_scale=0.5, seed=5),
            33, 50, 1),
    "3x5": (dict(d=3, dd=5, n_data=9, J=2, min_data=2, heuristic=True, zero_error_rows=1, dense_prior=True, seed=6),
            4097, 24, 1),
    "5x1": (dict(d=5, dd=1, n_data=2, J=2, min_data=3, heuristic=True, dense_prop=True, dense_prior=True, seed=7),
            1, 60, 1),
    "8x3": (dict(d=8, dd=3, n_data=9, J=5, min_data=2, heuristic=True, dense_prop=True, error_scale=0.1, prop_scale=0.5,
                seed=8), 33, 40, 1),
    "8x8": (dict(d=8, dd=8, n_data=129, J=2, min_data=8, heuristic=True, zero_error_rows=3, error_scale=0.1,
                prop_scale=0.5, seed=9), 33, 40, 1),
}

# Forced-decision cases, at least one per parameter capacity: the heuristic floors without clamping (d2_floor),
# clamps (d4_clamp) and neither (d8_one_component: one data component, scaling 2).  name: (kwargs, chains, steps)
AEM_FORCED = {
    "d2_floor": (dict(d=2, dd=3, n_data=9, J=5, min_data=3, heuristic=True, zero_error_rows=1, error_scale=0.02,
                      spread=0.0, seed=11), 64, 40),
    "d4_clamp": (dict(d=3, dd=4, n_data=2, J=3, min_data=2, heuristic=True, seed=12), 64, 40),
    "d8_one_component": (dict(d=6, dd=1, n_data=129, J=2, min_data=8, heuristic=True, dense_prop=True, seed=13), 64, 40),
    "d8_no_heuristic": (dict(d=8, dd=5, n_data=9, J=5, min_data=3, heuristic=False, zero_error_rows=1, seed=14), 64, 40),
}


def aem_forced_inputs(name, seed=0):
    """(meta, arrays, theta0, z, pattern) of an AEM_FORCED case."""
    kw, nc, ns = AEM_FORCED[name]
    meta, arrays = aem_problem(**kw)
    th0 = aem_start(arrays, nc, kw["seed"] + 100 + seed)
    z = schedule_noise(meta, nc, ns, kw["seed"] + 200 + seed)
    pattern = R.random_pattern(nc, ns, meta["J"], kw["seed"] + 300 + seed)
    return meta, arrays, th0, z, pattern


def schedule_noise(meta, nc, ns, seed):
    J = int(meta["J"]) if int(meta["levels"]) >= 2 else 1
    return np.random.default_rng(seed).standard_normal((nc, ns, J, int(meta["dim"])))


# ------------------------------------------------------------------------------------------------------------------
# chain diagnostics against the high-precision reference (test_diagnostics_reference_gpu)
# ------------------------------------------------------------------------------------------------------------------
def _drive(meta, arrays, th0, plan, record, kw):
    """Runs plan on a handle: ("run", k) | ("restart", theta) = set_state(theta, keep_diagnostics=True) |
    ("reload",) = state() loaded into a fresh handle.  Returns the last handle and, per run, its outputs, the state it
    started from, the restart state before it (or None) and the index of the handle that ran it."""
    nc = th0.shape[0]
    ens = ensemble(meta, arrays, nc, **kw)
    ens.set_state(th0)
    runs, x, restart, handle = [], np.asarray(th0, dtype=np.float64), None, 0
    for op in plan:
        if op[0] == "run":
            out = ens.run(op[1], samples=True, accepted=True, logpost=True, record=record)
            runs.append(dict(out=out, start=x, restart=restart, handle=handle, launch=ens.last_launch()))
            x, restart = out["samples"][-1].t().cpu().numpy(), None
        elif op[0] == "restart":
            ens.set_state(op[1], keep_diagnostics=True)
            x = restart = np.asarray(op[1], dtype=np.float64)
        else:
            st = ens.state()
            ens.close()
            ens = ensemble(meta, arrays, nc, **kw)
            ens.load_state(st)
            handle += 1
    torch.cuda.synchronize()
    return ens, runs


def _expected_counts(meta, arrays, runs, adaptive, nc):
    """Counters of the last handle and the per-chain accept / coarse-accept counts since the reset, from the oracle's
    replay of every run's recorded noise (its evaluation totals include one initial evaluation per chain per level)."""
    lv = meta["levels"]
    want = dict(transitions=0, accepted=0, coarse_evals=0, mid_evals=0, fine_evals=0, coarse_accepted=0)
    n_acc, c_acc = np.zeros(nc, dtype=np.int64), np.zeros(nc, dtype=np.int64)
    last = runs[-1]["handle"]
    for r in runs:
        ref = replay(meta, arrays, r["start"], r["out"], adaptive=adaptive)
        acc = r["out"]["accepted"].cpu().numpy().T
        assert np.array_equal(acc, ref["accepted"])
        n_acc += ref["accepted"].sum(axis=1, dtype=np.int64)
        c_acc += ref["coarse_accepted"]
        if r["handle"] != last:
            continue
        ev = [int(v) - nc for v in ref["n_evals"]]
        want["transitions"] += acc.size
        want["accepted"] += int(ref["accepted"].sum())
        want["coarse_accepted"] += int(ref["coarse_accepted"].sum())
        if meta.get("aem"):
            want["coarse_evals"] += int(ref["aem_model_evals"].sum())
            want["fine_evals"] += ev[1]
        elif lv == 1:
            want["fine_evals"] += ev[0]
        elif lv == 2:
            want["coarse_evals"] += ev[0]
            want["fine_evals"] += ev[1]
        else:
            want["coarse_evals"] += ev[0]
            want["mid_evals"] += ev[1]
            want["fine_evals"] += ev[2]
    return want, n_acc, c_acc


def _state_np(st):
    return {k: v.cpu().numpy() for k, v in st.items() if torch.is_tensor(v)}


def check_case(meta, arrays, th0, plan, seed=1, adaptive=None, aem=None, ws=None, smem=None, label="", **kw):
    """The whole check of one case (see test_diagnostics_reference_gpu's docstring).  ws: the Philox run must (True) or
    must not (False) run the warp-specialised kernel; smem: the tensor path's expected dynamic shared memory of every
    launch."""
    nc = th0.shape[0]
    kw = dict(kw, seed=seed, adaptive=adaptive, aem=aem)
    rec_ens, rec = _drive(meta, arrays, th0, plan, True, kw)
    ens, free = _drive(meta, arrays, th0, plan, False, kw)
    # 1. production instances == recording instances, bit for bit
    for a, b in zip(rec, free):
        for k in ("samples", "accepted", "logpost"):
            assert torch.equal(a["out"][k], b["out"][k]), (label, k)
        if ws is not None:
            assert a["launch"]["block"] != 64 and (b["launch"]["block"] == 64) == ws, (label, a["launch"], b["launch"])
        if smem is not None:
            assert a["launch"]["smem"] == b["launch"]["smem"] == smem, (label, a["launch"], b["launch"], smem)
    st_rec, st = rec_ens.state(), ens.state()
    for k, v in st.items():
        assert (torch.equal(v, st_rec[k]) if torch.is_tensor(v) else v == st_rec[k]), (label, k)
    c = ens.counters()
    assert c == rec_ens.counters(), label
    # 2. Welford moments against the long-double reference of the pre-transition states
    pre = pre_states(th0, [r["out"]["samples"].cpu().numpy() for r in rec], [r["restart"] for r in rec])
    s = _state_np(st)
    check_welford(s["w_mean"], s["w_m2"], c["welford_n"], pre, label)
    # 3. counts: the accept flags, the oracle replay, the counters
    flags = sum(r["out"]["accepted"].to(torch.int64).sum(dim=0) for r in rec).cpu().numpy()
    want, n_acc, c_acc = _expected_counts(meta, arrays, rec, adaptive, nc)
    assert np.array_equal(s["n_accept"], flags) and np.array_equal(s["n_accept"], n_acc), label
    got = {k: c[k] for k in want}
    assert got == want, (label, got, want)
    if meta["levels"] == 1:
        assert c["coarse_accepted"] == 0 and not c_acc.any(), label
    # 4. pooled statistics (d <= 8)
    if meta["dim"] <= 8:
        check_pooled(ens.pooled_stats().cpu().numpy(), s, c["welford_n"], pre, label)
    rec_ens.close()
    ens.close()
    return c


# ------------------------------------------------------------------------------------------------------------------
# log-posteriors against the long-double reference (test_logpost_reference_gpu)
# ------------------------------------------------------------------------------------------------------------------
def _check_level(meta, arrays, l, theta, got, label):
    """theta [n, d], got [n]: level l within the bound; -inf exactly where the reference says so."""
    lp, b = R.logpost_bound(meta, arrays, l, theta)
    ref = np.asarray(lp, dtype=np.float64)
    got = np.asarray(got, dtype=np.float64)
    inf = ref == -np.inf
    assert np.array_equal(got[inf], ref[inf]), (label, l, "-inf")
    e = np.abs(got[~inf].astype(np.longdouble) - lp[~inf]).astype(np.float64)
    assert np.all(e <= b[~inf]), (label, l, float((e / b[~inf]).max()), int(np.argmax(e / b[~inf])))


def _check_values(meta, arrays, theta, lp_dev, label):
    for l in range(int(meta["levels"])):
        _check_level(meta, arrays, l, theta, lp_dev[l], label)


def value_case(meta, arrays, th0, runs=(3, 2), sample=None, stored=None, seed=3, **kw):
    """Short Philox runs; after each, the state (and the stored steps of `stored` chains of the sample) against the
    reference, and yg_logpost at the same points."""
    nc = th0.shape[0]
    idx = np.arange(nc) if sample is None or sample >= nc else np.sort(
        np.random.default_rng(seed).choice(nc, sample, replace=False))
    st_idx = idx if stored is None else idx[:stored]
    ens = ensemble(meta, arrays, nc, seed=seed, **kw)
    ens.set_state(th0)
    label = f"{meta['model']} d={meta['dim']} L={meta['levels']} nc={nc}"
    for k in runs:
        out = ens.run(k, samples=True, logpost=True)
        torch.cuda.synchronize()
        st = ens.state()
        th = st["theta"].cpu().numpy().T[idx]
        _check_values(meta, arrays, th, st["logpost"].cpu().numpy()[:, idx], label)
        sm, lps = out["samples"].cpu().numpy(), out["logpost"].cpu().numpy()
        for s in range(k):
            _check_values(meta, arrays, sm[s].T[st_idx], lps[s][:, st_idx], f"{label} step {s}")
        for l in range(int(meta["levels"])):
            _check_level(meta, arrays, l, th, ens.logpost(l, th).cpu().numpy(), f"{label} yg_logpost")
    ens.close()


# ------------------------------------------------------------------------------------------------------------------
# linear models through the builders (test_pooled_samples_gpu)
# ------------------------------------------------------------------------------------------------------------------
def linear_chain(d, dd, two_level, nc, seed, thin, store=True, pcn=False):
    from yagre_mcmc_b200.parameter import ParameterVector
    from yagre_mcmc_b200.model import ForwardModel, LinearModelSolver
    from yagre_mcmc_b200.statistics import (IIDCovarianceMatrix, Gaussian, CentredGaussianNoise, Data,
                                            AdditiveGaussianNoiseLikelihood, BayesianRegressionModel,
                                            BayesianRegressionModelHierarchy)
    from yagre_mcmc_b200.utility import Hierarchy, SharedComponent
    from yagre_mcmc_b200.chain.method import MRWBuilder, MLDABuilder, PCNBuilder
    meta, a = bp.big_linear_problem(d, dd, 1, two_level=two_level, J=3)
    noise = CentredGaussianNoise(IIDCovarianceMatrix(dd, 0.05))
    prior = Gaussian(ParameterVector(np.zeros(d)), IIDCovarianceMatrix(d, 2.0))
    levels = 2 if two_level else 1
    lik = [AdditiveGaussianNoiseLikelihood(Data(a["L0_data"]), ForwardModel(LinearModelSolver(a[f"L{l}_G"], a[f"L{l}_b"])),
                                           noise) for l in range(levels)]
    prop = IIDCovarianceMatrix(d, float(a["prop_L"][0, 0]) ** 2)
    if two_level:
        b = MLDABuilder()
        b.bayesModel = BayesianRegressionModelHierarchy(Hierarchy(lik), SharedComponent(prior, 2))
        b.baseProposalCovariance = prop
        b.subChainLengths = [3]
    elif pcn:
        b = PCNBuilder()
        b.bayesModel = BayesianRegressionModel(lik[0], prior)
        b.stepSize = 0.01
    else:
        b = MRWBuilder()
        b.bayesModel = BayesianRegressionModel(lik[0], prior)
        b.proposalCovariance = prop
    b.nChains, b.seed, b.thin, b.storeTrajectory = nc, seed, thin, store
    return b.build_method(), bp.linear_gaussian_posterior(a, levels - 1)


def check_closed_form(out, mean, cov, C, label):
    """Chains started from exact posterior draws are stationary: each is worth at least one independent draw, so the
    pooled mean has variance <= Sigma_ii / C and the pooled covariance (Sigma_ii Sigma_jj + Sigma_ij^2) / C."""
    sm = np.sqrt(np.diag(cov) / C)
    assert np.all(np.abs(out["mean"] - mean) <= 5 * sm), (label, "mean", np.abs(out["mean"] - mean).max())
    dg = np.diag(cov)
    sc = np.sqrt((np.outer(dg, dg) + cov ** 2) / C)
    assert np.all(np.abs(out["covariance"] - cov) <= 5 * sc), (label, "covariance", (np.abs(out["covariance"] - cov) / sc).max())


# ------------------------------------------------------------------------------------------------------------------
# adaptive Metropolis (test_am_reference_cpu, test_am_reference_gpu)
# ------------------------------------------------------------------------------------------------------------------
def am_problem(d, dd=2, levels=1, J=3, n_data=4, offset=0.0, spread=0.3, frozen=None, prop_scale=1.0, seed=0):
    """Linear model G theta + b with d parameters and dd data components, one level or two (level 0 the fine model
    with G and b perturbed by 5 %).  The posterior sits near `offset` (every coordinate) with spreads of about
    `spread`; the proposal factor is prop_scale x spread x a random lower-triangular matrix with unit diagonal, with
    row `frozen` (if given) exactly zero: that coordinate never moves while the chain runs on this factor."""
    rng = np.random.default_rng(seed)
    truth = offset + spread * rng.standard_normal(d)
    G = rng.standard_normal((dd, d)) / np.sqrt(d)
    b = 0.1 * rng.standard_normal(dd)
    data = truth @ G.T + b + spread * rng.standard_normal((n_data, dd))
    fine = dict(G=G, b=b)
    coarse = dict(G=G * (1.0 + 0.05 * rng.standard_normal(G.shape)), b=b + 0.05 * spread * rng.standard_normal(dd))
    arrays = {}
    for l, lv in enumerate([coarse, fine] if levels == 2 else [fine]):
        arrays.update({f"L{l}_G": lv["G"], f"L{l}_b": lv["b"], f"L{l}_data": data,
                       f"L{l}_noise_prec": np.eye(dd) / spread ** 2,
                       f"L{l}_prior_mean": truth + spread * rng.standard_normal(d),
                       f"L{l}_prior_prec": np.eye(d) / (10.0 * spread) ** 2})
    L = np.tril(0.3 * rng.standard_normal((d, d)), -1) + np.eye(d)
    if frozen is not None:
        L[frozen] = 0.0
    arrays["prop_L"] = prop_scale * spread * L
    meta = dict(model="linear", dim=d, levels=levels, J=J if levels == 2 else 1, eq="exact")
    return meta, arrays


def am_start(meta, arrays, nc, seed):
    """nc initial states near the level-0 prior mean (a spread of a tenth of the proposal's)."""
    m = np.asarray(arrays["L0_prior_mean"], dtype=np.float64)
    sd = np.abs(np.diag(np.asarray(arrays["prop_L"]))).max() * 0.1 if m.size else 0.0
    return m + sd * np.random.default_rng(seed).standard_normal((nc, m.size))


def _am_lv(levels, frozen=None):
    meta, arrays = bp.lv_problem(levels == 2)
    if frozen is not None:
        L = np.array(arrays["prop_L"], dtype=np.float64)
        L[frozen] = 0.0
        arrays = dict(arrays, prop_L=L)
    return meta, arrays


# The AM value sweep: each case runs at one and at two levels (J from the kwargs), so together they cover every
# generic_mh_kernel<D, DD, TWO_LEVEL> instance that carries AM; the d = 2 cases run the warp-specialised instance under
# Philox noise.  name: (am_problem kwargs, adaptive, chains, steps)
AM_SWEEP = {
    "2x2": (dict(d=2, dd=2, J=3, seed=1), dict(idle=0, collection=2, refresh=1, eps=1e-4), 64, 24),
    "2x4": (dict(d=2, dd=3, J=2, seed=2, offset=1e4, spread=1e-3), dict(idle=3, collection=4, refresh=3, eps=1e-9,
                                                                         scale=0.8), 64, 24),
    "2x8": (dict(d=2, dd=7, J=2, seed=3), dict(idle=0, collection=1, refresh=0, eps=1e-5), 64, 24),
    "3x2": (dict(d=3, dd=1, J=3, seed=4), dict(idle=1, collection=5, refresh=2, eps=1e-4), 64, 24),
    "4x4": (dict(d=4, dd=4, J=2, seed=5), dict(idle=0, collection=3, refresh=1, eps=1e-4, scale=0.5), 64, 24),
    "3x8": (dict(d=3, dd=6, J=2, seed=6), dict(idle=2, collection=0, refresh=3, eps=1e-4), 64, 24),
    "5x2": (dict(d=5, dd=2, J=2, seed=7, frozen=2), dict(idle=0, collection=2, refresh=1, eps=1e-4), 64, 24),
    "8x4": (dict(d=8, dd=3, J=2, seed=8), dict(idle=0, collection=2, refresh=1, eps=1e-4), 64, 24),
    "8x8": (dict(d=8, dd=8, J=3, seed=9, offset=1e4, spread=1e-3), dict(idle=4, collection=6, refresh=2, eps=1e-9),
            64, 24),
}

LAUNCHES = (1, 2, 5)        # the first launches of every forced case; the rest of the steps make the last one

# Forced-decision cases.  name: (problem builder, adaptive, chains, steps, all-rejected chains, forced first accepts)
# All-rejected chains get noise 1e3 times larger (every proposal lands far in the tail) and a pattern of rejections;
# with eps = 0 the moving chains accept their first proposals, so that the first refresh sees d + 1 distinct states.
AM_FORCED = {
    "d2_collect0_rejected": (lambda: am_problem(2, dd=1, seed=21), dict(idle=0, collection=0, refresh=1, eps=1e-3),
                             48, 30, 8, 0),
    "d3_two_level_refresh3": (lambda: am_problem(3, dd=3, levels=2, J=3, seed=22),
                              dict(idle=4, collection=5, refresh=3, eps=1e-4), 32, 16, 0, 0),
    "d5_frozen_eps0": (lambda: am_problem(5, dd=6, frozen=4, seed=23), dict(idle=2, collection=8, refresh=0, eps=0.0),
                       32, 24, 0, 0),
    "d4_offset_eps0_rejected": (lambda: am_problem(4, dd=2, offset=1e4, spread=1e-3, seed=24),
                                dict(idle=1, collection=12, refresh=1, eps=0.0, scale=0.5), 48, 30, 8, 8),
    "d8_two_level_frozen": (lambda: am_problem(8, dd=3, levels=2, J=2, frozen=2, seed=25),
                            dict(idle=0, collection=1, refresh=1, eps=1e-4, scale=0.3), 32, 20, 0, 0),
    "lv_two_level": (lambda: _am_lv(2), dict(idle=0, collection=2, refresh=3, eps=1e-6), 16, 8, 0, 0),
    "lv_one_level_frozen": (lambda: _am_lv(1, frozen=1), dict(idle=0, collection=3, refresh=1, eps=0.0), 16, 12, 0, 0),
    "gauss_three_level": (three_level_gauss, dict(idle=3, collection=4, refresh=2, eps=1e-5), 32, 8, 0, 0),
}


def am_launches(ns):
    return list(LAUNCHES) + [ns - sum(LAUNCHES)]


def am_forced_inputs(name, seed=0):
    """(meta, arrays, adaptive, theta0, z, pattern, launches) of an AM_FORCED case."""
    make, adaptive, nc, ns, n_rej, n_first = AM_FORCED[name]
    meta, arrays = make()
    if meta["model"] == "lv":
        th0 = bp.lv_initial_states(nc, seed=31 + seed)
    elif meta["model"] == "gauss":
        th0 = np.tile([0.5, 1.0], (nc, 1)) + 0.01 * np.random.default_rng(31 + seed).standard_normal((nc, 2))
    else:
        th0 = am_start(meta, arrays, nc, 31 + seed)
    z = schedule_noise(meta, nc, ns, 41 + seed)
    J = z.shape[2]
    pattern = R.random_pattern(nc, ns, J, 51 + seed)
    if n_rej:
        z[:n_rej] *= 1e3
        pattern["coarse"][:n_rej] = False
        pattern["fine"][:n_rej] = False
    if n_first:
        pattern["coarse"][n_rej:, :n_first] = True
        pattern["fine"][n_rej:, :n_first] = True
    return meta, arrays, adaptive, th0, z, pattern, am_launches(ns)
