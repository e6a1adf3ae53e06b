"""CPU: pooled statistics from a stored sample buffer (yg_pooled_samples, parallel.pooled_diagnostics_from_samples).

The argument checks of the C-ABI run before any CUDA call, so they are exercised here through the built library.  The
long-double reference of the statistics vector (tests/pooled_samples_reference.py) is checked against a per-chain
restatement, its bounds against the kernel's formulation in double and against raw moments.  Two gloo ranks holding the
two halves of the chains must pool to the single-rank answer; the device kernel is covered by the -m gpu tests."""
import ctypes as C
import os

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

import pooled_samples_reference as psr
from support import free_port
from yagre_mcmc_b200 import _lib
from yagre_mcmc_b200.parallel import moments_from_stats, shard_range


def _call(lib, samples=1, ns=3, d=4, nc=5, ws=1, ws_len=None, out=1):
    if ws_len is None:
        ws_len = lib.yg_pooled_samples_workspace_len(d, nc)
    return lib.yg_pooled_samples(C.c_void_p(samples), ns, d, nc, C.c_void_p(ws), ws_len, C.c_void_p(out), None)


def test_arguments_are_refused_before_any_cuda_call():
    lib = _lib.load()
    assert _call(lib, samples=0) == _lib.YG_ERR_INVALID
    assert _call(lib, ws=0) == _lib.YG_ERR_INVALID
    assert _call(lib, out=0) == _lib.YG_ERR_INVALID
    assert _call(lib, ns=0) == _lib.YG_ERR_INVALID
    assert _call(lib, nc=0, ws_len=10 ** 6) == _lib.YG_ERR_INVALID
    assert _call(lib, d=0, ws_len=10 ** 6) == _lib.YG_ERR_INVALID
    assert _call(lib, ws_len=lib.yg_pooled_samples_workspace_len(4, 5) - 1) == _lib.YG_ERR_INVALID
    assert "workspace" in _lib.last_error()
    assert _call(lib, d=_lib.YG_BIG_MAX_DIM + 1) == _lib.YG_ERR_UNSUPPORTED
    with pytest.raises(NotImplementedError):
        _lib.check(_call(lib, d=_lib.YG_BIG_MAX_DIM + 1))


def test_workspace_length():
    lib = _lib.load()
    assert lib.yg_pooled_samples_workspace_len(0, 10) == 0 and lib.yg_pooled_samples_workspace_len(3, 0) == 0
    for d in (1, 8, 9, 64):
        plen = lib.yg_pooled_len(d)
        for nc in (1, 16, 17, 1000, 65536, 10 ** 7):
            n = lib.yg_pooled_samples_workspace_len(d, nc)
            parts = min(4 * 148, -(-nc // 16))                # per-CTA partial vectors + one mean per chain
            assert n == parts * plen + d * nc, (d, nc, n)


def _restated(x):
    """Per chain, straight from the definition (numpy mean / centred products): parallel.py's layout."""
    ns, d, nc = x.shape
    xc = x.transpose(2, 0, 1)                                  # [nc, ns, d]
    mean = xc.mean(axis=1)
    dev = xc - mean[:, None]
    m2 = np.einsum('cti,ctj->cij', dev, dev)
    var = xc.var(axis=1, ddof=1) if ns > 1 else np.zeros((nc, d))
    return np.concatenate([[nc, ns, 0.0], mean.sum(0), (mean.T @ mean).ravel(), m2.sum(0).ravel(), var.sum(0)])


@pytest.mark.parametrize("ns,d,nc", [(1, 3, 5), (2, 1, 1), (5, 9, 3), (40, 17, 9), (7, 64, 2)])
def test_reference_is_the_restated_vector_and_the_kernel_formulation_meets_its_bound(ns, d, nc):
    rng = np.random.default_rng(ns * 1000 + d * 10 + nc)
    x = rng.standard_normal((ns, d, nc)) * rng.uniform(0.1, 3.0, (1, d, 1)) + rng.standard_normal((1, d, nc))
    ref, tol = psr.reference(x)
    want = _restated(x)
    scale = np.concatenate([[1.0, 1.0, 1.0], np.abs(want[3:])]) + 1.0
    np.testing.assert_array_less(np.abs(ref.astype(np.float64) - want), 1e-12 * scale)
    assert psr.check_vector(psr.kernel_formulation(x), x) <= 1.0
    assert np.all(tol[3:3 + d + d * d] > 0.0)
    assert np.all(tol[3 + d + d * d:] > 0.0) == (ns > 1)     # M2 and variances of single samples: exact zeros


def test_raw_moments_fail_the_bound_on_offset_data():
    """A common offset of 1e4: the shifted formulation stays inside the M2 bound, raw moments are far outside it."""
    rng = np.random.default_rng(5)
    ns, d, nc = 40, 5, 1000
    x = 1e4 + rng.standard_normal((ns, d, nc))
    assert psr.check_vector(psr.kernel_formulation(x), x, "shifted") <= 1.0
    ref, tol = psr.reference(x)
    raw = psr.raw_formulation(x)
    o = 3 + d + d * d
    ratio = (np.abs(raw.astype(np.longdouble) - ref).astype(np.float64)[o:o + d * d] / tol[o:o + d * d]).max()
    assert ratio > 100.0, ratio


def _samples(seed=11, ns=30, d=5, nc=40):
    rng = np.random.default_rng(seed)
    return (rng.standard_normal((ns, d, nc)) * np.linspace(0.5, 2.0, d)[None, :, None]
            + 0.3 * rng.standard_normal((1, d, nc)) + 2.0)


class _RankEnsemble:
    """Records the factor pooled_proposal_covariance_from_samples installs."""

    def __init__(self):
        self.L = None

    def rebuild_proposal_factor(self, L):
        self.L = np.array(L)


def _worker(rank, world, port, q):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        from yagre_mcmc_b200 import ensemble, parallel
        # the device kernel is replaced by the long-double reference, rounded to double
        ensemble.pooled_sample_stats = lambda s: torch.from_numpy(psr.reference(s.numpy())[0].astype(np.float64))
        x = _samples()
        lo, hi = shard_range(x.shape[2], rank, world)
        acc = 7 * (hi - lo) + 3 * rank                         # accepted transitions of this rank's chains
        out = parallel.pooled_diagnostics_from_samples(torch.from_numpy(x[:, :, lo:hi].copy()), acc, 50)
        ens = _RankEnsemble()
        pooled = parallel.pooled_proposal_covariance_from_samples(ens, torch.from_numpy(x[:, :, lo:hi].copy()), acc,
                                                                  50, eps=1e-6)
        out["prop_L"], out["prop_L_set"] = pooled["prop_L"], ens.L
        q.put((rank, lo, hi, out))
    finally:
        dist.destroy_process_group()


@pytest.mark.timeout(180)
def test_two_rank_pooling_from_samples_equals_single_rank():
    world, port = 2, free_port()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_worker, args=(r, world, port, q)) for r in range(world)]
    for p in procs:
        p.start()
    res = sorted([q.get(timeout=150) for _ in range(world)], key=lambda t: t[0])
    for p in procs:
        p.join(30)
        assert p.exitcode == 0
    x = _samples()
    ns, d, nc = x.shape
    assert res[0][1] == 0 and res[0][2] == res[1][1] and res[1][2] == nc
    single = psr.reference(x)[0].astype(np.float64)
    single[2] = (7 * nc + 3) * ns / 50
    want = moments_from_stats(single, d)
    mu, cov = psr.pooled_moments(x)
    for _, _, _, out in res:
        assert out["n_chains"] == nc and out["samples_per_chain"] == ns
        np.testing.assert_allclose(out["mean"], want["mean"], rtol=1e-13)
        np.testing.assert_allclose(out["covariance"], want["covariance"], rtol=1e-12)
        np.testing.assert_allclose(out["rhat"], want["rhat"], rtol=1e-12)
        assert abs(out["acceptance_rate"] - (7 * nc + 3) / (50 * nc)) < 1e-15
        np.testing.assert_allclose(out["mean"], mu, rtol=1e-12)
        np.testing.assert_allclose(out["covariance"], cov, rtol=1e-10)
        L = np.linalg.cholesky(2.4 * 2.4 / d * (cov + 1e-6 * np.eye(d)))
        np.testing.assert_allclose(out["prop_L_set"], L, rtol=1e-9)
    np.testing.assert_array_equal(res[0][3]["prop_L_set"], res[1][3]["prop_L_set"])
