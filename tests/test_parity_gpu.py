"""GPU: the CUDA path (through the C-ABI) against the committed reference fixtures and
against the C oracle on the same injected noise."""
import numpy as np
import pytest
import torch

from golden_io import load, rel_err, CHAIN_CASES, MLDA3_CASES, TEMPERED_CASES, AM_CASES
from support import LOGPOST_RTOL, ensemble

pytestmark = pytest.mark.gpu


def to_device_layout(a):
    """chain-major fixture arrays -> the ABI's [step, (J), (d), chain] layout."""
    z = np.ascontiguousarray(np.transpose(a["z"], (1, 2, 3, 0)))        # [ns, J, d, nc]
    u_c = np.ascontiguousarray(np.transpose(a["u_c"], (1, 2, 0)))       # [ns, J, nc]
    u_f = np.ascontiguousarray(np.transpose(a["u_f"], (1, 0)))          # [ns, nc]
    return dict(z=z, u_c=u_c, u_f=u_f)


def run_gpu(meta, a, **kw):
    nc, ns = a["u_f"].shape
    ens = ensemble(meta, a, nc, **kw)
    ens.set_state(a["theta0"])
    st0 = ens.state()
    out = ens.run(ns, samples=True, accepted=True, logpost=True, inject=to_device_layout(a))
    torch.cuda.synchronize()
    traj = np.concatenate([a["theta0"][:, None, :],
                           out["samples"].cpu().numpy().transpose(2, 0, 1)], axis=1)      # [nc, ns+1, d]
    lp = np.concatenate([st0["logpost"].cpu().numpy().T[:, None, :],
                         out["logpost"].cpu().numpy().transpose(2, 0, 1)], axis=1)        # [nc, ns+1, levels]
    acc = out["accepted"].cpu().numpy().T
    return ens, traj, lp, acc


@pytest.mark.parametrize("name", CHAIN_CASES + MLDA3_CASES + TEMPERED_CASES)
def test_trajectory_parity_with_reference_fixture(name):
    meta, a = load(name)
    ens, traj, lp, acc = run_gpu(meta, a)
    flips = int((acc != a["accepted"]).sum())
    assert flips == 0, f"{name}: {flips} accept decisions differ from the reference"
    assert rel_err(traj, a["traj"]).max() <= 1e-12, name
    assert rel_err(lp[:, :, 0], a["logpost_L0"]).max() <= LOGPOST_RTOL, name
    if meta["levels"] >= 2:
        assert rel_err(lp[:, :, 1], a["logpost_L1"]).max() <= LOGPOST_RTOL, name
    if meta["levels"] == 3:       # MLDA with two surrogates as the reference runs it (mlda.py:12-43,60-71,112-117)
        assert rel_err(lp[:, :, 2], a["logpost_L2"]).max() <= LOGPOST_RTOL, name
    st = ens.state()
    assert np.array_equal(st["n_accept"].cpu().numpy(), a["accepted"].sum(axis=1))
    if "welford_mean" in a:       # FullDiagnostics (chain/diagnostics.py:67-107)
        ns = a["u_f"].shape[1]
        d = meta["dim"]
        wm = st["w_mean"].cpu().numpy().T
        wv = np.stack([st["w_m2"][i, i].cpu().numpy() for i in range(d)], axis=1) / (ns - 1)
        np.testing.assert_allclose(wm, a["welford_mean"], rtol=1e-12)
        np.testing.assert_allclose(wv, a["welford_var"], rtol=1e-12)
    c = ens.counters()
    assert c["transitions"] == acc.size and c["accepted"] == int(a["accepted"].sum())


@pytest.mark.parametrize("name", AM_CASES)
def test_adaptive_metropolis_parity_with_reference_interface_fixture(name):
    """a14: fixtures written by the UNMODIFIED AdaptiveMRWProposal + MetropolisHastings.run (chain/adaptive.py:37-64)
    driving our concrete AdaptiveCovarianceMatrix; generic kernel (Gaussian target, linear two level) and the LV
    kernel (single level, and as the coarse proposal of two-level delayed acceptance).  Identical decisions,
    trajectory 1e-12 (dense factors: numpy's BLAS fuses `L @ z`, the kernels do not), and the adaptation state."""
    meta, a = load(name)
    ens, traj, lp, acc = run_gpu(meta, a, adaptive=meta["am"])
    assert int((acc != a["accepted"]).sum()) == 0, name
    assert rel_err(traj, a["traj"]).max() <= 1e-12, name
    assert rel_err(lp[:, :, 0], a["logpost_L0"]).max() <= LOGPOST_RTOL, name
    if meta["levels"] == 2:
        assert rel_err(lp[:, :, 1], a["logpost_L1"]).max() <= LOGPOST_RTOL, name
    st = ens.state()
    np.testing.assert_allclose(st["am_mean"].cpu().numpy().T, a["am_mean"], rtol=1e-12, atol=1e-14)
    np.testing.assert_allclose(st["am_m2"].permute(2, 0, 1).cpu().numpy(), a["am_m2"], rtol=1e-11, atol=1e-14)
    np.testing.assert_allclose(st["prop_L"].permute(2, 0, 1).cpu().numpy(), a["am_L"], rtol=1e-11, atol=1e-14)
    assert st["am_steps"] == a["u_f"].shape[1]
