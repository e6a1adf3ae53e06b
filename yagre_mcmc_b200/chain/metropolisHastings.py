"""Batched Metropolis-Hastings (reference: yagremcmc/chain/metropolisHastings.py:12-125).

Same surface -- run(chainLength, initialState, verbose), .chain.trajectory, .diagnostics,
.target, .clear() -- but `run` advances an ENSEMBLE of independent chains on the GPU:
  * trajectory[0] is the initial state and len(trajectory) == chainLength (:107-108,112);
  * initialState.coefficient is [d] (every chain starts there) or [nChains, d];
  * with torch.distributed initialised (one process per GPU) `nChains` is the GLOBAL count:
    each rank runs a contiguous range of chains keyed by their global id, so results do not
    depend on the number of GPUs; no data-path collective is issued.
"""
import numpy as np
import torch

from .._lib import YG_MAX_DIM
from ..ensemble import ChainEnsemble
from .chain import Chain, Trajectory
from .verbosity import VerbosityController


def _dist():
    import torch.distributed as dist
    if dist.is_available() and dist.is_initialized():
        return dist
    return None


from ..parallel import shard_range     # contiguous chain-id range of a rank: [r n / g, (r+1) n / g)


class MetropolisHastings:

    def __init__(self, targetDensity, proposalMethod, diagnostics, lowered, nChains=1, seed=0,
                 device=None, adaptive=None, thin=1, storeTrajectory=True, launch=None, aem=None):
        self._tgtDensity = targetDensity
        self._proposalMethod = proposalMethod
        self._diagnostics = diagnostics
        self._chain = Chain()
        self._verbosityController = VerbosityController()
        self._lowered = lowered
        self._nGlobal = int(nChains)
        self._seed = int(seed)
        self._thin = int(thin)
        self._store = bool(storeTrajectory)
        dist = _dist()
        self._rank, self._world = (dist.get_rank(), dist.get_world_size()) if dist else (0, 1)
        lo, hi = shard_range(self._nGlobal, self._rank, self._world)
        if hi <= lo:
            raise ValueError(f"rank {self._rank} of {self._world} received no chains (nChains={self._nGlobal})")
        self._offset, self._nLocal = lo, hi - lo
        if device is None:
            device = torch.cuda.current_device() if torch.cuda.is_available() else 0
        self._ensemble = ChainEnsemble(lowered, self._nLocal, device=device, seed=self._seed,
                                       chain_offset=self._offset, adaptive=adaptive, aem=aem,
                                       welford=self._wants_moments(diagnostics), **(launch or {}))
        self._last = None
        self._accepted = 0              # accepted transitions (all local chains) since the device counters were reset
        self._lastRun = None            # (accepted, transitions per chain) of the last run()
        self._ran = False               # a run() has set the device state at least once
        self._diagnosticsCleared = True  # clear() was called since the last run(): restart the device accumulators

    @staticmethod
    def _wants_moments(diagnostics):
        """FullDiagnostics keeps Welford moments (chain/diagnostics.py:67-107); the builders' default
        AcceptanceRateDiagnostics does not (chain/builder.py:14-16).  Only the tensor-path kernel saves work by it:
        the other kernels keep the moments for free, and pooled() / pool_proposal_covariance() rely on them there."""
        from .diagnostics import FullDiagnostics
        return isinstance(diagnostics, FullDiagnostics)

    # ---- reference surface ------------------------------------------------------------------
    @property
    def chain(self):
        return self._chain

    @property
    def target(self):
        return self._tgtDensity

    @property
    def diagnostics(self):
        return self._diagnostics

    @property
    def ensemble(self):
        return self._ensemble

    @property
    def nChains(self):
        return self._nGlobal

    @property
    def localChainRange(self):
        return self._offset, self._offset + self._nLocal

    def clear(self):
        """reference chain/metropolisHastings.py:122-125: resets diagnostics and trajectory.  The device
        accumulators (accept counters, Welford moments) restart with the next run(); the state of an adaptive
        proposal / adaptive error model lives as long as the object, as in the reference."""
        self._diagnostics.reset()
        self._chain.clear()
        self._diagnosticsCleared = True

    def run(self, chainLength, initialState, verbose=True):
        chainLength = int(chainLength)
        if chainLength < 1:
            raise ValueError("chainLength must be >= 1")
        coef = np.asarray(initialState.coefficient, dtype=np.float64)
        d = self._lowered.dim
        if coef.ndim == 1:
            if coef.size != d:
                raise ValueError(f"initial state has dimension {coef.size}, chain has {d}")
            theta0 = np.broadcast_to(coef.reshape(1, d), (self._nLocal, d))
        elif coef.shape == (self._nGlobal, d):
            theta0 = coef[self._offset:self._offset + self._nLocal]
        elif coef.shape == (self._nLocal, d):
            theta0 = coef
        else:
            raise ValueError(f"initial state must be [{d}] or [{self._nGlobal}, {d}], got {coef.shape}")
        ens = self._ensemble
        # Like the reference, a further run() restarts only the chain: diagnostics accumulate until clear()
        # (metropolisHastings.py:107-108,122-125), adaptation state persists, and the noise stream keeps
        # advancing (numpy's global generator there, the Philox step index here) -- two runs from the same
        # state are different realisations.
        keep = self._ran and not self._diagnosticsCleared
        ens.set_state(np.ascontiguousarray(theta0), keep_diagnostics=keep, keep_adaptation=self._ran)
        accepted0 = self._accepted if keep else 0
        self._ran, self._diagnosticsCleared = True, False
        self._verbosityController.on = bool(verbose)
        nTrans = chainLength - 1
        thin = self._thin
        pieces = []
        if self._store:
            pieces.append(torch.from_numpy(np.array(theta0.T, dtype=np.float64)).to(ens.device).unsqueeze(0))
        interval = self._verbosityController.print_interval(chainLength) if verbose else max(nTrans, 1)
        interval = max(thin, (interval // thin) * thin)
        done = 0
        while done < nTrans:
            n = min(interval, nTrans - done)
            n_store = (n // thin) * thin
            if self._store and n_store:
                pieces.append(ens.run(n_store, thin=thin, samples=True)['samples'])
                if n > n_store:
                    ens.run(n - n_store, samples=False)
            else:
                ens.run(n, samples=False)
            done += n
            self._update_diagnostics()
            if verbose and done < nTrans:
                self._verbosityController.report(done, self._diagnostics)
        if nTrans == 0:
            self._update_diagnostics()
        if self._store:
            traj = torch.cat(pieces, dim=0) if len(pieces) > 1 else pieces[0]
            self._chain.set(Trajectory(traj, squeeze=(self._nGlobal == 1)))
            if d > YG_MAX_DIM:          # the acceptance of the run pooled() pools (_stored_samples)
                self._accepted = ens.counters()['accepted']
                self._lastRun = (self._accepted - accepted0, nTrans)
        return self

    # ---- internals ----------------------------------------------------------------------------
    def _update_diagnostics(self):
        ens = self._ensemble
        st = ens.state()
        d = self._lowered.dim
        w_m2 = st['w_m2']
        stats = dict(n_accept=st['n_accept'].cpu().numpy(), transitions=st['welford_n'],
                     welford_n=st['welford_n'], w_mean=st['w_mean'].t().cpu().numpy(),
                     w_m2_diag=(torch.stack([w_m2[i, i] for i in range(d)], dim=1) if w_m2.dim() == 3
                                else w_m2.t()).cpu().numpy(),
                     squeeze=(self._nGlobal == 1))
        self._last = st
        self._diagnostics.process_ensemble(stats)

    def _stored_samples(self):
        """(samples [length, d, nLocal], accepted, transitions per chain) of the last run(): the pooled path for
        d > YG_MAX_DIM, where the device keeps no full second moment per chain."""
        if not self._store or self._lastRun is None or not isinstance(self._chain.trajectory, Trajectory):
            raise NotImplementedError(
                f"pooled statistics at dim > {YG_MAX_DIM} are computed from the stored trajectory of the last run(): "
                "build the chain with storeTrajectory = True (and a thin that keeps it affordable), then run()")
        return (self._chain.trajectory.device_tensor,) + self._lastRun

    def pooled(self):
        """Pooled moments and R-hat over ALL chains (all ranks): see yagre_mcmc_b200.parallel.

        dim <= 8: from the chains' Welford moments, i.e. every pre-transition state since clear().  dim > 8 (the
        tensor path keeps a diagonal second moment only): from the trajectory of the LAST run() as stored, i.e. its
        initial state and every thin-th state after it; the acceptance rate is that run's.  Needs storeTrajectory."""
        if self._lowered.dim > YG_MAX_DIM:
            from ..parallel import pooled_diagnostics_from_samples
            return pooled_diagnostics_from_samples(*self._stored_samples())
        from ..parallel import pooled_diagnostics
        return pooled_diagnostics(self._ensemble)

    def pool_proposal_covariance(self, scale=None, eps=1e-8):
        """Optional pooled proposal covariance: replaces the proposal covariance of every chain (all ranks) by
        scale * (pooled covariance + eps I), scale = 2.4^2 / d by default.  The covariance is pooled as pooled()
        does: since clear() for dim <= 8, over the stored trajectory of the last run() for dim > 8 -- where a handle
        built with a diagonal proposal factor switches to the dense kernel instance.  The idiom mirrors the
        reference's burn-in restart (example_inference_linearModel_twoLevel.py:228,236): run a burn-in, pool, run
        again from chain.trajectory[-1].  Returns the pooled moments with the new factor under 'prop_L'."""
        if self._lowered.dim > YG_MAX_DIM:
            from ..parallel import pooled_proposal_covariance_from_samples
            return pooled_proposal_covariance_from_samples(self._ensemble, *self._stored_samples(), scale, eps)
        from ..parallel import pooled_proposal_covariance
        return pooled_proposal_covariance(self._ensemble, scale, eps)
