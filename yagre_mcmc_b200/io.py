"""Trajectory dump and checkpoint / resume.

The reference has no persistence; its only restart idiom is "start a new run from
trajectory[-1]" (example_inference_linearModel_twoLevel.py:228,236), which loses the
diagnostics, the adaptive state and the RNG position.  Here:

  save_trajectory / load_trajectory   one .npy file, float64, shape [chainLength, d, nChains] (the
      device layout: chain index fastest) plus a small JSON side-car (thin, chain range, problem
      summary); `as_reference_layout` gives [chainLength, nChains, d].
  save_checkpoint / load_checkpoint   every per-chain array of yg_state (theta, log-posteriors,
      accept counts, Welford moments, adaptive-Metropolis and error-model state) plus the step
      index and the Welford count in one .npz: a resumed run continues BIT-EXACTLY, because the
      Philox streams are keyed on (seed, global chain id, step index) and nothing else.
"""
import json
import os

import numpy as np
import torch

FORMAT_VERSION = 1


def save_trajectory(path, samples, thin=1, chain_offset=0, meta=None):
    """samples: device or host tensor / array [n_out, d, n_chains]."""
    a = samples.detach().cpu().numpy() if torch.is_tensor(samples) else np.asarray(samples, dtype=np.float64)
    if a.ndim != 3 or a.dtype != np.float64:
        raise ValueError("trajectory must be float64 [length, d, n_chains]")
    np.save(path, a, allow_pickle=False)
    side = dict(format='yagre_mcmc_b200.trajectory', version=FORMAT_VERSION, layout='[length, d, n_chains]',
                length=int(a.shape[0]), dim=int(a.shape[1]), n_chains=int(a.shape[2]), thin=int(thin),
                chain_offset=int(chain_offset), meta=meta or {})
    base = path if path.endswith('.npy') else path + '.npy'
    with open(base + '.json', 'w') as f:
        json.dump(side, f, indent=1)
    return base


def load_trajectory(path, mmap=False):
    base = path if path.endswith('.npy') else path + '.npy'
    a = np.load(base, mmap_mode='r' if mmap else None, allow_pickle=False)
    side = {}
    if os.path.exists(base + '.json'):
        with open(base + '.json') as f:
            side = json.load(f)
        if side.get('version', FORMAT_VERSION) > FORMAT_VERSION:
            raise ValueError(f"trajectory file version {side['version']} is newer than this reader ({FORMAT_VERSION})")
    return a, side


def as_reference_layout(samples):
    """[length, d, n_chains] -> [length, n_chains, d] (what reference scripts index)."""
    return np.transpose(np.asarray(samples), (0, 2, 1))


def save_checkpoint(path, ensemble, extra=None):
    """Writes the complete per-chain state of a ChainEnsemble (this rank's chains)."""
    st = ensemble.state()
    arrays = {k: st[k].cpu().numpy() for k in ensemble.layout()}
    head = dict(format='yagre_mcmc_b200.checkpoint', version=FORMAT_VERSION, step_index=int(st['step_index']),
                welford_n=int(st['welford_n']), am_steps=int(st.get('am_steps', 0)), n_chains=int(ensemble.n_chains), dim=int(ensemble.dim),
                levels=int(ensemble.levels), seed=int(ensemble.cfg.seed), chain_offset=int(ensemble.cfg.chain_offset),
                model=ensemble.problem.model, adaptive=int(ensemble.cfg.adaptive), aem=int(ensemble.cfg.aem),
                extra=extra or {})
    np.savez(path, header=json.dumps(head), **arrays)
    return path if path.endswith('.npz') else path + '.npz'


def load_checkpoint(path, ensemble):
    """Restores a checkpoint into an ensemble built for the same problem, chain range and seed."""
    base = path if path.endswith('.npz') else path + '.npz'
    f = np.load(base, allow_pickle=False)
    head = json.loads(str(f['header']))
    if head.get('format') != 'yagre_mcmc_b200.checkpoint' or head.get('version', 0) > FORMAT_VERSION:
        raise ValueError(f"{base} is not a readable yagre_mcmc_b200 checkpoint")
    for key, have in (('n_chains', ensemble.n_chains), ('dim', ensemble.dim), ('levels', ensemble.levels),
                      ('seed', int(ensemble.cfg.seed)), ('chain_offset', int(ensemble.cfg.chain_offset)),
                      ('model', ensemble.problem.model), ('adaptive', int(ensemble.cfg.adaptive)),
                      ('aem', int(ensemble.cfg.aem))):
        if head[key] != have:
            raise ValueError(f"checkpoint {key}={head[key]!r} does not match the ensemble ({have!r}): "
                             "a resumed run would not continue the saved chains")
    st = {k: torch.from_numpy(np.ascontiguousarray(f[k])) for k in ensemble.layout() if k in f.files}
    st['step_index'], st['welford_n'] = head['step_index'], head['welford_n']
    st['am_steps'] = head.get('am_steps', head['welford_n'])
    ensemble.load_state(st)
    return head
