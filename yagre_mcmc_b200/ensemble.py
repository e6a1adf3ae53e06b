"""Host-side handle over libyagre_b200: an ensemble of independent chains on one GPU.

PyTorch is plumbing only (device memory, streams); every computation happens in
the hand-written sm_100a kernels behind the C-ABI.  Layout on the device is
struct-of-arrays with the chain index fastest (theta[d, n], samples[n_out, d, n]).
"""
import copy
import ctypes as C

import numpy as np
import torch

from . import _lib
from ._lib import (YgConfig, YgProblem, YgNoise, YgOutputs, YgState, check,
                   MODEL_GAUSS, MODEL_LINEAR, MODEL_LV, EQ_EXACT, EQ_ISCLOSE,
                   NOISE_PHILOX, NOISE_INJECT, NOISE_RECORD)

_MODEL = {'gauss': MODEL_GAUSS, 'linear': MODEL_LINEAR, 'lv': MODEL_LV}
_EQ = {'exact': EQ_EXACT, 'isclose': EQ_ISCLOSE}
_dp = C.POINTER(C.c_double)


def _f64(a):
    return np.ascontiguousarray(np.asarray(a, dtype=np.float64))


def state_layout(n, d, levels, adaptive, aem_data_dim):
    """{name: (shape, torch dtype)} of the per-chain state (yg_state) of n chains; aem_data_dim 0: no error model."""
    f64, i64 = torch.float64, torch.int64
    lay = dict(theta=((d, n), f64), logpost=((levels, n), f64), n_accept=((n,), i64), w_mean=((d, n), f64),
               w_m2=((d, d, n) if d <= _lib.YG_MAX_DIM else (d, n), f64))        # large linear model: diagonal only
    if adaptive:
        lay.update(prop_L=((d, d, n), f64), am_mean=((d, n), f64), am_m2=((d, d, n), f64))
    if aem_data_dim:
        lay.update(aem_n=((n,), i64), aem_mean=((aem_data_dim, n), f64), aem_m2=((aem_data_dim, n), f64),
                   aem_cache=((3 * (d + 1) + 1, n), f64))
    return lay


def check_state(r, layout):
    """ValueError unless r has theta and logpost and each array the layout names is a tensor of its shape and dtype."""
    if 'theta' not in r or 'logpost' not in r:
        raise ValueError("a state needs at least theta and logpost")
    for k, (shape, dtype) in layout.items():
        v = r.get(k)
        if v is not None and (not torch.is_tensor(v) or tuple(v.shape) != shape or v.dtype != dtype):
            raise ValueError(f"state {k!r} must be a {dtype} tensor of shape {shape}, got {type(v).__name__} "
                             f"{tuple(getattr(v, 'shape', ()))} {getattr(v, 'dtype', '')}")


class LoweredProblem:
    """The plain-array form of a (hierarchy of) Bayesian model(s) + proposal, i.e.
    what ChainBuilder.build_method() (reference chain/builder.py:72-83) boils down to.

    meta:   model ('gauss'|'linear'|'lv'), dim, levels (1|2|3), J, eq ('exact'|'isclose'),
            proposal ('mrw'|'pcn') and pcn_step for pCN (prop_L is then the prior's factor and the
            level's prior_prec is zero: the pCN target is the likelihood alone, pcn.py:52-57)
    arrays: prop_L[d,d] and per level l: L{l}_g_mean/g_prec/g_logconst (gauss),
            L{l}_data/noise_prec/prior_mean/prior_prec (+ L{l}_G/b | L{l}_design/lv=[alpha,gamma,T,N]),
            optionally L{l}_tempering (TemperedUnnormalisedPosterior, chain/target.py:25-43)
    levels == 3 is MLDA with two surrogates as the reference runs it (mlda.py:12-43,60-71,112-117): level 0
    drives the MRW sub-chain of J = subChainLengths[1] steps, level 1 (the finest surrogate) screens, level 2
    is the target.
    """

    def __init__(self, meta, arrays):
        self.model = meta['model']
        self.dim = int(meta['dim'])
        self.levels = int(meta['levels'])
        self.J = int(meta.get('J', 1))
        self.eq = meta.get('eq', 'exact')
        self.proposal = meta.get('proposal', 'mrw')
        self.pcn_step = float(meta.get('pcn_step', 0.0))
        if self.proposal not in ('mrw', 'pcn'):
            raise NotImplementedError(f"proposal {self.proposal!r} has no device implementation")
        if self.model not in _MODEL:
            raise NotImplementedError(
                f"model {self.model!r} has no device implementation; the backend accepts Gaussian targets, "
                "linear models and the Lotka-Volterra RK4 model only (no CPU fallback)")
        self.arrays = {k: _f64(v) for k, v in arrays.items()
                       if k in ('prop_L', 'pcn_mean') or k[:3] in ('L0_', 'L1_', 'L2_')}
        if 'prop_L' not in self.arrays:
            raise ValueError("Proposal Covariance not set")

    def c_struct(self):
        pb = YgProblem()
        a = self.arrays
        pb.prop_L = a['prop_L'].ctypes.data_as(_dp)
        if self.proposal == 'pcn':
            pb.proposal, pb.pcn_step = _lib.PROPOSAL_PCN, self.pcn_step
            if 'pcn_mean' in a:
                pb.pcn_mean = a['pcn_mean'].ctypes.data_as(_dp)
        for l in range(self.levels):
            lv = pb.level[l]
            pre = f"L{l}_"
            for f in ("g_mean", "g_prec", "data", "noise_prec", "prior_mean", "prior_prec", "G", "b", "design"):
                if pre + f in a:
                    setattr(lv, f, a[pre + f].ctypes.data_as(_dp))
            if pre + "g_logconst" in a:
                lv.g_logconst = float(np.asarray(a[pre + "g_logconst"]).reshape(-1)[0])
            if pre + "data" in a:
                lv.n_data, lv.data_dim = (int(x) for x in a[pre + "data"].shape)
            if pre + "lv" in a:
                p = a[pre + "lv"]
                lv.alpha, lv.gamma, lv.T, lv.rk4_steps = float(p[0]), float(p[1]), float(p[2]), int(p[3])
            if pre + "tempering" in a:
                lv.tempered, lv.tempering = 1, float(np.asarray(a[pre + "tempering"]).reshape(-1)[0])
        return pb


class ChainEnsemble:
    """n_chains independent chains of one problem on one device."""

    def __init__(self, problem, n_chains, device=0, seed=0, chain_offset=0,
                 adaptive=None, blocks_per_sm=0, threads_per_block=0, rk4_segment=0, aem=None, welford=True,
                 early_reject=True):
        self.lib = _lib.load()
        if not torch.cuda.is_available():
            raise _lib.BackendUnavailable("no CUDA device visible: the batched-chain backend has no CPU fallback")
        self.problem = problem
        self.n_chains = int(n_chains)
        self.dim = problem.dim
        self.levels = problem.levels
        self.J = problem.J if problem.levels >= 2 else 1
        self.device = torch.device('cuda', int(device))
        cfg = YgConfig()
        cfg.abi_version = _lib.YG_ABI_VERSION
        cfg.device = int(device)
        cfg.n_chains = self.n_chains
        cfg.chain_offset = int(chain_offset)
        cfg.seed = int(seed) & 0xFFFFFFFFFFFFFFFF
        cfg.model = _MODEL[problem.model]
        cfg.dim = problem.dim
        cfg.n_levels = problem.levels
        cfg.sub_chain_length = self.J
        cfg.eq_mode = _EQ[problem.eq]
        cfg.blocks_per_sm = int(blocks_per_sm)
        cfg.threads_per_block = int(threads_per_block)
        cfg.rk4_segment = int(rk4_segment)
        # welford=False: AcceptanceRateDiagnostics only (the reference builders' default, chain/builder.py:14-16);
        # honoured by the tensor-path kernel, whose Welford moments live in L2
        cfg.acceptance_only = 0 if welford else 1
        # early_reject=False: the LV kernel integrates every design point of every proposal (same results)
        cfg.early_reject_off = 0 if early_reject else 1
        self.aem = None
        if aem:             # adaptive error model: dict(min_data=..., heuristic=...)
            cfg.aem = 1
            cfg.aem_min_data = int(aem['min_data'])
            cfg.aem_heuristic = int(bool(aem.get('heuristic', False)))
            self.aem = dict(aem)
        if adaptive:
            cfg.adaptive = 1
            cfg.am_idle_steps = int(adaptive.get('idle', 0))
            cfg.am_collection_steps = int(adaptive.get('collection', 100))
            cfg.am_refresh = int(adaptive.get('refresh', 1))
            cfg.am_eps = float(adaptive.get('eps', 1e-4))
            cfg.am_scale = float(adaptive.get('scale', 0.0))
        self.cfg = cfg
        self._h = C.c_void_p()
        check(self.lib.yg_create(C.byref(cfg), C.byref(self._h)))
        pb = problem.c_struct()
        check(self.lib.yg_set_problem(self._h, C.byref(pb)))

    # ------------------------------------------------------------------ plumbing
    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def _empty(self, *shape, dtype=torch.float64):
        return torch.empty(shape, dtype=dtype, device=self.device)

    def close(self):
        if getattr(self, "_h", None) is not None and self._h.value:
            self.lib.yg_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ------------------------------------------------------------------ state
    def set_state(self, theta0, keep_diagnostics=False, keep_adaptation=False, step_index=None):
        """theta0: [n_chains, d] (or [d], broadcast) host or device array.

        Resets the diagnostics (accept counters, Welford moments, evaluation counters) and the adaptation state
        (adaptive-Metropolis moments / factors, adaptive error model) unless told to keep them -- the reference
        keeps both across run() calls (diagnostics until clear()).  The Philox stream position is NOT reset: like
        numpy's generator in the reference it keeps advancing, so a second run from the same state sees fresh
        noise; pass step_index to reposition it (yg_seek)."""
        t = theta0.to(torch.float64) if torch.is_tensor(theta0) else torch.from_numpy(np.array(theta0, dtype=np.float64))
        if t.dim() == 1:
            t = t.reshape(1, -1).expand(self.n_chains, -1)
        if tuple(t.shape) != (self.n_chains, self.dim):
            raise ValueError(f"initial state must be [{self.n_chains}, {self.dim}], got {tuple(t.shape)}")
        soa = t.to(self.device).t().contiguous()            # [d, n]
        flags = (_lib.KEEP_DIAGNOSTICS if keep_diagnostics else 0) | (_lib.KEEP_ADAPTATION if keep_adaptation else 0)
        with torch.cuda.device(self.device):
            check(self.lib.yg_set_state(self._h, C.c_void_p(soa.data_ptr()), flags, self._stream()))
        if step_index is not None:
            self.seek(step_index)
        return self

    def seek(self, step_index):
        """Positions the Philox stream: the next run draws the noise of steps step_index, step_index + 1, ..."""
        check(self.lib.yg_seek(self._h, int(step_index)))
        return self

    def set_proposal_factor(self, L):
        """Replaces the proposal factor (lower triangular [d, d], proposal covariance = L L') for the following
        runs; see parallel.pooled_proposal_covariance."""
        Lh = np.ascontiguousarray(np.asarray(L, dtype=np.float64))
        if Lh.shape != (self.dim, self.dim):
            raise ValueError(f"proposal factor must be [{self.dim}, {self.dim}], got {Lh.shape}")
        with torch.cuda.device(self.device):
            check(self.lib.yg_set_proposal_factor(self._h, Lh.ctypes.data_as(C.c_void_p), self._stream()))
        return self

    def rebuild_proposal_factor(self, L):
        """Replaces the proposal factor by re-issuing yg_set_problem with the problem's prop_L replaced by L (lower
        triangular [d, d], positive diagonal).  Unlike set_proposal_factor it may switch the kind of factor: a
        tensor-path handle built with a diagonal factor takes a dense one and runs the dense kernel instance from then
        on.  The chains' state is kept (the target does not change).  Refused for pCN, whose factor is the prior's
        (pcn.py:23-35)."""
        if self.problem.proposal == 'pcn':
            raise NotImplementedError("the proposal factor of a pCN chain is the prior's (pcn.py:23-35) and cannot be "
                                      "replaced")
        Lh = _f64(L)
        if Lh.shape != (self.dim, self.dim):
            raise ValueError(f"proposal factor must be [{self.dim}, {self.dim}], got {Lh.shape}")
        if not np.all(np.isfinite(Lh)) or np.any(np.triu(Lh, 1) != 0.0) or not np.all(np.diag(Lh) > 0.0):
            raise ValueError("proposal factor must be finite, lower triangular with a positive diagonal")
        problem = copy.copy(self.problem)
        problem.arrays = dict(self.problem.arrays, prop_L=Lh)
        with torch.cuda.device(self.device):
            check(self.lib.yg_set_problem(self._h, C.byref(problem.c_struct())))
        self.problem = problem
        return self

    def run(self, n_steps, thin=1, samples=True, accepted=False, logpost=False, inject=None, record=False,
            samples_out=None):
        """Runs n_steps transitions of every chain.

        inject: dict(z=[n_steps,J,d,n], u_c=[n_steps,J,n], u_f=[n_steps,n]) device or host arrays.
        record: Philox noise, and the noise actually used is returned in the same layout.
        samples_out: optional preallocated device tensor [n_steps/thin, d, n] to write the samples into
                (no allocation in the call; the caller owns its lifetime across streams).
        Returns a dict of device tensors: samples [n_steps/thin, d, n], accepted [n_steps, n] uint8,
        logpost [n_steps/thin, levels, n].
        """
        n, d, J = self.n_chains, self.dim, self.J
        n_steps = int(n_steps)
        out = YgOutputs()
        res = {}
        n_out = n_steps // thin
        if samples_out is not None:
            if (tuple(samples_out.shape) != (n_out, d, n) or samples_out.dtype != torch.float64
                    or not samples_out.is_contiguous() or samples_out.device != self.device):
                raise ValueError(f"samples_out must be a contiguous float64 device tensor of shape {(n_out, d, n)}")
            res['samples'] = samples_out
            out.samples_dev = samples_out.data_ptr()
        elif samples:
            res['samples'] = self._empty(n_out, d, n)
            out.samples_dev = res['samples'].data_ptr()
        if accepted:
            res['accepted'] = self._empty(n_steps, n, dtype=torch.uint8)
            out.accepted_dev = res['accepted'].data_ptr()
        if logpost:
            res['logpost'] = self._empty(n_out, self.levels, n)
            out.logpost_dev = res['logpost'].data_ptr()
        noise = YgNoise()
        noise.mode = NOISE_PHILOX
        keep = []
        if inject is not None:
            noise.mode = NOISE_INJECT
            z = torch.as_tensor(inject['z'], dtype=torch.float64).to(self.device).contiguous()
            u_f = torch.as_tensor(inject['u_f'], dtype=torch.float64).to(self.device).contiguous()
            assert tuple(z.shape) == (n_steps, J, d, n), (tuple(z.shape), (n_steps, J, d, n))
            assert tuple(u_f.shape) == (n_steps, n)
            noise.z_dev, noise.u_f_dev = z.data_ptr(), u_f.data_ptr()
            keep += [z, u_f]
            if self.levels >= 2:
                u_c = torch.as_tensor(inject['u_c'], dtype=torch.float64).to(self.device).contiguous()
                assert tuple(u_c.shape) == (n_steps, J, n)
                noise.u_c_dev = u_c.data_ptr()
                keep.append(u_c)
        elif record:
            noise.mode = NOISE_RECORD
            res['z'] = torch.zeros(n_steps, J, d, n, dtype=torch.float64, device=self.device)
            res['u_c'] = torch.full((n_steps, J, n), float('nan'), dtype=torch.float64, device=self.device)
            res['u_f'] = torch.full((n_steps, n), float('nan'), dtype=torch.float64, device=self.device)
            noise.z_dev, noise.u_c_dev, noise.u_f_dev = (res['z'].data_ptr(), res['u_c'].data_ptr(),
                                                        res['u_f'].data_ptr())
        with torch.cuda.device(self.device):
            check(self.lib.yg_run(self._h, n_steps, int(thin), C.byref(out), C.byref(noise), self._stream()))
        res['_keep'] = keep
        return res

    def layout(self):
        dd = int(np.asarray(self.problem.arrays['L0_data']).shape[1]) if self.cfg.aem else 0
        return state_layout(self.n_chains, self.dim, self.levels, self.cfg.adaptive, dd)

    def state(self):
        r = {k: self._empty(*shape, dtype=dtype) for k, (shape, dtype) in self.layout().items()}
        st = YgState(**{k + '_dev': v.data_ptr() for k, v in r.items()})
        with torch.cuda.device(self.device):
            check(self.lib.yg_get_state(self._h, C.byref(st), self._stream()))
        c = self.counters()
        r['step_index'], r['welford_n'], r['am_steps'] = c['step_index'], c['welford_n'], c['am_steps']
        return r

    def accept_counts(self):
        """Per-chain accepted transitions since set_state: device tensor [n_chains] int64 (asynchronous)."""
        out = self._empty(self.n_chains, dtype=torch.int64)
        st = YgState(n_accept_dev=out.data_ptr())
        with torch.cuda.device(self.device):
            check(self.lib.yg_get_state(self._h, C.byref(st), self._stream()))
        return out

    def load_state(self, r):
        """Restores state(); theta and logpost are required, arrays of features this ensemble lacks are ignored."""
        layout = self.layout()
        check_state(r, layout)          # yg_load_state reads the layout's byte count from every pointer it is given
        keep = {k: r[k].to(self.device).contiguous() for k in layout if k in r}
        st = YgState(**{k + '_dev': v.data_ptr() for k, v in keep.items()})
        with torch.cuda.device(self.device):
            check(self.lib.yg_load_state(self._h, C.byref(st), int(r.get('step_index', 0)),
                                         int(r.get('welford_n', 0)),
                                         int(r.get('am_steps', r.get('welford_n', 0))), self._stream()))
            torch.cuda.current_stream(self.device).synchronize()
        return self

    def _counters(self):
        buf = (C.c_int64 * 10)()
        with torch.cuda.device(self.device):
            check(self.lib.yg_get_counters(self._h, buf, self._stream()))
        return [int(x) for x in buf]

    def counters(self):
        keys = ('step_index', 'transitions', 'accepted', 'coarse_evals', 'fine_evals', 'welford_n', 'am_steps',
                'mid_evals', 'coarse_accepted')
        c = dict(zip(keys, self._counters()))
        if self.levels == 1:        # single level: level 0 IS the target
            c['fine_evals'], c['coarse_evals'] = c['coarse_evals'], 0
        return c

    def skipped_evals(self):
        """Level-0 integrations (proposal, design point) skipped since set_state because the proposal's rejection
        was already certain.  Unlike counters(), it depends on the launch geometry and the scheduling."""
        return self._counters()[9]

    def logpost(self, level, theta):
        t = torch.as_tensor(theta, dtype=torch.float64).to(self.device)
        if t.dim() == 1:
            t = t.reshape(1, -1)
        m = t.shape[0]
        soa = t.t().contiguous()
        out = self._empty(m)
        with torch.cuda.device(self.device):
            check(self.lib.yg_logpost(self._h, int(level), C.c_void_p(soa.data_ptr()), m,
                                      C.c_void_p(out.data_ptr()), self._stream()))
        return out

    def pooled_stats(self):
        """Device vector of sufficient statistics (plain sums over local chains)."""
        out = self._empty(int(self.lib.yg_pooled_len(self.dim)))
        with torch.cuda.device(self.device):
            check(self.lib.yg_pooled_stats(self._h, C.c_void_p(out.data_ptr()), self._stream()))
        return out

    def last_launch(self):
        g, b, s, l = C.c_int32(), C.c_int32(), C.c_int32(), C.c_int64()
        check(self.lib.yg_last_launch(self._h, C.byref(g), C.byref(b), C.byref(s), C.byref(l)))
        return dict(grid=g.value, block=b.value, smem=s.value, launches=l.value)


def iat_ess(samples, method='max', sokal=5.0):
    """samples: device tensor [n_samples, d, n_chains] -> (iat[n_chains], ess[n_chains]) int64 tensors.
    Restates integrated_autocorrelation (postprocessing/autocorrelation.py:92-140) per chain."""
    lib = _lib.load()
    assert samples.is_cuda and samples.dtype == torch.float64 and samples.dim() == 3
    samples = samples.contiguous()
    ns, d, n = samples.shape
    iat = torch.empty(n, dtype=torch.int64, device=samples.device)
    ess = torch.empty(n, dtype=torch.int64, device=samples.device)
    with torch.cuda.device(samples.device):
        st = C.c_void_p(torch.cuda.current_stream(samples.device).cuda_stream)
        check(lib.yg_iat_ess(C.c_void_p(samples.data_ptr()), ns, d, n, 1 if method == 'max' else 0,
                             float(sokal), C.c_void_p(iat.data_ptr()), C.c_void_p(ess.data_ptr()), st))
    return iat, ess


def split_moments(samples):
    lib = _lib.load()
    samples = samples.contiguous()
    ns, d, n = samples.shape
    hm = torch.empty(2, d, n, dtype=torch.float64, device=samples.device)
    hv = torch.empty(2, d, n, dtype=torch.float64, device=samples.device)
    with torch.cuda.device(samples.device):
        st = C.c_void_p(torch.cuda.current_stream(samples.device).cuda_stream)
        check(lib.yg_split_moments(C.c_void_p(samples.data_ptr()), ns, d, n, C.c_void_p(hm.data_ptr()),
                                   C.c_void_p(hv.data_ptr()), st))
    return hm, hv


def pooled_sample_stats(samples):
    """samples: device tensor [n_samples, d, n_chains] float64 (yg_run's samples layout, d <= 64) -> device vector of
    the pooled sufficient statistics (parallel.py's layout, yg_pooled_samples) over the stored samples of every chain.
    Entry [2] (accepts) is 0.  Asynchronous on the current stream; the workspace is allocated here."""
    lib = _lib.load()
    if not (torch.is_tensor(samples) and samples.is_cuda and samples.dtype == torch.float64 and samples.dim() == 3):
        raise ValueError("samples must be a float64 CUDA tensor [n_samples, d, n_chains]")
    samples = samples.contiguous()
    ns, d, n = samples.shape
    ws = torch.empty(max(1, int(lib.yg_pooled_samples_workspace_len(d, n))), dtype=torch.float64, device=samples.device)
    out = torch.empty(int(lib.yg_pooled_len(d)), dtype=torch.float64, device=samples.device)
    with torch.cuda.device(samples.device):
        st = C.c_void_p(torch.cuda.current_stream(samples.device).cuda_stream)
        check(lib.yg_pooled_samples(C.c_void_p(samples.data_ptr()), ns, d, n, C.c_void_p(ws.data_ptr()), ws.numel(),
                                    C.c_void_p(out.data_ptr()), st))
    return out


def fp64_peak_tflops(device=0, ms=20.0):
    lib = _lib.load()
    out = C.c_double()
    check(lib.yg_fp64_peak(int(device), float(ms), C.byref(out)))
    return out.value


def rk4_loop_steps_per_s(device=0, ms=20.0):
    """Bare LV RK4 integrator loop (nothing but lv_integrate, 1024 threads per SM): RK4 steps/s of the GPU,
    the ceiling for lv_mh_kernel."""
    lib = _lib.load()
    out = C.c_double()
    check(lib.yg_rk4_loop_rate(int(device), float(ms), C.byref(out)))
    return out.value


def fp64_tensor_peak_tflops(device=0, ms=20.0):
    """FP64 tensor-path (DMMA) micro-benchmark: the roofline denominator of the large linear model."""
    lib = _lib.load()
    out = C.c_double()
    check(lib.yg_fp64_tensor_peak(int(device), float(ms), C.byref(out)))
    return out.value
