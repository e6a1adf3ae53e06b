"""ctypes binding of oracle/_build/libyagre_oracle.so (TEST INFRASTRUCTURE).

A problem is a plain dict of numpy arrays in the lowered form the golden
fixtures use: meta (model/dim/levels/J/eq), prop_L and per level L{0,1}_*.
"""
import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(_HERE, "_build", "libyagre_oracle.so")
MODEL = {'gauss': 0, 'linear': 1, 'lv': 2}
EQ = {'exact': 0, 'isclose': 1}
_dp = C.POINTER(C.c_double)


class YoLevel(C.Structure):
    _fields_ = [("g_mean", _dp), ("g_prec", _dp), ("g_logconst", C.c_double),
                ("n_data", C.c_int32), ("data_dim", C.c_int32),
                ("data", _dp), ("noise_prec", _dp), ("prior_mean", _dp), ("prior_prec", _dp),
                ("G", _dp), ("b", _dp), ("design", _dp),
                ("alpha", C.c_double), ("gamma", C.c_double), ("T", C.c_double),
                ("rk4_steps", C.c_int32), ("tempered", C.c_int32), ("tempering", C.c_double)]


class YoProblem(C.Structure):
    _fields_ = [("model", C.c_int32), ("dim", C.c_int32), ("n_levels", C.c_int32), ("J", C.c_int32),
                ("eq_mode", C.c_int32), ("_pad", C.c_int32), ("prop_L", _dp), ("level", YoLevel * 3),
                ("adaptive", C.c_int32), ("am_refresh", C.c_int32), ("am_idle", C.c_int64),
                ("am_collect", C.c_int64), ("am_eps", C.c_double), ("am_scale", C.c_double),
                ("pcn", C.c_int32), ("_pad2", C.c_int32), ("pcn_a", C.c_double), ("pcn_b", C.c_double),
                ("pcn_mean", _dp),
                ("aem", C.c_int32), ("aem_min_data", C.c_int32), ("aem_heuristic", C.c_int32), ("_pad3", C.c_int32)]


def build(force=False):
    src = os.path.join(_HERE, "yagre_oracle.c")
    if force or not os.path.exists(_SO) or (
            os.path.exists(src) and os.path.getmtime(src) > os.path.getmtime(_SO)):
        subprocess.check_call(["make", "-s", "-C", _HERE])
    return _SO


_lib = None


def lib():
    global _lib
    if _lib is None:
        build()
        _lib = C.CDLL(_SO)
        _lib.yo_logpost.restype = C.c_double
        _lib.yo_philox_uniform.restype = C.c_double
        _lib.yo_iat.restype = C.c_int64
    return _lib


def _arr(a):
    return np.ascontiguousarray(np.asarray(a, dtype=np.float64))


def _ptr(a):
    return a.ctypes.data_as(_dp)


class Problem:
    """Keeps the numpy buffers alive next to the ctypes struct."""

    def __init__(self, meta, arrays, adaptive=None):
        self.meta = dict(meta)
        adaptive = adaptive or meta.get('am')
        self.keep = {}
        pb = YoProblem()
        pb.model = MODEL[meta['model']]
        pb.dim = int(meta['dim'])
        pb.n_levels = int(meta['levels'])
        pb.J = int(meta['J'])
        pb.eq_mode = EQ[meta.get('eq', 'exact')]
        pb.am_refresh = 1
        if adaptive:
            pb.adaptive = 1
            pb.am_idle = int(adaptive.get('idle', 0))
            pb.am_collect = int(adaptive.get('collection', 100))
            pb.am_refresh = max(1, int(adaptive.get('refresh', 1)))      # abi.cu make_args: 0 refreshes every step
            pb.am_eps = float(adaptive.get('eps', 1e-4))
            sc = float(adaptive.get('scale') or 0.0)
            pb.am_scale = sc if sc > 0 else 2.4 * 2.4 / int(meta['dim'])

        if meta.get('proposal', 'mrw') == 'pcn':
            import math
            t = 2. * float(meta['pcn_step'])
            pb.pcn, pb.pcn_a, pb.pcn_b = 1, math.sqrt(1. - t), math.sqrt(t)
            self.keep['pcn_mean'] = _arr(arrays.get('pcn_mean', np.zeros(int(meta['dim']))))
            pb.pcn_mean = _ptr(self.keep['pcn_mean'])

        if meta.get('aem'):
            pb.aem, pb.aem_min_data, pb.aem_heuristic = 1, int(meta['aem']['min_data']), int(bool(meta['aem']['heuristic']))

        def put(obj, field, key):
            if key in arrays:
                a = _arr(arrays[key])
                self.keep[key] = a
                setattr(obj, field, _ptr(a))
        put(pb, "prop_L", "prop_L")
        for l in range(pb.n_levels):
            lv = pb.level[l]
            pre = f"L{l}_"
            for f in ("g_mean", "g_prec", "data", "noise_prec", "prior_mean", "prior_prec", "G", "b", "design"):
                put(lv, f, pre + f)
            if pre + "g_logconst" in arrays:
                lv.g_logconst = float(np.asarray(arrays[pre + "g_logconst"]))
            if pre + "data" in arrays:
                lv.n_data, lv.data_dim = (int(x) for x in np.asarray(arrays[pre + "data"]).shape)
            if pre + "lv" in arrays:
                a = np.asarray(arrays[pre + "lv"], dtype=np.float64)
                lv.alpha, lv.gamma, lv.T, lv.rk4_steps = float(a[0]), float(a[1]), float(a[2]), int(a[3])
            if pre + "tempering" in arrays:
                lv.tempered, lv.tempering = 1, float(np.asarray(arrays[pre + "tempering"]).reshape(-1)[0])
        self.pb = pb
        self.dim, self.J, self.n_levels = pb.dim, pb.J, pb.n_levels


def run_injected(problem, theta0, z, u_c, u_f, n_threads=0):
    """theta0[nc,d] z[nc,ns,J,d] u_c[nc,ns,J] u_f[nc,ns] -> dict of outputs (chain-major).
    coarse_accepted[nc]: accepted sub-steps of the coarse sub-chain per chain (zero for a single level)."""
    theta0, z, u_c, u_f = _arr(theta0), _arr(z), _arr(u_c), _arr(u_f)
    nc, ns = u_f.shape
    d = problem.dim
    assert z.shape == (nc, ns, problem.J, d) and u_c.shape == (nc, ns, problem.J)
    traj = np.empty((nc, ns + 1, d))
    acc = np.empty((nc, ns), dtype=np.uint8)
    lp0 = np.empty((nc, ns + 1))
    lp1 = np.full((nc, ns + 1), np.nan)
    lp2 = np.full((nc, ns + 1), np.nan)
    wm = np.empty((nc, d))
    wv = np.empty((nc, d))
    ev = np.zeros(3, dtype=np.int64)
    dd = int(problem.pb.level[0].data_dim)
    aem = np.zeros((nc, 2 + 2 * max(dd, 1)))
    am = np.zeros((nc, d + 2 * d * d))
    cacc = np.zeros(nc, dtype=np.int64)
    rc = lib().yo_run_injected(C.byref(problem.pb), C.c_int64(nc), C.c_int64(ns),
                               _ptr(theta0), _ptr(z), _ptr(u_c), _ptr(u_f), _ptr(traj),
                               acc.ctypes.data_as(C.c_void_p), _ptr(lp0), _ptr(lp1), _ptr(lp2), _ptr(wm), _ptr(wv),
                               ev.ctypes.data_as(C.c_void_p), C.c_int(n_threads), _ptr(aem), _ptr(am),
                               cacc.ctypes.data_as(C.c_void_p))
    assert rc == 0
    out = dict(traj=traj, accepted=acc, logpost_L0=lp0, logpost_L1=lp1, logpost_L2=lp2,
               welford_mean=wm, welford_var=wv, n_evals=ev, coarse_accepted=cacc)
    if problem.pb.adaptive:
        out.update(am_mean=am[:, :d].copy(), am_m2=am[:, d:d + d * d].reshape(nc, d, d).copy(),
                   am_L=am[:, d + d * d:].reshape(nc, d, d).copy())
    if problem.pb.aem:
        out.update(aem_n=aem[:, 0].astype(np.int64), aem_model_evals=aem[:, 1].astype(np.int64),
                   aem_mean=aem[:, 2:2 + dd], aem_var=aem[:, 2 + dd:2 + 2 * dd])
    return out


def run_philox(problem, theta, seed, n_steps, chain_offset=0, step0=0, thin=1, store=True, n_threads=0):
    theta = _arr(theta).copy()
    nc, d = theta.shape
    n_out = n_steps // thin
    traj = np.empty((nc, n_out, d)) if store else None
    nacc = np.zeros(nc, dtype=np.int64)
    ev = np.zeros(2, dtype=np.int64)
    rc = lib().yo_run_philox(C.byref(problem.pb), C.c_int64(nc), C.c_int64(chain_offset),
                             C.c_uint64(seed), C.c_uint64(step0), C.c_int64(n_steps), C.c_int64(thin),
                             _ptr(theta), _ptr(traj) if store else None,
                             nacc.ctypes.data_as(C.c_void_p), ev.ctypes.data_as(C.c_void_p),
                             C.c_int(n_threads))
    assert rc == 0
    return dict(theta=theta, traj=traj, n_accept=nacc, n_evals=ev)


def logpost(problem, level, theta):
    t = _arr(theta)
    return lib().yo_logpost(C.byref(problem.pb), C.c_int(level), _ptr(t), None)


def forward(problem, level, theta):
    t = _arr(theta)
    lv = problem.pb.level[level]
    F = np.empty((lv.n_data, lv.data_dim)) if problem.pb.model == 2 else np.empty(lv.data_dim)
    assert lib().yo_forward(C.byref(problem.pb), C.c_int(level), _ptr(t), _ptr(F)) == 0
    return F


def philox4x32_10(ctr, key):
    c = (C.c_uint32 * 4)(*[int(x) for x in ctr])
    k = (C.c_uint32 * 2)(*[int(x) for x in key])
    o = (C.c_uint32 * 4)()
    lib().yo_philox4x32_10(c, k, o)
    return [int(x) for x in o]


def philox_uniform(seed, chain, step, sub):
    return lib().yo_philox_uniform(C.c_uint64(seed), C.c_uint64(chain), C.c_uint64(step), C.c_uint32(sub))


def philox_normals(seed, chain, step, sub, d):
    z = np.empty(d)
    lib().yo_philox_normals(C.c_uint64(seed), C.c_uint64(chain), C.c_uint64(step), C.c_uint32(sub),
                            C.c_int(d), _ptr(z))
    return z


def iat(seq, method='max', sokal=5.0):
    s = _arr(seq)
    n, d = s.shape
    return int(lib().yo_iat(_ptr(s), C.c_int64(n), C.c_int(d), C.c_int(1 if method == 'max' else 0),
                            C.c_double(sokal)))


def acf(x):
    x = _arr(x)
    out = np.empty_like(x)
    lib().yo_acf(_ptr(x), C.c_int64(x.size), _ptr(out))
    return out


def welford(x):
    x = _arr(x)
    n, d = x.shape
    m, v = np.empty(d), np.empty(d)
    lib().yo_welford(_ptr(x), C.c_int64(n), C.c_int(d), _ptr(m), _ptr(v))
    return m, v


def cholesky(Cm):
    Cm = _arr(Cm)
    d = Cm.shape[0]
    L = np.empty((d, d))
    rc = lib().yo_cholesky(_ptr(Cm), C.c_int(d), _ptr(L))
    if rc != 0:
        raise np.linalg.LinAlgError("not positive definite")
    return L


def chol_apply(L, x):
    L, x = _arr(L), _arr(x)
    y = np.empty_like(x)
    lib().yo_chol_apply(_ptr(L), C.c_int(L.shape[0]), _ptr(x), _ptr(y))
    return y


def chol_solve(L, x):
    L, x = _arr(L), _arr(x)
    y = np.empty_like(x)
    lib().yo_chol_solve(_ptr(L), C.c_int(L.shape[0]), _ptr(x), _ptr(y))
    return y


def num_threads():
    return int(lib().yo_num_threads())
