"""Synthetic problem definitions of the BASELINE.json configs in lowered (plain-array)
form -- shared by bench.py, __graft_entry__.smoke() and the tests.  Constants follow
SURVEY section 8d; sources in the reference:
  C2  example_mcmc_2d_singleLevel.py:19-27          (2-D Gaussian target)
  C3  example_inference_linearModel_twoLevel.py:33-74,128-129,173
  C4  example_inference_lotkaVolterra_singleLevel.py:29-59,82-83
  C5  example_inference_lotkaVolterra_twoLevel.py:29-44,56-77,95-106

Only data SYNTHESIS happens here (a 10-line numpy RK4 to make the observations);
no sampling code.
"""
import numpy as np
from numpy.random import Generator, Philox


def _diag_prec(var, dim):
    return np.diag(np.reciprocal(np.full(dim, float(var))))


def _iid_L(var, dim):
    v = np.full(dim, float(var))
    return np.diag(np.sqrt(np.reciprocal(np.reciprocal(v))))      # covariance.py:37-38,51-52


def lv_forward_numpy(theta, design, alpha, gamma, T, N):
    """RK4 end state per design row (specification: oracle/ref_harness.py)."""
    beta, delta = np.exp(theta[0]), np.exp(theta[1])
    x, y = design[:, 0].copy(), design[:, 1].copy()
    h = T / N
    h2, h6 = 0.5 * h, h / 6.0

    def f(x, y):
        return alpha * x - beta * x * y, delta * x * y - gamma * y
    for _ in range(N):
        k1x, k1y = f(x, y)
        k2x, k2y = f(x + h2 * k1x, y + h2 * k1y)
        k3x, k3y = f(x + h2 * k2x, y + h2 * k2y)
        k4x, k4y = f(x + h * k3x, y + h * k3y)
        x = x + h6 * (((k1x + 2.0 * k2x) + 2.0 * k3x) + k4x)
        y = y + h6 * (((k1y + 2.0 * k2y) + 2.0 * k3y) + k4y)
    return np.stack([x, y], axis=1)


LV_TRUTH = np.log(np.array([0.4, 0.6]))


def lv_problem(two_level=True, Nc=64, Nf=512, J=3, n_data=10, T=10.0, seed=1112, prop_var=None):
    """C5 (two_level) / C4 (single level, fine model only)."""
    rng = Generator(Philox(seed))
    design = rng.uniform(0.5, 1.5, (n_data, 2))
    alpha, gamma = 0.8, 0.4
    data = lv_forward_numpy(LV_TRUTH, design, alpha, gamma, T, Nf) + np.sqrt(0.04) * rng.standard_normal((n_data, 2))
    if prop_var is None:
        prop_var = 0.1 if two_level else 0.15

    def level(N):
        return dict(data=data, noise_prec=_diag_prec(0.04, 2), prior_mean=np.zeros(2),
                    prior_prec=_diag_prec(1.4, 2), design=design, lv=np.array([alpha, gamma, T, float(N)]))
    arrays = dict(prop_L=_iid_L(prop_var, 2))
    lv = [level(Nc), level(Nf)] if two_level else [level(Nf)]
    for l, L in enumerate(lv):
        arrays.update({f"L{l}_{k}": v for k, v in L.items()})
    meta = dict(model='lv', dim=2, levels=2 if two_level else 1, J=J if two_level else 1, eq='exact',
                Nc=Nc, Nf=Nf, n_data=n_data)
    return meta, arrays


def lv_pcn_problem(step=0.004, prior_var=1.4, Nf=512, n_data=10):
    """pCN on the C4 likelihood (chain/method/pcn.py; test/test_inference_mcmc_singleLevel.py:121-148):
    prop_L is the prior's factor and the level's prior precision is zero (likelihood-only target)."""
    meta, arrays = lv_problem(False, Nf=Nf, n_data=n_data)
    arrays['prop_L'] = _iid_L(prior_var, 2)
    arrays['L0_prior_prec'] = np.zeros((2, 2))
    arrays['pcn_mean'] = np.zeros(2)
    meta.update(proposal='pcn', pcn_step=step)
    return meta, arrays


def lv_initial_states(n_chains, seed=7, chain_offset=0):
    """theta0 = theta* + 0.05 N(0, I) per chain (the example's [-7, 2.8] is unusable with RK4; SURVEY 7).
    Keyed on the global chain id so a sharded run starts exactly like the single-GPU run."""
    rng = Generator(Philox(key=seed, counter=[0, 0, 0, chain_offset]))
    return LV_TRUTH + 0.05 * rng.standard_normal((n_chains, 2))


def linear_problem(two_level=True, J=5):
    """C3."""
    G_f = np.array([[1.4, -0.2], [-0.6, 0.7]])
    b_f = np.zeros(2)
    G_c = G_f + np.array([[-0.6, -0.2], [0.4, 1.1]])
    b_c = np.array([0.5, -0.9])
    truth = np.array([1.5, 0.5])
    rng = Generator(Philox(2222))
    data = np.array([G_f @ truth + b_f + np.sqrt(0.3) * rng.standard_normal(2) for _ in range(5)])

    def level(G, b):
        return dict(data=data, noise_prec=_diag_prec(0.3, 2), prior_mean=truth + np.array([-0.2, 0.4]),
                    prior_prec=_diag_prec(5.0, 2), G=G, b=b)
    arrays = dict(prop_L=_iid_L(0.5, 2))
    lv = [level(G_c, b_c), level(G_f, b_f)] if two_level else [level(G_f, b_f)]
    for l, L in enumerate(lv):
        arrays.update({f"L{l}_{k}": v for k, v in L.items()})
    meta = dict(model='linear', dim=2, levels=2 if two_level else 1, J=J if two_level else 1, eq='exact')
    return meta, arrays


def linear_posterior(level='f'):
    """Closed-form Gaussian posterior of the C3 linear model (for moment checks)."""
    meta, a = linear_problem(True)
    pre = 'L1_' if level == 'f' else 'L0_'
    G, b, data = a[pre + 'G'], a[pre + 'b'], a[pre + 'data']
    P0, m0, Pn = a[pre + 'prior_prec'], a[pre + 'prior_mean'], a[pre + 'noise_prec']
    n = data.shape[0]
    P = P0 + n * G.T @ Pn @ G
    rhs = P0 @ m0 + G.T @ Pn @ (data - b).sum(axis=0)
    cov = np.linalg.inv(P)
    return cov @ rhs, cov


def big_linear_problem(d=64, data_dim=256, n_data=1, two_level=False, J=2, seed=3, prop_var=None):
    """GEMM-sized linear model (SURVEY 8d: d = 64, dataDim = 256, nData = 1, G ~ N(0, 1/d), seed 3): served
    by the DMMA kernel.  Diagonal noise / prior / proposal.  Two level: coarse = perturbed fine model."""
    rng = Generator(Philox(seed))
    G_f = rng.standard_normal((data_dim, d)) / np.sqrt(d)
    b_f = 0.1 * rng.standard_normal(data_dim)
    G_c = G_f + 0.05 * rng.standard_normal((data_dim, d)) / np.sqrt(d)
    b_c = b_f + 0.02 * rng.standard_normal(data_dim)
    truth = rng.standard_normal(d)
    noise_var, prior_var = 0.05, 2.0
    data = np.array([G_f @ truth + b_f + np.sqrt(noise_var) * rng.standard_normal(data_dim) for _ in range(n_data)])
    if prop_var is None:
        prop_var = 2.4 ** 2 / d * noise_var / max(n_data * data_dim / d, 1.0)      # ~ optimal RWM scaling

    def level(G, b):
        return dict(data=data, noise_prec=_diag_prec(noise_var, data_dim), prior_mean=np.zeros(d),
                    prior_prec=_diag_prec(prior_var, d), G=G, b=b)
    arrays = dict(prop_L=_iid_L(prop_var, d))
    lv = [level(G_c, b_c), level(G_f, b_f)] if two_level else [level(G_f, b_f)]
    for l, L in enumerate(lv):
        arrays.update({f"L{l}_{k}": v for k, v in L.items()})
    meta = dict(model='linear', dim=d, levels=2 if two_level else 1, J=J if two_level else 1, eq='exact',
                truth=truth.tolist())
    return meta, arrays


def big_linear_three_level_problem(d=64, data_dims=(256, 256, 256), n_data=1, J=3, tempering=None, dense_prior=False,
                                   seed=3, prop_var=None):
    """MLDA with two surrogates on a GEMM-sized linear model: one smooth operator observed on three grids, level l on
    data_dims[l] points (coarse, medium, fine; the fine level is the target).  G_l[i, k] = cos(pi (k + 1) x_i + phi_k)
    sqrt(2 / d) at the grid points x_i of level l, the surrogates' operators perturbed by 5 % and 2 %, one truth,
    data per level, diagonal noise.  tempering: {level: t} (TemperedUnnormalisedPosterior); dense_prior: a dense prior
    precision shared by the levels.  The proposal is diagonal."""
    rng = Generator(Philox(seed))
    phase = rng.uniform(0.0, np.pi, d)
    truth = rng.standard_normal(d)
    noise_var, prior_var = 0.05, 2.0
    prior_prec = _diag_prec(prior_var, d)
    prior_mean = np.zeros(d)
    if dense_prior:
        A = rng.standard_normal((d, d))
        cov = prior_var * (A @ A.T / d + 0.5 * np.eye(d))
        prior_prec = np.linalg.inv(cov)
        prior_prec = 0.5 * (prior_prec + prior_prec.T)
        prior_mean = 0.1 * rng.standard_normal(d)
    arrays = {}
    for l, (dd, pert) in enumerate(zip(data_dims, (0.05, 0.02, 0.0))):
        x = (np.arange(dd) + 0.5) / dd
        G = np.cos(np.pi * np.outer(x, np.arange(1, d + 1)) + phase) * np.sqrt(2.0 / d)
        G = G + pert * rng.standard_normal((dd, d)) / np.sqrt(d)
        b = 0.1 * np.sin(2.0 * np.pi * x) + pert * rng.standard_normal(dd)
        data = np.array([G @ truth + b + np.sqrt(noise_var) * rng.standard_normal(dd) for _ in range(n_data)])
        arrays.update({f"L{l}_G": G, f"L{l}_b": b, f"L{l}_data": data, f"L{l}_noise_prec": _diag_prec(noise_var, dd),
                       f"L{l}_prior_mean": prior_mean, f"L{l}_prior_prec": prior_prec})
    for l, t in (tempering or {}).items():
        arrays[f"L{l}_tempering"] = np.array(float(t))
    if prop_var is None:
        prop_var = 2.4 ** 2 / d * noise_var / max(n_data * data_dims[0] / d, 1.0)
    arrays["prop_L"] = _iid_L(prop_var, d)
    meta = dict(model='linear', dim=d, levels=3, J=J, eq='exact', truth=truth.tolist())
    return meta, arrays


def linear_gaussian_posterior(arrays, level):
    """Closed-form Gaussian posterior (mean, covariance) of one level of a lowered linear problem."""
    pre = f"L{level}_"
    G, b, data = arrays[pre + 'G'], arrays[pre + 'b'], arrays[pre + 'data']
    P0, m0, Pn = arrays[pre + 'prior_prec'], arrays[pre + 'prior_mean'], arrays[pre + 'noise_prec']
    P = P0 + data.shape[0] * G.T @ Pn @ G
    rhs = P0 @ m0 + G.T @ Pn @ (data - b).sum(axis=0)
    cov = np.linalg.inv(P)
    return cov @ rhs, cov


def big_linear_flops_per_eval(d, data_dim):
    """Algorithmic work of one forward evaluation of the linear model: the GEMV G theta (2 d dataDim)."""
    return 2.0 * d * data_dim


GAUSS2D_MEAN = np.array([1.0, 1.5])
GAUSS2D_COV = np.array([[2.4, -0.5], [-0.5, 0.7]])


def gauss2d_problem(prop_var=1.0):
    """C2 target."""
    prec = np.linalg.inv(GAUSS2D_COV)
    prec = 0.5 * (prec + prec.T)
    logconst = -0.5 * (2 * np.log(2 * np.pi) + np.log(np.linalg.det(GAUSS2D_COV)))
    arrays = dict(prop_L=_iid_L(prop_var, 2), L0_g_mean=GAUSS2D_MEAN, L0_g_prec=prec, L0_g_logconst=logconst)
    meta = dict(model='gauss', dim=2, levels=1, J=1, eq='exact')
    return meta, arrays


LV_FLOP_PER_RK4_STEP = 58.0      # textbook (unfused) RK4 step of the 2-state system, SURVEY 8d


def lv_flops_per_eval(n_data, N):
    """Algorithmic work of one forward evaluation: 58 flop per RK4 step per ODE (SURVEY 8d)."""
    return LV_FLOP_PER_RK4_STEP * n_data * N
