/*
 * yagre_b200.h -- C-ABI of libyagre_b200.so: the B200 (sm_100a) batched-chain
 * backend for the Metropolis-Hastings hot path of rkutri/yagre-mcmc.
 *
 * The reference is pure Python and has no FFI; its boundaries for this path
 * are Python ABCs.  Each entry point below names the reference interface it
 * replaces (paths relative to the reference root):
 *
 *   yg_create / yg_destroy   ChainBuilder.build_method()  chain/builder.py:72-83,
 *                            MRWBuilder chain/method/mrw.py:60-91,
 *                            MLDABuilder chain/method/mlda.py:157-344
 *                            (object wiring -> one POD config + one POD problem)
 *   yg_set_problem           the objects the builders are given:
 *                            UnnormalisedPosterior chain/target.py:4-22,
 *                            AdditiveGaussianNoiseLikelihood statistics/likelihood.py:49-87,
 *                            CentredGaussianNoise statistics/noise.py:8-22,
 *                            Gaussian prior statistics/gaussian.py:27-66,
 *                            CovarianceMatrix family statistics/covariance.py:8-94,
 *                            SolverInterface plugins model/interface.py:7-67
 *                            (LV: test/testSetup.py:61-141, linear: exampleSetup.py:8-52,
 *                            Gaussian targets: test/testSetup.py:15-44)
 *   yg_set_state / yg_seek   initialState of MetropolisHastings.run  chain/metropolisHastings.py:103-110; the
 *                            stream position plays the role of numpy's global generator state
 *                            (statistics/gaussian.py:2,63, chain/metropolisHastings.py:2,68)
 *   yg_run                   the loop of MetropolisHastings.run :112-120 with
 *                            MRWProposal mrw.py:27-38, PCNProposal pcn.py:23-35, _accept_reject :55-73,
 *                            MLDAProposal.generate_proposal mlda.py:100-110 and
 *                            MLDA._acceptance_probability mlda.py:146-154,
 *                            AdaptiveMRWProposal.set_state chain/adaptive.py:55-60,
 *                            AdaptiveErrorModel._process_transition chain/method/aem.py:25-58
 *   yg_get_state/yg_load_state   .chain.trajectory[-1] restart idiom
 *                            (example_inference_linearModel_twoLevel.py:228,236) + diagnostics
 *                            (AcceptanceRateDiagnostics / FullDiagnostics chain/diagnostics.py:19-107,
 *                            WelfordAccumulator statistics/estimation.py:4-58)
 *   yg_get_counters          global_acceptance_rate() chain/diagnostics.py:44-46 (+ forward-evaluation
 *                            counters used for the roofline; cf. AEMLikelihood.number_of_model_evaluations
 *                            statistics/likelihood.py:114-115)
 *   yg_iat_ess               integrated_autocorrelation postprocessing/autocorrelation.py:92-140 and the
 *                            ESS idiom example_inference_lotkaVolterra_twoLevel.py:117-118,132
 *   yg_pooled_stats          (new) sufficient statistics for pooled moments / R-hat, summed over local
 *                            chains; the host all-reduces them across GPUs (NCCL, torch.distributed)
 *   yg_pooled_samples_workspace_len / yg_pooled_samples
 *                            (new) the same sufficient statistics from a stored sample buffer, any d <= 64
 *   yg_set_proposal_factor   (new) pooled proposal covariance; cf. AdaptiveMRWProposal.set_state
 *                            chain/adaptive.py:55-60
 *   yg_logpost               DensityInterface.evaluate_log statistics/interface.py:6-10
 *   yg_fp64_peak             (new) DFMA micro-benchmark: the measured FP64 roofline denominator
 *   yg_rk4_loop_rate         (new) bare RK4 integrator loop (the replacement of LotkaVolterraSolver.invoke,
 *                            test/testSetup.py:109-141): ceiling of RK4 steps/s for the LV step kernel
 *
 * Conventions
 *   - All `*_dev` pointers are DEVICE pointers owned by the caller (PyTorch
 *     allocates them); host pointers are copied during the call.
 *   - Ensemble arrays are struct-of-arrays with the chain index fastest:
 *     theta[d][n_chains], samples[n_out][d][n_chains], ...
 *   - `stream` is a cudaStream_t (as void*); yg_run / yg_iat_ess / yg_pooled_stats
 *     are asynchronous on it, do not allocate and do not synchronise.
 *   - Every function returns YG_OK (0) or a negative yg_status; the message is
 *     available from yg_last_error() (thread local).  Nothing throws across the ABI.
 *   - A handle is bound to one device and is not thread-safe; distinct handles
 *     are independent (one process or thread per GPU).
 */
#ifndef YAGRE_B200_H
#define YAGRE_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define YG_ABI_VERSION 5u
#define YG_MAX_LEVELS 3         /* densities per problem: up to two surrogates + the target */
#define YG_MAX_DIM 8           /* parameter dimension of the one-chain-per-thread kernels */
#define YG_MAX_DATA_DIM 8
/* YG_MODEL_LINEAR beyond those sizes runs on the FP64 tensor path (DMMA GEMM, linear_dmma_kernel.cu): MRW, pCN,
 * two-level delayed acceptance and MLDA with two surrogates, tempered levels; diagonal measurement noise; diagonal or
 * dense prior precision and proposal factor; every combination up to YG_BIG_MAX_DIM x YG_BIG_MAX_DATA_DIM per level (an
 * operand that does not fit shared memory -- level 1's G, level 2's G, then the dense factor -- is read from L2; rates
 * measured on a B200 in profiles/streamed_operand.md and profiles/three_level_tensor.md);
 * no adaptive Metropolis / adaptive error model;
 * Welford M2 is then diagonal only ([d, n_chains] instead of [d, d, n_chains]). */
#define YG_BIG_MAX_DIM 64
#define YG_BIG_MAX_DATA_DIM 256

typedef enum yg_status {
    YG_OK = 0,
    YG_ERR_INVALID = -1,       /* bad argument / inconsistent config (ValueError)         */
    YG_ERR_CUDA = -2,          /* CUDA runtime error (RuntimeError)                        */
    YG_ERR_UNSUPPORTED = -3,   /* model / shape outside the kernels (NotImplementedError)  */
    YG_ERR_ABI = -4,           /* abi_version mismatch                                     */
    YG_ERR_STATE = -5          /* call order: problem / state not set                      */
} yg_status;

typedef enum yg_model { YG_MODEL_GAUSS = 0, YG_MODEL_LINEAR = 1, YG_MODEL_LV_RK4 = 2 } yg_model;
typedef enum yg_eq_mode { YG_EQ_EXACT = 0, YG_EQ_ISCLOSE = 1 } yg_eq_mode;
typedef enum yg_noise_mode { YG_NOISE_PHILOX = 0, YG_NOISE_INJECT = 1, YG_NOISE_RECORD = 2 } yg_noise_mode;

typedef struct yg_ensemble yg_ensemble;     /* opaque */

/* One level of the model hierarchy (host pointers, row-major, copied by yg_set_problem). */
typedef struct yg_level {
    /* YG_MODEL_GAUSS: logp = -0.5 (t-m)' P (t-m) + logconst */
    const double *g_mean;       /* [d]   */
    const double *g_prec;       /* [d,d] */
    double g_logconst;
    /* regression levels: log-likelihood + log-prior */
    int32_t n_data, data_dim;
    const double *data;         /* [n_data, data_dim] */
    const double *noise_prec;   /* [data_dim, data_dim]; exact zeros are skipped (large linear model: diagonal) */
    const double *prior_mean;   /* [d] */
    const double *prior_prec;   /* [d,d] */
    /* YG_MODEL_LINEAR: F = G theta + b */
    const double *G;            /* [data_dim, d] */
    const double *b;            /* [data_dim] */
    /* YG_MODEL_LV_RK4: one 2-state ODE per design row, output = state at T */
    const double *design;       /* [n_data, 2] */
    double alpha, gamma, T;
    int32_t rk4_steps;
    /* TemperedUnnormalisedPosterior (chain/target.py:25-43): tempering * logL + logprior when tempered != 0
     * (regression levels of every kernel; tempering in [0, 1]) */
    int32_t tempered;
    double tempering;
} yg_level;

typedef enum yg_proposal { YG_PROPOSAL_MRW = 0, YG_PROPOSAL_PCN = 1 } yg_proposal;

typedef struct yg_problem {
    const double *prop_L;       /* [d,d] lower-triangular proposal factor, p = s + L z */
    /* level[n_levels-1] is the target.  n_levels == 2: level[0] is the surrogate of two-level delayed
     * acceptance.  n_levels == 3 is MLDA with TWO surrogates exactly as the reference runs it
     * (chain/method/mlda.py:12-43,60-71,112-117): the proposal is the end point of an MRW sub-chain on
     * level[0] of sub_chain_length = subChainLengths[1] steps (subChainLengths[0] is ignored there), and the
     * screen is min(1, exp(pi_2(p) + pi_1(s) - pi_1(p) - pi_2(s))) with the FINEST surrogate level[1]. */
    yg_level level[YG_MAX_LEVELS];
    /* YG_PROPOSAL_PCN (chain/method/pcn.py:9-57, single level): prop_L is the factor of the PRIOR
     * covariance, p = sqrt(1 - 2h) s + sqrt(2h) (pcn_mean + L z); the target is the likelihood
     * alone, i.e. the caller passes a zero prior_prec for the level. */
    int32_t proposal;           /* yg_proposal */
    int32_t _pad;
    double pcn_step;            /* h in (0, 0.5] */
    const double *pcn_mean;     /* [d] prior mean (the reference requires zeros, pcn.py:44-46); NULL = zeros */
} yg_problem;

typedef struct yg_config {
    uint32_t abi_version;       /* = YG_ABI_VERSION, first field */
    int32_t device;             /* CUDA device ordinal */
    int64_t n_chains;           /* chains held by THIS handle */
    int64_t chain_offset;       /* global id of local chain 0 (Philox keying: results do not depend on the GPU count) */
    uint64_t seed;
    int32_t model;              /* yg_model */
    int32_t dim;                /* parameter dimension, 1..YG_MAX_DIM (LV: 2) */
    int32_t n_levels;           /* 1 = MRW, 2 = two-level delayed acceptance (MLDA with one surrogate),
                                   3 = MLDA with two surrogates (see yg_problem.level) */
    int32_t sub_chain_length;   /* J (n_levels >= 2), else ignored */
    int32_t eq_mode;            /* yg_eq_mode: ParameterVector (exact) / ScalarParameter (isclose) */
    /* 1 = per-chain adaptive Metropolis: AdaptiveMRWProposal.set_state -> update() (chain/adaptive.py:55-60)
     * before EVERY proposal of the MRW chain it drives, with that chain's current state -- the chain state for
     * one level, the sub-chain state for the coarse MRW of delayed acceptance (then idle / collection count
     * coarse proposals).  All models of the one-chain-per-thread and LV kernels, dim >= 2. */
    int32_t adaptive;
    int64_t am_idle_steps;      /* updates before moments are collected */
    int64_t am_collection_steps;/* collected states before the proposal switches */
    int32_t am_refresh;         /* recompute the Cholesky factor every R steps (>= 1) */
    int32_t _pad0;
    double am_eps;              /* regularisation: C = s (Cov + eps I) */
    double am_scale;            /* s; <= 0 selects 2.4^2 / d */
    int32_t blocks_per_sm;      /* 0 = default; tuning knob of the LV kernel */
    int32_t threads_per_block;  /* 0 = default */
    int32_t rk4_segment;        /* 0 = default (128): RK4 steps per work unit of the LV kernel */
    /* adaptive error model (chain/method/aem.py, statistics/likelihood.py:90-155, statistics/noise.py:25-61):
     * n_levels == 2, YG_MODEL_LINEAR (dim, data_dim <= 8), diagonal measurement noise.  Per chain: Welford of
     * F_fine - F_coarse on accepted fine steps; the coarse residual is shifted by its mean once aem_min_data
     * errors were seen, the noise variance is inflated by (scaling x) its variance from aem_min_data + 1 on; the
     * coarse likelihood's LRU(3) cache is reproduced, including that cached values survive model updates. */
    int32_t aem;                /* 0 / 1 */
    int32_t aem_min_data;       /* minDataSize >= 2 */
    int32_t aem_heuristic;      /* useNoiseHeuristic: scaling = min(2 max(var) / max(min(var), 1e-6), 100) */
    /* 0 (default) = FullDiagnostics: the Welford moments w_mean / w_m2 of the pre-transition states are maintained
     * (chain/diagnostics.py:67-107); 1 = AcceptanceRateDiagnostics only -- the default diagnostics of the reference's
     * builders (chain/builder.py:14-16) -- : they stay zero.  Honoured by the tensor-path kernel, where the moments
     * live in L2 (d x 2 doubles per chain); the other kernels keep them in registers / shared memory for free. */
    int32_t acceptance_only;
    /* 1 = the LV kernel evaluates every design point of every proposal.  0 (default): at level 0 it skips the
     * remaining integrations of a proposal whose partial misfit already certifies its rejection (diagonal noise
     * precision only); results are bit-identical either way. */
    int32_t early_reject_off;
} yg_config;

typedef struct yg_noise {
    int32_t mode;               /* yg_noise_mode */
    int32_t _pad;
    double *z_dev;              /* [n_steps, J, d, n_chains] (single level: J = 1) */
    double *u_c_dev;            /* [n_steps, J, n_chains]    (two level only)      */
    double *u_f_dev;            /* [n_steps, n_chains]                             */
} yg_noise;

typedef struct yg_outputs {
    double *samples_dev;        /* [n_steps/thin, d, n_chains] state after every thin-th transition, or NULL */
    uint8_t *accepted_dev;      /* [n_steps, n_chains] 0/1 per transition, or NULL */
    double *logpost_dev;        /* [n_steps/thin, n_levels, n_chains] log-posterior of the stored state, or NULL */
} yg_outputs;

/* yg_set_state flags.  The reference keeps diagnostics until clear() (chain/metropolisHastings.py:122-125) and
 * the state of an adaptive proposal / error model for the life of the object; a second run() only restarts the chain. */
#define YG_KEEP_DIAGNOSTICS 1   /* keep accept counters, Welford moments and the evaluation counters */
#define YG_KEEP_ADAPTATION  2   /* keep adaptive-Metropolis moments / factors and the adaptive error model */

/* Per-chain state, for diagnostics and bit-exact resume.  Any pointer may be NULL. */
typedef struct yg_state {
    double *theta_dev;          /* [d, n_chains] */
    double *logpost_dev;        /* [n_levels, n_chains] */
    int64_t *n_accept_dev;      /* [n_chains] */
    double *w_mean_dev;         /* [d, n_chains]    Welford mean of the pre-transition states */
    double *w_m2_dev;           /* [d, d, n_chains] Welford second central moment (diagonal = WelfordAccumulator M2) */
    double *prop_L_dev;         /* [d, d, n_chains] current proposal factor (adaptive only) */
    double *am_mean_dev;        /* [d, n_chains]    adaptive Metropolis running mean (adaptive only) */
    double *am_m2_dev;          /* [d, d, n_chains] adaptive Metropolis second central moment (adaptive only) */
    /* adaptive error model only */
    int64_t *aem_n_dev;         /* [n_chains] error realisations seen (WelfordAccumulator.nData) */
    double *aem_mean_dev;       /* [data_dim, n_chains] mean of F_fine - F_coarse */
    double *aem_m2_dev;         /* [data_dim, n_chains] second central moment (variance = m2 / (n - 1)) */
    double *aem_cache_dev;      /* [3 (d + 1) + 1, n_chains] coarse LRU(3): keys, values, entry count (oldest first) */
} yg_state;

const char *yg_last_error(void);
uint32_t yg_abi_version(void);

int yg_create(const yg_config *cfg, yg_ensemble **out);
int yg_destroy(yg_ensemble *e);
int yg_set_problem(yg_ensemble *e, const yg_problem *pb);

/* theta0_dev[d, n_chains]; evaluates the log-posterior(s) of the initial state and resets the diagnostics
 * and the adaptation state unless `flags` keeps them.  The Philox stream position (step index) is NOT
 * touched: like the reference's numpy generator it keeps advancing across runs, so two runs from the same
 * state see different noise.  yg_seek repositions it explicitly. */
int yg_set_state(yg_ensemble *e, const double *theta0_dev, int32_t flags, void *stream);
/* Sets the Philox stream position: the next yg_run draws the noise of steps step_index, step_index + 1, ... */
int yg_seek(yg_ensemble *e, int64_t step_index);

/* Replaces the proposal factor L (host, [d, d] row-major, lower triangular, positive diagonal) for the
 * following yg_run calls: every chain of an adaptive ensemble restarts from it, a non-adaptive ensemble
 * uses it as is.  This is the hook for a POOLED proposal covariance (covariance of all chains of all GPUs,
 * all-reduced by the host; the reference swaps a chain's proposal covariance in
 * AdaptiveMRWProposal.set_state, chain/adaptive.py:55-60).  Refused for pCN (the factor is the prior's). */
int yg_set_proposal_factor(yg_ensemble *e, const double *L_host, void *stream);

/* n_steps transitions of every chain.  thin >= 1; n_steps % thin == 0 when samples are stored. */
int yg_run(yg_ensemble *e, int64_t n_steps, int32_t thin,
           const yg_outputs *out, const yg_noise *noise, void *stream);

int yg_get_state(yg_ensemble *e, const yg_state *dst, void *stream);
/* am_steps: transitions since the adaptation state was reset (index base of the adaptive-Metropolis updates). */
int yg_load_state(yg_ensemble *e, const yg_state *src, int64_t step_index, int64_t welford_n, int64_t am_steps,
                  void *stream);

/* out_host[10] = {step index, transitions done (all chains), accepted, level-0 forward evals,
 * target-level forward evals, welford n, am_steps, level-1 forward evals of a three-level hierarchy,
 * accepted coarse sub-steps (the acceptance the reference's surrogate diagnostics record, mlda.py:58-62),
 * level-0 integrations (proposal, design point) the LV kernel skipped because the rejection was already
 * certain}.  The last one depends on the launch geometry and the scheduling, the others do not.
 * Synchronises `stream`. */
int yg_get_counters(yg_ensemble *e, int64_t *out_host, void *stream);

/* log-posterior of theta_dev[d, n] at `level` -> out_dev[n] (same kernels' device functions). */
int yg_logpost(yg_ensemble *e, int32_t level, const double *theta_dev, int64_t n, double *out_dev, void *stream);

/* samples_dev[n_samples, d, n_chains] -> iat_dev[n_chains] (max over coordinates, Sokal window c),
 * ess_dev[n_chains] = n_samples / max(iat,1) (integer division), either may be NULL.  A chain whose stored
 * series is constant or non-finite (no autocorrelation function; the reference fails on it) reports
 * iat = n_samples and ess = 0.
 * method: 0 = 'mean', 1 = 'max'.  Series of more than 25,600 samples use a stream-ordered scratch
 * allocation (cudaMallocAsync / cudaFreeAsync on `stream`; still no host synchronisation). */
int yg_iat_ess(const double *samples_dev, int64_t n_samples, int32_t d, int64_t n_chains,
               int32_t method, double sokal_const, int64_t *iat_dev, int64_t *ess_dev, void *stream);

/* Sufficient statistics over the local chains, written to out_dev[yg_pooled_len(d)]:
 *   [0] n_chains  [1] welford n  [2] sum accepts
 *   then sum_c mean_c [d], sum_c mean_c mean_c' [d*d], sum_c M2_c [d*d], sum_c var_c [d].
 * Every entry is a plain sum over chains, so an all-reduce(sum) pools GPUs. */
int64_t yg_pooled_len(int32_t d);
int yg_pooled_stats(yg_ensemble *e, double *out_dev, void *stream);

/* The same vector from a stored sample buffer samples_dev[n_samples, d, n_chains] (yg_run's samples layout), for any
 * 1 <= d <= YG_BIG_MAX_DIM: with mean_c the mean of chain c's stored samples and M2_c = sum_t (x_ct - mean_c)(x_ct - mean_c)':
 *   [0] n_chains  [1] n_samples  [2] 0 (the caller fills in the accepts it wants pooled)
 *   then sum_c mean_c [d], sum_c mean_c mean_c' [d*d], sum_c M2_c [d*d] (symmetric), sum_c diag(M2_c)/(n_samples-1) [d]
 *   (0 for n_samples == 1).
 * M2_c is formed from data shifted by each chain's first sample, so a large common offset costs no accuracy.  One read
 * of the buffer; deterministic (fixed-order sums, bitwise repeatable).  workspace_dev holds at least
 * yg_pooled_samples_workspace_len(d, n_chains) doubles.  Asynchronous on `stream`, no allocation, no synchronisation. */
int64_t yg_pooled_samples_workspace_len(int32_t d, int64_t n_chains);   /* doubles; 0 if d < 1 or n_chains < 1 */
int yg_pooled_samples(const double *samples_dev, int64_t n_samples, int32_t d, int64_t n_chains,
                      double *workspace_dev, int64_t workspace_len, double *out_dev, void *stream);

/* Per-chain mean and unbiased variance of each half of samples_dev[n_samples, d, n_chains]
 * -> half_mean_dev[2, d, n_chains], half_var_dev[2, d, n_chains] (split-R-hat inputs). */
int yg_split_moments(const double *samples_dev, int64_t n_samples, int32_t d, int64_t n_chains,
                     double *half_mean_dev, double *half_var_dev, void *stream);

/* Dependent-free DFMA chains on every SM for about `ms` milliseconds; returns TFLOP/s (FMA = 2). */
int yg_fp64_peak(int32_t device, double ms, double *tflops_out);
/* The bare LV RK4 integrator (one integration per thread, 1024 threads per SM, nothing else) for about
 * `ms` milliseconds per launch; returns RK4 steps/s of the whole GPU. */
int yg_rk4_loop_rate(int32_t device, double ms, double *steps_per_s_out);
/* The same for the FP64 tensor path (independent m16n8k4 DMMA accumulator chains). */
int yg_fp64_tensor_peak(int32_t device, double ms, double *tflops_out);

/* Launch geometry and kernel count of the last yg_run (for bench.py's gpu_launches). */
int yg_last_launch(yg_ensemble *e, int32_t *grid, int32_t *block, int32_t *smem_bytes, int64_t *launches);

#ifdef __cplusplus
}
#endif
#endif /* YAGRE_B200_H */
