// ensemble.h -- host-side handle and the argument block passed to the step kernels.
#pragma once
#include <vector>
#include "common.cuh"
#include "lv_model.cuh"

struct RunArgs {
    const DevProblemHeader *problem;
    uint32_t problem_bytes;
    int32_t thin;
    int64_t n_chains, chain_offset;
    uint64_t seed;
    int64_t step0, n_steps, welford_n0;
    int64_t am_t0;                  // transitions since the adaptation state was reset (base of the AM update index)
    // per-chain state, SoA, chain index fastest
    double *theta;                  // [d, n]
    double *logpost;                // [n_levels, n]
    unsigned long long *n_accept;   // [n]
    double *w_mean;                 // [d, n]
    double *w_m2;                   // [d*d, n]
    // adaptive Metropolis (generic kernel only)
    double *am_mean;                // [d, n]
    double *am_m2;                  // [d*d, n]
    double *prop_L;                 // [d*d, n]
    int32_t adaptive, am_refresh;
    int64_t am_idle, am_collect;
    double am_eps, am_scale;
    // adaptive error model (generic kernel, two level, linear model)
    int32_t aem, aem_min_data, aem_heuristic;
    int32_t welford;                // 0: acceptance-only diagnostics, the Welford moments are not maintained (tensor path)
    unsigned long long *aem_n;      // [n]
    double *aem_mean, *aem_m2;      // [data_dim, n]
    double *aem_cache;              // [3 (d + 1) + 1, n]
    // outputs
    double *samples;                // [n_steps/thin, d, n]
    uint8_t *accepted;              // [n_steps, n]
    double *lp_out;                 // [n_steps/thin, n_levels, n]
    // noise
    int32_t noise_mode, _pad;
    double *z, *u_c, *u_f;
    // LV kernel: per-level step size and the chain-independent scaled rates (lv_model.cuh).
    // Passed by value so the integration loop reads them as constant-bank operands (a DFMA with
    // three vector-register sources issues slower than one with two + a constant operand).
    double lv_h[2];
    LvStepConsts lv_k[2];
    // [0] transitions [1] accepted [2] level-0 evals [3] target-level evals [4] level-1 evals of three levels
    // [5] accepted coarse sub-steps (what the reference's surrogate diagnostics count, chain/method/mlda.py:58-62)
    unsigned long long *counters;
};

// The per-chain state buffers, in the order of yg_state; their sizes and groups are the table in abi.cu.
enum StateBuf {
    SB_THETA, SB_LOGPOST, SB_N_ACCEPT, SB_W_MEAN, SB_W_M2, SB_PROP_L, SB_AM_MEAN, SB_AM_M2,
    SB_AEM_N, SB_AEM_MEAN, SB_AEM_M2, SB_AEM_CACHE, SB_COUNT
};

struct yg_ensemble {
    yg_config cfg;
    int sm_count = 0;
    bool problem_set = false, state_set = false;
    bool big = false;                  // large linear model: DevBigHeader blob, linear_dmma_kernel.cu
    std::vector<char> h_problem;
    void *d_problem = nullptr;         // DevBigHeader blob if big, else DevProblemHeader blob
    void *buf[SB_COUNT] = {};          // per-chain state, chain index fastest (RunArgs lists the shapes)
    int aem_data_dim = 0;
    unsigned long long *counters = nullptr;
    double *pool_partials = nullptr;   // [POOL_PARTS][yg_pooled_len(d)] scratch of yg_pooled_stats
    long long *big_done = nullptr;     // [tiles] steps completed per 8-chain tile within a launch (linear_dmma_kernel.cu)
    int64_t step_index = 0, welford_n = 0, am_steps = 0;
    int last_grid = 0, last_block = 0, last_smem = 0;
    int64_t launches = 0;
};

// kernels' host launchers (lv_kernel.cu, generic_kernel.cu, diag_kernels.cu)
int yg_launch_lv(yg_ensemble *e, const RunArgs &a, cudaStream_t st);
int yg_launch_generic(yg_ensemble *e, const RunArgs &a, cudaStream_t st);
int yg_launch_logpost(yg_ensemble *e, int level, const double *theta, int64_t n, double *out, cudaStream_t st);
int yg_launch_linear_big(yg_ensemble *e, const RunArgs &a, cudaStream_t st);
int yg_launch_logpost_big(yg_ensemble *e, int level, const double *theta, int64_t n, double *out, cudaStream_t st);
int yg_dmma_peak(int device, double ms, double *tflops_out);
