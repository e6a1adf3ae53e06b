// big_linear.h -- device problem blob of the large linear model (linear_dmma_kernel.cu):
// d up to YG_BIG_MAX_DIM, data_dim up to YG_BIG_MAX_DATA_DIM, diagonal noise; diagonal or dense prior precision and
// proposal factor.
#pragma once
#include <stdint.h>
#include "../../include/yagre_b200.h"

struct BigLevel {
    int32_t n_data, data_dim, np, n_rows;           // n_rows = rows of the GEMM operand: data_dim (+ dim when a dense prior
                                                    // precision is folded in as extra rows); np = n_rows rounded up to 16
    int32_t G_off, bd_off, pmean_off, pprec_off;    // offsets (doubles) into the tail
    double q_const, _pad3;                          // sum_col prec_col * sum_rows (d_row,col - mean_col)^2
};

struct DevBigHeader {
    int32_t dim, kp, ks, n_levels;                  // kp in {16, 32, 64} >= dim; ks = kp + 4 (row stride of G)
    int32_t J, tail_len, propL_off, proposal;       // proposal: yg_proposal
    int32_t pcn_mean_off, dense_L, Ld_off, stream;  // dense_L: the proposal factor is a full lower triangle Ld[kp][ks];
                                                    // stream: BigStream bits (smem_plan.h) of the operands the step
                                                    // kernel reads from this global copy instead of shared memory
    double pcn_a, pcn_b;                            // sqrt(1 - 2h), sqrt(2h)   (pcn.py:30-35)
    BigLevel lvl[3];                                // up to two surrogates and the target
    double _pad[2];
    // followed by double tail[tail_len]: per level
    //   Gw[np][ks] = sqrt(w_row) G_row,  bdw[np] = sqrt(w_row) (b_row - mean over the data rows),  w = n_data * noise
    //   precision (the weights are folded into the operands once on the host, so the accumulator epilogue is one add
    //   and one FMA per element), pmean[kp], pprec[kp];
    // A TEMPERED level (tempering t * logL + logprior, target.py:40-43) has fl(sqrt(t)) folded into the same data rows
    //   as one more factor of sqrt(w_row), and q_const multiplied by t; its prior rows are left alone.  t = 1 leaves
    //   every operand as it is untempered, t = 0 makes the data rows zero.
    // A DENSE prior precision P = R'R (R = chol(P)') is folded into the same operands as d more rows:
    //   Gw[data_dim + r] = R_r,  bdw[data_dim + r] = -(R m)_r,  pprec = 0:  ||R (theta - m)||^2 = (theta - m)' P (theta - m).
    // then propL[kp] (diagonal of the factor), pcn_mean[kp] and, for a dense factor, Ld[kp][ks].  Padding is zero.
    // When the plan streams operands (big_tensor_plan), the same items are laid out without the streamed ones up to
    // the staged prefix of BigTensorPlan::resident doubles, and the streamed ones follow it, 32-byte aligned, level 1's
    // G before level 2's before Ld; the offsets above say where every item is.
    // sum_rows ||F - d_row||^2_P = sum_col w_col (F_col - mean_col)^2 + q_const.
};
static_assert(sizeof(DevBigHeader) % 32 == 0, "header must keep the tail on 32-byte sectors (streamed operands)");

// Welford second moment of the large model is diagonal only (like the reference's
// WelfordAccumulator, statistics/estimation.py:4-58): w_m2 is [d, n] when d > YG_MAX_DIM and the
// diagonal of the [d, d, n] layout otherwise.
__host__ __device__ inline int big_w2_index(int k, int d) { return d > YG_MAX_DIM ? k : k * d + k; }
