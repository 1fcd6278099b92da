/*
 * icpcuda_debug.h - introspection and micro-benchmark entry points of libicpcuda.so used by bench.py, tools/ and the
 * tests. NOT part of the drop-in boundary (include/icpcuda.h): a Scala/Panama binding has no use for them.
 */
#ifndef ICPCUDA_DEBUG_H
#define ICPCUDA_DEBUG_H

#include "icpcuda.h"

#ifdef __cplusplus
extern "C" {
#endif

/* Philox4x32-10 block as the chain runner draws it: out[4] for (seed, chain, step, block) */
int32_t icp_debug_philox(icp_ctx ctx, uint64_t seed, uint64_t chain, uint32_t step, uint32_t block, uint32_t out[4]);
/* measured FP64 peaks of this device (TFLOP/s): out[0] = DFMA (CUDA cores), out[1] = DMMA m8n8k4 */
int32_t icp_debug_fp64_peak(icp_ctx ctx, double out[2]);
/* DMMA issue-rate experiment: TFLOP/s of mma.sync.m8n8k4.f64 with warps_per_cta x ctas_per_sm resident warps per SM and
 * nacc (1, 2, 4, 8) independent accumulators per warp */
int32_t icp_debug_dmma_sweep(icp_ctx ctx, int32_t warps_per_cta, int32_t ctas_per_sm, int32_t nacc, double *tflops);
/* eager (graph-less) run of n_steps of the chain with every kernel class bracketed by CUDA events on
 * the library stream: stage_ms[ICP_N_STAGES] summed device milliseconds, stage_launches[ICP_N_STAGES]
 * number of launches. Stage names through icp_stage_name. theta0 is host memory, Philox RNG. */
#define ICP_N_STAGES 11
int32_t icp_chain_profile(icp_chain c, int32_t C, int32_t n_steps, const double *theta0, uint64_t seed,
                          double *stage_ms, int64_t *stage_launches);
const char *icp_stage_name(int32_t stage);
/* closest-point traversal timed in isolation: average milliseconds per launch over `iters` launches of
 * nq device-resident queries (CUDA events on the library stream, after one warm-up launch) */
int32_t icp_debug_time_closest_point(icp_target t, int64_t nq, const double *q_dev, int32_t *tri_dev, double *cp_dev,
                                     double *d2_dev, int32_t iters, double *ms);

/* L2 -> SM read bandwidth (GB/s) of this device over a working set of the given size that stays resident in L2 (L1
 * bypassed, 16-byte loads): the roofline denominator of the cache-resident closest-point traversal (SURVEY 8d) */
int32_t icp_debug_l2_bandwidth(icp_ctx ctx, int64_t working_set_bytes, double *gbps);

/* tcgen05 INT8 self-test / micro-benchmark (csrc/tc_i8.cu): D (128 x 128 row-major int32, columns < 112 valid) = A^T A of an
 * int8 matrix A (rows x 128 row-major, rows a multiple of 32) through tcgen05.mma kind::i8 with the accumulator in TMEM; then
 * `ctas` CTAs repeat the product `iters` times and *ms is the device time of that launch (MMA rate of the rank update's
 * tile shape M = 128, N = 112, K = 32). */
int32_t icp_debug_i8_gram(icp_ctx ctx, int32_t rows, const int8_t *A, int32_t *D, int32_t iters, int32_t ctas, double *ms);

/* Posterior factorisation of C host matrices M (C x K x K, symmetric) and right-hand sides b (C x K) on the device path the
 * posterior pipeline takes at rank K. ymean = 0: mean = mu = M^-1 b (icp_posterior's form); ymean = 1: mean = y = L^-1 b, the
 * chain runner's form, which skips the back substitution. L: lower triangle of the Cholesky factor (C x K x K). q (nullable):
 * |L^T (w - mu)|^2 per matrix, w = theta_post + (theta_other - theta_post) / step over the coefficients (theta_* C x (K + 10)),
 * formed as the chain runner forms its backward transition form. status[c] != 0: M_c was not positive definite. */
int32_t icp_debug_factor(icp_ctx ctx, int32_t C, int32_t K, const double *M, const double *b, const double *theta_post,
                         const double *theta_other, double step, int32_t ymean, double *L, double *mean, double *q, int32_t *status);

/* The reference's covariance factor W = D^-1 Ubar diag(sqrt(lambda')) (ICP_FACTOR_SVD) of C posteriors from their Cholesky factors
 * L (C x K x K, lower triangle read) and the model variances (K), on the device path the proposal takes: W (C x K x K) and per
 * posterior the one-sided Jacobi sweeps that rotated (40, the cap, means the loop did not converge). tol <= 0: the library's
 * stopping threshold; > 0: that threshold instead. */
int32_t icp_debug_svd_factor(icp_ctx ctx, int32_t C, int32_t K, const double *L, const double *variance, double tol, double *W,
                             int32_t *sweeps);

/* Posterior schedule of the step-by-step chain runner (DESIGN.md section 5). The runner factors an ICP posterior of a state only
 * when a proposal from that state picks the component, or when a step's ICP transition terms are not certified negligible;
 * the chain log is bit-identical to the eager schedule's, which factors both posteriors of every proposal.
 * schedule for later runs from theta0: 0 the runner chooses (default), 1 eager, 2 lazy wherever it applies, also below the
 * chain count from which the runner chooses it; -1 unchanged.
 * lazy (nullable): whether the resident run uses the lazy schedule. counters (nullable) of the resident run, summed over the
 * steps of the last call: [0] posteriors factored when picked, [1] chain-steps that fell back to the eager factorisations,
 * [2] chain-steps certified (all zero under the eager schedule). */
int32_t icp_debug_chain_schedule(icp_chain c, int32_t schedule, int32_t *lazy, int64_t counters[3]);

#ifdef __cplusplus
}
#endif
#endif /* ICPCUDA_DEBUG_H */
