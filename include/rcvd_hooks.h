/* rcvd_hooks.h -- test / bench hooks exported by librcvd_b200.so.  NOT part of the drop-in boundary (include/rcvd.h):
 * nothing in the reference corresponds to these; tests/, bench.py and tools/ use them to look inside the solver. */
#ifndef RCVD_HOOKS_H_
#define RCVD_HOOKS_H_
#include "rcvd.h"
#ifdef __cplusplus
extern "C" {
#endif

/* kernels launched so far by this handle / by the filter / by the constraint builder (the "did the CUDA path run" evidence) */
int64_t rcvd_launch_count(rcvd_problem* p);
int64_t rcvd_filter_launch_count(void);
int64_t rcvd_builder_launch_count(void);
int64_t rcvd_static_flag_launch_count(void);
int64_t rcvd_builder_last_rounds(void);          /* selection rounds of the last rcvd_build_constraints call */

/* {frames, off-diagonal factor blocks, levels, H blocks, npad, stride, tiles, update tasks} */
int32_t rcvd_structure_info(rcvd_problem* p, int32_t out[8]);

/* y = (S H S + diag(D2))^-1 b with the current H (exercises factorisation + substitution alone) */
int32_t rcvd_debug_linear_solve(rcvd_problem* p, const double* S, const double* D2, const double* b, double* y);

/* one damped LM step at the current state with trust-region `radius`; out = {|(S H S + D2) y - S g| / |S g| (device SpMV over the
 * assembled H), |S g|, cost, |g|_2, |y|_2, non-positive-pivot flag}: the parity evidence bench.py prints at the size it times */
int32_t rcvd_debug_linear_residual(rcvd_problem* p, double radius, double out[6]);

/* what the last step of rcvd_time_iteration computed, in the caller's frame order (N x stride doubles each): the gradient at the
 * state, the LM step and the candidate state (state + step, projected onto the bounds); costs = {cost at the state, candidate cost} */
int32_t rcvd_debug_iteration_outputs(rcvd_problem* p, double* gradient, double* step, double* candidate, double costs[2]);

/* per-kernel-class device time of one factorisation + solve: out_ms[0..5] = load, potrf, trinv, trsm, update GEMM,
 * substitution; [6] = update-GEMM launches, [7] = their algorithmic flops.  reps > 0: serialised on one stream;
 * reps < 0: two-stream overlap kept, main-stream view. */
int32_t rcvd_debug_profile_linear(rcvd_problem* p, int32_t reps, double out_ms[8]);
/* per-level view of the last rcvd_debug_profile_linear call: out[level][6] ms of {load, potrf, trinv, trsm, update, substitution} */
int32_t rcvd_debug_level_profile(rcvd_problem* p, double* out, int32_t max_levels);
/* fp64 tensor-core (DMMA) peak of the device in TFLOP/s, measured live */
int32_t rcvd_debug_fp64_tensor_peak(int32_t device, double* tflops);

/* A/B switches (defaults in parentheses) */
int32_t rcvd_debug_set_fast_path(rcvd_problem* p, int32_t on);        /* (1) specialised accumulate kernel */
int32_t rcvd_debug_set_overlap(rcvd_problem* p, int32_t on);          /* (1) two-stream factorisation graph */
int32_t rcvd_debug_set_trsm_ll(rcvd_problem* p, int32_t on);          /* (1) left-looking tensor-core TRSM */
int32_t rcvd_debug_set_order_slack(rcvd_problem* p, int32_t slack);   /* (4) multiple-elimination degree slack; -1 greedy */
int32_t rcvd_debug_set_trim_gemm(rcvd_problem* p, int32_t on);        /* (1) update GEMMs skip the zero padding beyond ceil8(unknowns) */
int32_t rcvd_debug_set_potrf_chain_warp(rcvd_problem* p, int32_t on); /* (1) warp 0 of k_potrf_smem is dedicated to the pivot chain; bit 1 set: round-1 shuffle Cholesky of the 16x16 pivot tile */
int32_t rcvd_debug_set_fused_substitution(rcvd_problem* p, int32_t on); /* (1) forward + backward substitution of the narrow levels as one persistent dataflow kernel; 0 = level-scheduled GEMV launches; n > 1: levels of <= n tasks per phase */
int32_t rcvd_debug_set_eval_only(rcvd_problem* p, int32_t on);        /* (0) cost / gradient evaluations only: no matrix storage (the whole-problem check of a multi-GPU bench) */
int32_t rcvd_debug_set_distributed(rcvd_problem* p, int32_t on);      /* (1) nranks > 1: distributed factorisation; 0 = all-reduce H + replicated factorisation */
int32_t rcvd_distribution_info(rcvd_problem* p, int32_t out[4]);       /* {distributed, first replicated level, levels, frames owned by this rank} */
int32_t rcvd_debug_set_side_slice(rcvd_problem* p, int32_t ctas);     /* (0) grid cap of one overlapped update launch */
int32_t rcvd_debug_set_update_kernel(rcvd_problem* p, int32_t tma, int32_t side_items_per_cta); /* (1, 0) persistent TMA-fed update kernel / round-1 cp.async kernel; items-per-CTA cap of overlapped launches */

#ifdef __cplusplus
}
#endif
#endif /* RCVD_HOOKS_H_ */
