#pragma once
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "w4a8_gemm.h"  // error codes

namespace ob {

constexpr int MOE_MAX_EXPERTS = 64;   // experts per layer the routing kernels take
constexpr int MOE_MAX_TOPK = 8;       // experts per token
constexpr int MOE_DEV_ROWS = 64;      // rows per expert the device-offset grouped GEMM serves (one 64-row token tile)

// The rows the device-offset grouped GEMM gives slot (== expert) g from the offsets table: [off_g, off_g1) clamped to
// [0, total_rows], made non-decreasing, and cut at one 64-row tile.  A malformed table yields wrong rows, never an address
// outside the activation / output rows.  Shared by the kernel and by the host-only plan query.
__host__ __device__ inline void moe_slot_rows(int off_g, int off_g1, int total_rows, int* row0, int* rows) {
  const int lo = off_g < 0 ? 0 : (off_g > total_rows ? total_rows : off_g);
  const int hi = off_g1 < lo ? lo : (off_g1 > total_rows ? total_rows : off_g1);
  *row0 = lo;
  *rows = hi - lo < MOE_DEV_ROWS ? hi - lo : MOE_DEV_ROWS;
}

// Router logits (mixtral_w4a8_unpad.py:277,305, `self.gate(hidden_states).float()`): logits[t, e] = fp16(sum_h x[t,h] *
// wg[e,h]) held in fp32.  Fixed reduction order per (t, e), independent of T and of the other rows.
int moe_router_logits_run(const __half* x, const __half* wg, float* logits, int T, int H, int E, cudaStream_t st);
// Top-k softmax routing + stable counting sort by expert (moe_helpers.moe_topk_gating_softmax, :315).  One CTA.
int moe_topk_sort_run(const float* logits, float* weights, int* expert_indices, int* perm, int* offsets, int T, int E, int k,
                      cudaStream_t st);
// Gather of the per-token INT8 rows, scales and sums into permuted order (moe_expand_inputs_and_scales, :345).
int moe_expand_run(const int8_t* q, const __half* ssums /*nullable*/, const __half* scales, const int* perm, int8_t* q_out,
                   __half* ssums_out /*nullable*/, __half* scales_out, int* inv, int T, int k, int H, cudaStream_t st);
// Weighted combine of the k expert rows of every token (moe_finalize_routing, :388).
int moe_finalize_run(const __half* y, const float* weights, const int* inv, __half* out, int T, int k, int H, int ldy,
                     cudaStream_t st);

}  // namespace ob
