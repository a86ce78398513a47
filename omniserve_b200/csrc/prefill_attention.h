#pragma once
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "w4a8_gemm.h"  // error codes

namespace ob {

// Token-streaming ("Lambda"-masked) causal prefill attention of LServe's streaming heads, fp16, head_dim 128.
// Query position i of a sequence attends key j  iff  j <= i  and  (j < sink  or  i - j < local).
struct StreamingPrefillArgs {
  const __half* q; const __half* k; const __half* v;   // [T, Hq, 128] / [T, Hkv, 128] views; head stride 128
  long long q_row_stride, k_row_stride, v_row_stride;   // token strides in elements
  __half* out;                                          // [T, Hq, 128] contiguous; only computed heads are written
  const int* cu_seqlens_host;                           // HOST [B + 1]
  int B, T, Hq, Hkv, head_dim;
  int num_compute_heads;                                // kv heads to compute (<= SP_MAX_HEADS)
  const int* kv_heads_host;                             // HOST [num_compute_heads]: kv head index
  const int* sink_host; const int* local_host;          // HOST [num_compute_heads]: (sink, local) of that kv group
};

int streaming_prefill_run(const StreamingPrefillArgs& a, cudaStream_t st);

// Host-only view of the launch plan (no CUDA call).  out[0] launches, out[1] grid.x / out[2] grid.y of launch `launch`,
// out[3] sequence, out[4] / out[5] first / last query position of CTA (cta_x, cta_y) within the sequence, out[6] kv head,
// out[7] key tiles of 64 the CTA visits (their indices go to key_tiles[0 .. min(out[7], max_key_tiles))).
int streaming_prefill_plan(const StreamingPrefillArgs& a, int launch, int cta_x, int cta_y, int* out, int* key_tiles,
                           int max_key_tiles);

}  // namespace ob
