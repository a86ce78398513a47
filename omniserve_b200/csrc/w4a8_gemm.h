#pragma once
#include <cuda.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/omniserve_b200.h"  // OB_ERR_* codes

namespace ob {

struct W4A8GemmArgs {
  const int8_t* in_feats;    // [M, K] int8 row-major
  const int8_t* qweight;     // [N, K/2] int8 in the reference tile layout
  const int8_t* s2_scales;   // per-group only: [K/128, N]
  const int8_t* s2_zeros;    // per-group only: [K/128, N]  (= -z*s2, two's complement)
  const __half* wscales;     // [N]
  const __half* ascales;     // [M]
  const __half* w_szs;       // per-channel only: [N]
  const __half* a_ssums;     // per-channel only: [M]
  __half* out_feats;         // [M, ldc]
  int M, N, K, ldc;
  int force_bn = 0;          // testing knobs: 0 = auto
  int force_mode = -1;       // -1 auto, 0 = data-parallel tiles, 1 = stream-K
  int force_ctas = 0;
  // optional fused tail (extension): hidden_out = hidden_in + out_feats (fp16), then rms_norm_general(_fuse_sum) of it
  const __half* tail_hidden_in = nullptr;   // [M, N]
  __half* tail_hidden_out = nullptr;        // [M, N]
  const __half* tail_gamma = nullptr;       // [N]
  int8_t* tail_q = nullptr;                 // [M, N]
  __half* tail_scale = nullptr;             // [M]
  __half* tail_sum = nullptr;               // [M] or null
  float tail_eps = 0.f;
};

int w4a8_gemm_run(const W4A8GemmArgs& a, bool per_group, cudaStream_t st);

// Decode-specialised kernel (w4a8_gemm_decode.cu): M <= 64, small enough (<= 113 KB shared memory, 256 tensor-memory
// columns, <= 80 registers) for two CTAs per SM -- of the same GEMM, or of this GEMM and its PDL-launched successor.
// force_ctas = grid override (0 = auto).  Returns OB_ERR_SHAPE for shapes it does not take (caller falls back).
int w4a8_gemm_decode_run(const W4A8GemmArgs& a, bool per_group, cudaStream_t st);
int w4a8_gemm_decode_plan(int M, int N, int K, int sms, int ctas_per_sm, int use_cluster, int* bn, int* units_per_cta, int* grid,
                          int* cluster_s);

// Grouped (mixture-of-experts) W4A8 per-channel GEMM (w4a8_gemm_decode.cu), see include/omniserve_b200.h.
int w4a8_moe_gemm_run(const int8_t* x, const int8_t* qweight, const __half* wscales, const __half* ascales, const __half* w_szs,
                      const __half* a_ssums, __half* out, const int* problem_sizes_host, int num_experts, int T, int N, int K,
                      int ldc, cudaStream_t st);
// Same GEMM with the expert row ranges in DEVICE memory (offsets [E+1]), at most 64 rows per expert: no host read-back, CUDA-graph
// capturable.  total_rows = rows of x / out.  w4a8_moe_dev_plan: host-only view of its schedule for an offsets table.
int w4a8_moe_gemm_dev_run(const int8_t* x, const int8_t* qweight, const __half* wscales, const __half* ascales, const __half* w_szs,
                          const __half* a_ssums, __half* out, const int* offsets, int num_experts, int total_rows, int N, int K,
                          int ldc, cudaStream_t st);
int w4a8_moe_dev_plan(int num_experts, int N, int K, int sms, const int* offsets_host, int total_rows, int* grid, int* tiles_per_cta,
                      int* entries, int max_entries);

// W8A8 GEMM (w8a8_gemm.cu): out = (in . W^T) * wscales[n] * ascales[m], W plain row-major [N, K] int8.
int w8a8_gemm_run(const int8_t* in_feats, const int8_t* weight, const __half* wscales, const __half* ascales, __half* out,
                  int M, int N, int K, int ldc, cudaStream_t st);

// ---- shared host-side helpers (w4a8_gemm.cu)
int make_act_map(CUtensorMap* out, const void* ptr, int M, int K, int BN);          // [M, K] int8, box {128, BN}, SW128
int make_w_map(CUtensorMap* out, const void* ptr, int N, int K, bool rows2k);       // packed W4 tiles, 8 KB per box
int dev_sms(int dev);
// split-K workspace of (device, stream): ws = [2 * #SMs][64 * 128] int32 (== [#SMs][128 * 128]), zero between launches;
// cnt = GEMM_CNT_INTS(#SMs) int32 arrival counters, zero between launches
#define GEMM_CNT_INTS(sms) (4 * (sms) + 8)
int get_workspace(int dev, cudaStream_t st, int32_t** ws, int32_t** cnt);

}  // namespace ob
