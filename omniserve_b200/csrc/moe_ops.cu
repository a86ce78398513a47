// Mixture-of-experts routing, permutation and combine for sm_100a: the ops the reference's Mixtral block calls but never
// released (omniserve/modeling/models/mixtral_w4a8_unpad.py:300-395, `moe_helpers.*`).  Semantics are pinned by
// oracle/moe.py.  Every kernel is deterministic (no atomics whose order shows in a result) and row-independent: a token's
// router logits, expert choice, weights and combined output do not depend on which other tokens share the launch.
//
//   moe_router_logits   one CTA per token row, one warp per expert: fp32 FMA chain per lane + fixed xor butterfly
//   moe_topk_sort       ONE CTA: softmax + top-k per token, histogram, exclusive scan, stable counting-sort scatter
//   moe_expand          one CTA per permuted row: 16-byte gather of the INT8 row + its scale / sum
//   moe_finalize        one CTA per token: out = fp16(sum_j w_j * y[row_j]) in fp32, j ascending
#include "launch.h"
#include "moe_ops.h"
#include "ptx.cuh"

#include <math.h>

namespace ob {
namespace {

union H8 {
  uint4 u;
  __half h[8];
};

OB_DEVICE float warp_sum32(float v) {
#pragma unroll
  for (int m = 16; m >= 1; m >>= 1) v += __shfl_xor_sync(0xffffffffu, v, m);
  return v;
}

constexpr int ROUTER_THREADS = 256;

__global__ void __launch_bounds__(ROUTER_THREADS) router_logits_kernel(const __half* __restrict__ x, const __half* __restrict__ wg,
                                                                       float* __restrict__ logits, int H, int E) {
  pdl_trigger();
  pdl_wait();
  const size_t t = blockIdx.x;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int nvec = H >> 3;
  const uint4* xr = reinterpret_cast<const uint4*>(x + t * H);
  for (int e = warp; e < E; e += ROUTER_THREADS / 32) {
    const uint4* wr = reinterpret_cast<const uint4*>(wg + (size_t)e * H);
    float acc = 0.f;
    for (int i = lane; i < nvec; i += 32) {
      H8 a, b;
      a.u = xr[i];
      b.u = wr[i];
#pragma unroll
      for (int j = 0; j < 8; ++j) acc = __fmaf_rn(__half2float(a.h[j]), __half2float(b.h[j]), acc);
    }
    acc = warp_sum32(acc);
    if (lane == 0) logits[t * E + e] = __half2float(__float2half_rn(acc));   // the fp16 nn.Linear output, then .float()
  }
}

constexpr int SORT_THREADS = 1024;

// Routing of one token: softmax over the E logits (fp32, expf, sums in expert order), the k most probable experts by
// repeated arg-max (strict '>' over ascending indices: ties go to the lower index; slots come out in descending p), and
// Mixtral's renormalised weights p_sel / sum(p_sel).
OB_DEVICE void route_token(const float* lr, int E, int k, float* w_out, int* e_out) {
  float m = -INFINITY;
  for (int e = 0; e < E; ++e) m = fmaxf(m, lr[e]);
  float s = 0.f;
  for (int e = 0; e < E; ++e) s += expf(lr[e] - m);
  uint64_t taken = 0;
  float psel[MOE_MAX_TOPK];
  int esel[MOE_MAX_TOPK];
#pragma unroll
  for (int j = 0; j < MOE_MAX_TOPK; ++j) {
    psel[j] = 0.f;
    esel[j] = 0;
    if (j < k) {
      int best = -1;
      float bp = 0.f;
      for (int e = 0; e < E; ++e) {
        if ((taken >> e) & 1ull) continue;
        const float p = expf(lr[e] - m) / s;
        if (best < 0 || p > bp) { best = e; bp = p; }
      }
      taken |= 1ull << best;
      psel[j] = bp;
      esel[j] = best;
    }
  }
  float ps = 0.f;
#pragma unroll
  for (int j = 0; j < MOE_MAX_TOPK; ++j)
    if (j < k) ps += psel[j];
#pragma unroll
  for (int j = 0; j < MOE_MAX_TOPK; ++j)
    if (j < k) { w_out[j] = psel[j] / ps; e_out[j] = esel[j]; }
}

__global__ void __launch_bounds__(SORT_THREADS) topk_sort_kernel(const float* __restrict__ logits, float* __restrict__ weights,
                                                                 int* __restrict__ idx, int* __restrict__ perm,
                                                                 int* __restrict__ offsets, int T, int E, int k) {
  __shared__ int cnt[MOE_MAX_EXPERTS];                        // histogram, then the running cursor of each expert
  __shared__ int wcnt[SORT_THREADS / 32][MOE_MAX_EXPERTS];    // per-warp counts of a chunk, then the warp's base position
  pdl_trigger();
  pdl_wait();
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  if (tid < E) cnt[tid] = 0;
  __syncthreads();
  // 1. route every token; the histogram is an integer count, so the order of the shared-memory atomics does not show
  for (int t = tid; t < T; t += SORT_THREADS) {
    float w[MOE_MAX_TOPK];
    int e[MOE_MAX_TOPK];
    route_token(logits + (size_t)t * E, E, k, w, e);
#pragma unroll
    for (int j = 0; j < MOE_MAX_TOPK; ++j) {
      if (j < k) {
        weights[(size_t)t * k + j] = w[j];
        idx[(size_t)t * k + j] = e[j];
        atomicAdd(&cnt[e[j]], 1);
      }
    }
  }
  __syncthreads();
  // 2. exclusive scan -> expert_offsets; cnt becomes each expert's write cursor
  if (tid == 0) {
    int run = 0;
    for (int e = 0; e < E; ++e) {
      const int c = cnt[e];
      offsets[e] = run;
      cnt[e] = run;
      run += c;
    }
    offsets[E] = run;
  }
  __syncthreads();
  // 3. stable scatter, SORT_THREADS flat entries (t * k + j ascending) per chunk: an entry's position is its expert's cursor
  //    + the entries of the same expert in lower warps of the chunk + those in lower lanes of its warp
  const int n = T * k;
  for (int base = 0; base < n; base += SORT_THREADS) {
    for (int i = tid; i < (SORT_THREADS / 32) * MOE_MAX_EXPERTS; i += SORT_THREADS) (&wcnt[0][0])[i] = 0;
    const int i = base + tid;
    const int e = i < n ? idx[i] : -1;        // written by this CTA in step 1 (ordered by the barriers)
    const unsigned same = __match_any_sync(0xffffffffu, e);
    const int rank = __popc(same & ((1u << lane) - 1u));
    __syncthreads();
    if (e >= 0 && rank == 0) wcnt[warp][e] = __popc(same);
    __syncthreads();
    if (tid < E) {
      int run = cnt[tid];
      for (int w = 0; w < SORT_THREADS / 32; ++w) {
        const int c = wcnt[w][tid];
        wcnt[w][tid] = run;
        run += c;
      }
      cnt[tid] = run;
    }
    __syncthreads();
    if (e >= 0) perm[wcnt[warp][e] + rank] = i;
    __syncthreads();
  }
}

constexpr int EXPAND_THREADS = 128;

__global__ void __launch_bounds__(EXPAND_THREADS) expand_kernel(const int8_t* __restrict__ q, const __half* __restrict__ ssums,
                                                                const __half* __restrict__ scales, const int* __restrict__ perm,
                                                                int8_t* __restrict__ q_out, __half* __restrict__ ssums_out,
                                                                __half* __restrict__ scales_out, int* __restrict__ inv, int n,
                                                                int k, int H) {
  pdl_trigger();
  pdl_wait();
  const int r = blockIdx.x;
  const int src = perm[r];
  if (src < 0 || src >= n) return;   // not a permutation entry: leave the row alone
  const size_t t = (size_t)(src / k);
  const uint4* s = reinterpret_cast<const uint4*>(q + t * H);
  uint4* d = reinterpret_cast<uint4*>(q_out + (size_t)r * H);
  for (int i = threadIdx.x; i < (H >> 4); i += EXPAND_THREADS) d[i] = s[i];
  if (threadIdx.x == 0) {
    scales_out[r] = scales[t];
    if (ssums) ssums_out[r] = ssums[t];
    inv[src] = r;
  }
}

constexpr int FIN_THREADS = 128;

__global__ void __launch_bounds__(FIN_THREADS) finalize_kernel(const __half* __restrict__ y, const float* __restrict__ weights,
                                                               const int* __restrict__ inv, __half* __restrict__ out, int n,
                                                               int k, int H, int ldy) {
  pdl_trigger();
  pdl_wait();
  const size_t t = blockIdx.x;
  size_t row[MOE_MAX_TOPK];
  float w[MOE_MAX_TOPK];
#pragma unroll
  for (int j = 0; j < MOE_MAX_TOPK; ++j) {
    row[j] = 0;
    w[j] = 0.f;
    if (j < k) {
      const int r = inv[t * k + j];
      row[j] = (size_t)(r < 0 ? 0 : (r >= n ? n - 1 : r));
      w[j] = weights[t * k + j];
    }
  }
  for (int i = threadIdx.x; i < (H >> 3); i += FIN_THREADS) {
    float acc[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
#pragma unroll
    for (int j = 0; j < MOE_MAX_TOPK; ++j) {
      if (j < k) {
        H8 v;
        v.u = reinterpret_cast<const uint4*>(y + row[j] * ldy)[i];
#pragma unroll
        for (int c = 0; c < 8; ++c) acc[c] = __fadd_rn(acc[c], __fmul_rn(w[j], __half2float(v.h[c])));
      }
    }
    H8 o;
#pragma unroll
    for (int c = 0; c < 8; ++c) o.h[c] = __float2half_rn(acc[c]);
    reinterpret_cast<uint4*>(out + t * H)[i] = o.u;
  }
}

bool misaligned(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) != 0; }

}  // namespace

int moe_router_logits_run(const __half* x, const __half* wg, float* logits, int T, int H, int E, cudaStream_t st) {
  if (T <= 0) return 0;
  if (H <= 0 || H % 8 != 0 || E <= 0 || E > MOE_MAX_EXPERTS) return OB_ERR_SHAPE;
  if (misaligned(x) || misaligned(wg)) return OB_ERR_ALIGN;
  return launch_pdl(router_logits_kernel, dim3(T), dim3(ROUTER_THREADS), 0, st, x, wg, logits, H, E) == cudaSuccess ? 0 : OB_ERR_CUDA;
}

int moe_topk_sort_run(const float* logits, float* weights, int* expert_indices, int* perm, int* offsets, int T, int E, int k,
                      cudaStream_t st) {
  if (T < 0 || E <= 0 || E > MOE_MAX_EXPERTS || k < 1 || k > MOE_MAX_TOPK || k > E) return OB_ERR_SHAPE;
  if ((long long)T * k > (1LL << 30)) return OB_ERR_SHAPE;
  return launch_pdl(topk_sort_kernel, dim3(1), dim3(SORT_THREADS), 0, st, logits, weights, expert_indices, perm, offsets, T, E, k) ==
                 cudaSuccess ? 0 : OB_ERR_CUDA;
}

int moe_expand_run(const int8_t* q, const __half* ssums, const __half* scales, const int* perm, int8_t* q_out, __half* ssums_out,
                   __half* scales_out, int* inv, int T, int k, int H, cudaStream_t st) {
  if (T <= 0) return 0;
  if (k < 1 || k > MOE_MAX_TOPK || H <= 0 || H % 16 != 0 || (long long)T * k > (1LL << 30)) return OB_ERR_SHAPE;
  if ((ssums == nullptr) != (ssums_out == nullptr)) return OB_ERR_ARG;
  if (misaligned(q) || misaligned(q_out)) return OB_ERR_ALIGN;
  return launch_pdl(expand_kernel, dim3(T * k), dim3(EXPAND_THREADS), 0, st, q, ssums, scales, perm, q_out, ssums_out, scales_out, inv,
                    T * k, k, H) == cudaSuccess ? 0 : OB_ERR_CUDA;
}

int moe_finalize_run(const __half* y, const float* weights, const int* inv, __half* out, int T, int k, int H, int ldy,
                     cudaStream_t st) {
  if (T <= 0) return 0;
  if (k < 1 || k > MOE_MAX_TOPK || H <= 0 || H % 8 != 0 || ldy < H || ldy % 8 != 0 || (long long)T * k > (1LL << 30))
    return OB_ERR_SHAPE;
  if (misaligned(y) || misaligned(out)) return OB_ERR_ALIGN;
  return launch_pdl(finalize_kernel, dim3(T), dim3(FIN_THREADS), 0, st, y, weights, inv, out, T * k, k, H, ldy) == cudaSuccess
             ? 0 : OB_ERR_CUDA;
}

}  // namespace ob
