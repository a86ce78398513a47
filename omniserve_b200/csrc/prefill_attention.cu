// Token-streaming prefill attention: the context-stage attention of LServe's STREAMING heads, fp16 in, fp32 accumulate,
// fp16 out, head_dim 128, variable-length sequences packed along T.
//
// Mask ("Lambda" shape).  Query position i of a sequence (0-based within the sequence) attends key position j iff
//     j <= i   and   ( j < sink   or   i - j < local ).
// With sink + local >= i + 1 this is plain causal attention.  The boundary is the one the decode kernel uses for a
// streaming head (kv4_attention.cu: the sink plus the last `local` tokens, the current token included; reference
// decoderMaskedMultiheadAttentionTemplate.hpp:1570-1584), so a prompt prefilled here and then decoded sees one window.
// The third-party library the reference calls for this op (block_sparse_attn.token_streaming_attn_func) is not available
// to compare against, so whether its window is off by one from this definition is NOT checked.
//
// Work decomposition.  One CTA per (query tile, streaming kv head); it serves all g = Hq / Hkv query heads of the GQA group,
// so each K / V tile is staged once per group.  A CTA owns 128 (token, q-head) rows: QT = 128 / g query tokens x g heads,
// row r = (token q_lo + r / g, head r % g).  The grid is built on the host from cu_seqlens (no empty CTAs; up to
// SP_MAX_SEQ sequences per launch, query tiles of the latest positions -- the ones with full windows -- first).
//
//   * warp 0 also streams the 64-token K and V tiles of the kv head into a 4-stage shared-memory ring, STAGES - 1 tiles
//     ahead, with one cp.async.bulk per 256-byte row (the rows are strided views into the qkv activation) completing on
//     an mbarrier per stage; a CTA barrier after each tile frees its stage.  Rows are padded to 272 bytes so that the
//     ldmatrix reads below are conflict-free.  (A dedicated ninth producer warp would put three warps on one SM
//     sub-partition, whose 16K registers cannot hold three warps of this kernel's ~200 registers.)
//   * warps 0-7 each own 16 rows: S = Q.K^T with mma.sync.m16n8k16 (f16 x f16 -> f32), online softmax in fp32 with
//     exp2f and Dh^-1/2 * log2(e) folded into one scale, P rounded to fp16 for P.V (and for its row sums), the output
//     normalised in fp32 and rounded to fp16 once;
//   * the key-tile loop visits only the tiles that meet [0, sink) U [q_lo - local + 1, q_hi]; element masking runs only on
//     the tiles that straddle an edge of the mask.  Per query tile that is at most
//     ceil(sink / 64) + ceil((local + QT - 1) / 64) + 1 tiles, independent of the sequence length.
// No atomics: every output element is written once by one thread, in a fixed order -- the result is deterministic.
// Address arithmetic is 64-bit (T * row stride passes 2^31 at 1M tokens).
#include <stdio.h>

#include <algorithm>
#include <vector>

#include "launch.h"
#include "prefill_attention.h"
#include "ptx.cuh"

namespace ob {

namespace sp {

constexpr int DH = 128;
constexpr int KT = 64;                    // keys per tile
constexpr int ROWS = 128;                 // (token, head) rows per CTA
constexpr int WARPS = 8;                  // 16 rows each; warp 0 also issues the tile copies
constexpr int THREADS = WARPS * 32;
constexpr int STAGES = 4;
constexpr int PITCH = DH + 8;             // halfs per shared-memory row (272 B)
constexpr int TILE_HALFS = KT * PITCH;
constexpr int STAGE_BYTES = 2 * TILE_HALFS * 2;
constexpr int SMEM_BYTES = STAGES * STAGE_BYTES + STAGES * 8;
constexpr int MAX_SEQ = 64;
constexpr int MAX_HEADS = 64;

// The key tiles a query tile [q_lo, q_hi] visits: [0, a_end) then [b_begin, b_end) (b_begin >= a_end).
struct KeyTiles {
  int a_end, b_begin, b_end, n;
  __host__ __device__ void init(int q_lo, int q_hi, int sink, int local) {
    const int a_keys = sink < q_hi + 1 ? sink : q_hi + 1;
    a_end = (a_keys + KT - 1) / KT;
    const int lo_key = q_lo - local + 1 > 0 ? q_lo - local + 1 : 0;
    b_begin = lo_key / KT > a_end ? lo_key / KT : a_end;
    b_end = q_hi / KT + 1;
    n = a_end + (b_end > b_begin ? b_end - b_begin : 0);
  }
  __host__ __device__ int tile(int i) const { return i < a_end ? i : b_begin + (i - a_end); }
};

struct Params {
  const __half* q; const __half* k; const __half* v;
  long long qs, ks, vs;
  __half* out;
  int Hq, g, qt, nseq;
  float scale_log2;
  int tile_start[MAX_SEQ + 1];
  long long seq_tok0[MAX_SEQ];
  int seq_len[MAX_SEQ];
  int kvh[MAX_HEADS], sink[MAX_HEADS], local[MAX_HEADS];
};

struct Cta { int seq, q_lo, q_hi; };

// blockIdx.x -> (sequence, query tile); the latest query tiles (most key tiles) are scheduled first.
__host__ __device__ inline Cta locate(const Params& p, int bx, int gx) {
  const int tt = gx - 1 - bx;
  int s = 0;
  while (s + 1 < p.nseq && p.tile_start[s + 1] <= tt) ++s;
  Cta c;
  c.seq = s;
  c.q_lo = (tt - p.tile_start[s]) * p.qt;
  c.q_hi = (c.q_lo + p.qt < p.seq_len[s] ? c.q_lo + p.qt : p.seq_len[s]) - 1;
  return c;
}

OB_DEVICE void mma16816(float (&c)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
               : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
               : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
OB_DEVICE void ldsm_x4(uint32_t addr, uint32_t& r0, uint32_t& r1, uint32_t& r2, uint32_t& r3) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];"
               : "=r"(r0), "=r"(r1), "=r"(r2), "=r"(r3) : "r"(addr));
}
OB_DEVICE void ldsm_x4_t(uint32_t addr, uint32_t& r0, uint32_t& r1, uint32_t& r2, uint32_t& r3) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];"
               : "=r"(r0), "=r"(r1), "=r"(r2), "=r"(r3) : "r"(addr));
}
__global__ void __launch_bounds__(THREADS, 1) streaming_prefill_kernel(const __grid_constant__ Params p) {
  extern __shared__ __align__(128) uint8_t smem[];
  __half* tiles = reinterpret_cast<__half*>(smem);
  uint64_t* full = reinterpret_cast<uint64_t*>(smem + STAGES * STAGE_BYTES);
  pdl_trigger();
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const Cta c = locate(p, blockIdx.x, gridDim.x);
  const int len = p.seq_len[c.seq];
  const long long tok0 = p.seq_tok0[c.seq];
  const int hs = blockIdx.y;
  const int kvh = p.kvh[hs], S = p.sink[hs], W = p.local[hs];
  KeyTiles kt;
  kt.init(c.q_lo, c.q_hi, S, W);
  if (tid == 0) {
    for (int s = 0; s < STAGES; ++s) mbar_init(&full[s], 1);
    mbar_fence_init();
  }
  __syncthreads();
  pdl_wait();   // q / k / v are written by the kernels before this one

  const __half* kg = p.k + (long long)kvh * DH;
  const __half* vg = p.v + (long long)kvh * DH;
  // warp 0: copy key tile number `it` of the visit list into its stage (the stage's previous tile is finished by all warps)
  auto issue = [&](int it) {
    const int st = it % STAGES;
    const int k0 = kt.tile(it) * KT;
    const int n = len - k0 < KT ? len - k0 : KT;
    __half* kd = tiles + st * 2 * TILE_HALFS;
    __half* vd = kd + TILE_HALFS;
    if (n < KT) {   // the sequence ends inside the tile: zero the rest (masked, but 0 * NaN garbage would poison P.V)
      const uint4 z = make_uint4(0, 0, 0, 0);
      for (int i = lane; i < (KT - n) * (DH / 8); i += 32) {
        const int r = n + i / (DH / 8), c8 = (i % (DH / 8)) * 8;
        *reinterpret_cast<uint4*>(kd + r * PITCH + c8) = z;
        *reinterpret_cast<uint4*>(vd + r * PITCH + c8) = z;
      }
    }
    fence_proxy_async_smem();   // this stage's generic reads / writes before the bulk (async-proxy) writes into it
    __syncwarp();
    if (lane == 0) mbar_arrive_expect_tx(&full[st], (uint32_t)n * DH * 2 * 2);
    __syncwarp();
    for (int r = lane; r < n; r += 32) {
      const long long t = tok0 + k0 + r;
      bulk_g2s(kd + r * PITCH, kg + t * p.ks, DH * 2, &full[st]);
      bulk_g2s(vd + r * PITCH, vg + t * p.vs, DH * 2, &full[st]);
    }
  };
  if (warp == 0)
    for (int it = 0; it < STAGES - 1 && it < kt.n; ++it) issue(it);

  // ---------------------------------------------------------------------- compute warps
  const int g = p.g;
  const int r0 = warp * 16 + (lane >> 2), r1 = r0 + 8;
  const int i0 = c.q_lo + r0 / g, i1 = c.q_lo + r1 / g;          // query positions of this thread's two rows
  const int h0 = kvh * g + r0 % g, h1 = kvh * g + r1 % g;
  const int t_lo = c.q_lo + (warp * 16) / g;
  const int t_hi = min(c.q_lo + (warp * 16 + 15) / g, c.q_hi);   // last real query position of the warp
  const bool has_rows = t_lo <= c.q_hi;
  uint32_t qa[DH / 16][4];
  {
    const __half* q0 = p.q + (tok0 + min(i0, c.q_hi)) * p.qs + (long long)h0 * DH + 2 * (lane & 3);
    const __half* q1 = p.q + (tok0 + min(i1, c.q_hi)) * p.qs + (long long)h1 * DH + 2 * (lane & 3);
#pragma unroll
    for (int kk = 0; kk < DH / 16; ++kk) {
      qa[kk][0] = *reinterpret_cast<const uint32_t*>(q0 + 16 * kk);
      qa[kk][1] = *reinterpret_cast<const uint32_t*>(q1 + 16 * kk);
      qa[kk][2] = *reinterpret_cast<const uint32_t*>(q0 + 16 * kk + 8);
      qa[kk][3] = *reinterpret_cast<const uint32_t*>(q1 + 16 * kk + 8);
    }
  }
  float o[DH / 8][4];
#pragma unroll
  for (int j = 0; j < DH / 8; ++j) o[j][0] = o[j][1] = o[j][2] = o[j][3] = 0.f;
  float m0 = -INFINITY, m1 = -INFINITY, l0 = 0.f, l1 = 0.f;
  const uint32_t tiles_u32 = smem_u32(tiles);
  // ldmatrix lane offsets (bytes): K (non-transposed) and V (transposed) 8x8 blocks, see the fragment maps below
  const uint32_t k_off = (uint32_t)((((lane >> 4) * 8 + (lane & 7)) * PITCH + ((lane >> 3) & 1) * 8) * 2);
  const uint32_t v_off = (uint32_t)(((((lane >> 3) & 1) * 8 + (lane & 7)) * PITCH + (lane >> 4) * 8) * 2);

  for (int it = 0; it < kt.n; ++it) {
    const int st = it % STAGES;
    if (warp == 0 && it + STAGES - 1 < kt.n) issue(it + STAGES - 1);   // into the stage tile it - 1 used
    mbar_wait(&full[st], (it / STAGES) & 1);
    const int k0 = kt.tile(it) * KT, k1 = k0 + KT;
    const int jmax = min(k1 - 1, t_hi);
    const bool needed = has_rows && k0 <= t_hi && (k0 < S || t_lo - jmax < W);   // some (i, j) of the warp attended
    if (needed) {
      const bool unmasked = k1 - 1 <= t_lo && k1 <= len && (k1 <= S || t_hi - k0 < W);
      const uint32_t kb = tiles_u32 + st * STAGE_BYTES;
      const uint32_t vb = kb + TILE_HALFS * 2;
      float s[KT / 8][4];
#pragma unroll
      for (int j = 0; j < KT / 8; ++j) s[j][0] = s[j][1] = s[j][2] = s[j][3] = 0.f;
#pragma unroll
      for (int kk = 0; kk < DH / 16; ++kk) {
#pragma unroll
        for (int np = 0; np < KT / 16; ++np) {
          uint32_t b0, b1, b2, b3;   // keys 16np + [0,8) / [8,16), dims 16kk + [0,8) / [8,16)
          ldsm_x4(kb + k_off + (uint32_t)((16 * np * PITCH + 16 * kk) * 2), b0, b1, b2, b3);
          mma16816(s[2 * np], qa[kk], b0, b1);
          mma16816(s[2 * np + 1], qa[kk], b2, b3);
        }
      }
      float mx0 = -INFINITY, mx1 = -INFINITY;
#pragma unroll
      for (int j = 0; j < KT / 8; ++j) {
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          float x = s[j][e] * p.scale_log2;
          if (!unmasked) {
            const int kj = k0 + 8 * j + 2 * (lane & 3) + (e & 1);
            const int qi = e < 2 ? i0 : i1;
            if (!(kj <= qi && kj < len && (kj < S || qi - kj < W))) x = -INFINITY;
          }
          s[j][e] = x;
        }
        mx0 = fmaxf(mx0, fmaxf(s[j][0], s[j][1]));
        mx1 = fmaxf(mx1, fmaxf(s[j][2], s[j][3]));
      }
      mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, 1));
      mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, 2));
      mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, 1));
      mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, 2));
      const float mn0 = fmaxf(m0, mx0), mn1 = fmaxf(m1, mx1);
      const float base0 = mn0 == -INFINITY ? 0.f : mn0, base1 = mn1 == -INFINITY ? 0.f : mn1;
      const float al0 = exp2f(m0 - base0), al1 = exp2f(m1 - base1);
      m0 = mn0; m1 = mn1;
      float sum0 = 0.f, sum1 = 0.f;
      uint32_t pa[KT / 16][4];
#pragma unroll
      for (int j = 0; j < KT / 8; ++j) {
        const float p0 = exp2f(s[j][0] - base0), p1 = exp2f(s[j][1] - base0);
        const float p2 = exp2f(s[j][2] - base1), p3 = exp2f(s[j][3] - base1);
        // C fragment of key tile j -> A fragment of k-step j / 2 (keys 8j..8j+7 are its low or high k half); the row sums
        // take the same fp16-rounded weights that enter P.V, so the weights of a row sum to exactly one
        const __half2 h01 = __floats2half2_rn(p0, p1), h23 = __floats2half2_rn(p2, p3);
        sum0 += __low2float(h01) + __high2float(h01);
        sum1 += __low2float(h23) + __high2float(h23);
        pa[j >> 1][(j & 1) * 2 + 0] = *reinterpret_cast<const uint32_t*>(&h01);
        pa[j >> 1][(j & 1) * 2 + 1] = *reinterpret_cast<const uint32_t*>(&h23);
      }
      l0 = l0 * al0 + sum0; l1 = l1 * al1 + sum1;
#pragma unroll
      for (int j = 0; j < DH / 8; ++j) { o[j][0] *= al0; o[j][1] *= al0; o[j][2] *= al1; o[j][3] *= al1; }
#pragma unroll
      for (int kk = 0; kk < KT / 16; ++kk) {
#pragma unroll
        for (int dp = 0; dp < DH / 16; ++dp) {
          uint32_t b0, b1, b2, b3;   // keys 16kk + [0,8) / [8,16) x dims 16dp + [0,8) / [8,16), transposed
          ldsm_x4_t(vb + v_off + (uint32_t)((16 * kk * PITCH + 16 * dp) * 2), b0, b1, b2, b3);
          mma16816(o[2 * dp], pa[kk], b0, b1);
          mma16816(o[2 * dp + 1], pa[kk], b2, b3);
        }
      }
    }
    __syncthreads();   // every warp is done with this stage before warp 0 refills it
  }

  l0 += __shfl_xor_sync(0xffffffffu, l0, 1);
  l0 += __shfl_xor_sync(0xffffffffu, l0, 2);
  l1 += __shfl_xor_sync(0xffffffffu, l1, 1);
  l1 += __shfl_xor_sync(0xffffffffu, l1, 2);
  const float inv0 = l0 > 0.f ? 1.f / l0 : 0.f, inv1 = l1 > 0.f ? 1.f / l1 : 0.f;
  const long long ostride = (long long)p.Hq * DH;
  __half* out0 = p.out + (tok0 + i0) * ostride + (long long)h0 * DH + 2 * (lane & 3);
  __half* out1 = p.out + (tok0 + i1) * ostride + (long long)h1 * DH + 2 * (lane & 3);
#pragma unroll
  for (int j = 0; j < DH / 8; ++j) {
    if (i0 <= c.q_hi) *reinterpret_cast<__half2*>(out0 + 8 * j) = __floats2half2_rn(o[j][0] * inv0, o[j][1] * inv0);
    if (i1 <= c.q_hi) *reinterpret_cast<__half2*>(out1 + 8 * j) = __floats2half2_rn(o[j][2] * inv1, o[j][3] * inv1);
  }
}

// Validates the arguments and splits the batch into launches of <= MAX_SEQ sequences.
static int plan(const StreamingPrefillArgs& a, Params& base, std::vector<std::pair<int, int>>& launches) {
  if (a.head_dim != DH) return OB_ERR_SHAPE;
  if (a.B <= 0 || a.Hkv <= 0 || a.Hq <= 0 || a.Hq % a.Hkv) return OB_ERR_SHAPE;
  const int g = a.Hq / a.Hkv;
  if (ROWS % g) return OB_ERR_SHAPE;
  if (a.num_compute_heads < 0 || a.num_compute_heads > MAX_HEADS) return OB_ERR_SHAPE;
  if (!a.cu_seqlens_host || (a.num_compute_heads && (!a.kv_heads_host || !a.sink_host || !a.local_host))) return OB_ERR_ARG;
  if (a.cu_seqlens_host[0] != 0 || a.cu_seqlens_host[a.B] != a.T) return OB_ERR_ARG;
  for (int b = 0; b < a.B; ++b)
    if (a.cu_seqlens_host[b + 1] < a.cu_seqlens_host[b]) return OB_ERR_ARG;
  for (int h = 0; h < a.num_compute_heads; ++h) {
    if (a.kv_heads_host[h] < 0 || a.kv_heads_host[h] >= a.Hkv || a.sink_host[h] < 0 || a.local_host[h] < 1) return OB_ERR_ARG;
    base.kvh[h] = a.kv_heads_host[h]; base.sink[h] = a.sink_host[h]; base.local[h] = a.local_host[h];
  }
  base.Hq = a.Hq; base.g = g; base.qt = ROWS / g;
  base.q = a.q; base.k = a.k; base.v = a.v; base.out = a.out;
  base.qs = a.q_row_stride; base.ks = a.k_row_stride; base.vs = a.v_row_stride;
  base.scale_log2 = 1.4426950408889634f / sqrtf((float)DH);
  for (int b0 = 0; b0 < a.B; b0 += MAX_SEQ) {
    const int n = std::min(MAX_SEQ, a.B - b0);
    long long tiles = 0;
    for (int b = b0; b < b0 + n; ++b) tiles += (a.cu_seqlens_host[b + 1] - a.cu_seqlens_host[b] + base.qt - 1) / base.qt;
    if (tiles > 0x7fffffffLL) return OB_ERR_SHAPE;
    if (tiles > 0) launches.emplace_back(b0, n);
  }
  return 0;
}

static void fill(const StreamingPrefillArgs& a, Params& p, int b0, int n) {
  p.nseq = n;
  p.tile_start[0] = 0;
  for (int i = 0; i < n; ++i) {
    const int len = a.cu_seqlens_host[b0 + i + 1] - a.cu_seqlens_host[b0 + i];
    p.seq_tok0[i] = a.cu_seqlens_host[b0 + i];
    p.seq_len[i] = len;
    p.tile_start[i + 1] = p.tile_start[i] + (len + p.qt - 1) / p.qt;
  }
}

}  // namespace sp

int streaming_prefill_run(const StreamingPrefillArgs& a, cudaStream_t st) {
  using namespace sp;
  if (a.T <= 0 || a.num_compute_heads == 0) return a.T < 0 ? OB_ERR_ARG : 0;
  if (!a.q || !a.k || !a.v || !a.out) return OB_ERR_ARG;
  Params p{};
  std::vector<std::pair<int, int>> launches;
  if (int e = plan(a, p, launches)) return e;
  // every K / V row is one 256-byte bulk copy: 16-byte aligned rows
  if ((reinterpret_cast<uintptr_t>(a.k) & 15) || (reinterpret_cast<uintptr_t>(a.v) & 15) || (a.k_row_stride & 7) ||
      (a.v_row_stride & 7) || (reinterpret_cast<uintptr_t>(a.q) & 3) || (a.q_row_stride & 1) ||
      (reinterpret_cast<uintptr_t>(a.out) & 3))
    return OB_ERR_ALIGN;
  int dev = 0;
  cudaGetDevice(&dev);
  static bool attr_done[16] = {};
  if (dev < 0 || dev >= 16) return OB_ERR_ARG;
  if (!attr_done[dev]) {
    const cudaError_t e = cudaFuncSetAttribute(streaming_prefill_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES);
    if (e != cudaSuccess) { fprintf(stderr, "streaming_prefill: set smem: %s\n", cudaGetErrorString(e)); return OB_ERR_CUDA; }
    attr_done[dev] = true;
  }
  for (const auto& l : launches) {
    fill(a, p, l.first, l.second);
    const cudaError_t e = launch_pdl(streaming_prefill_kernel, dim3(p.tile_start[p.nseq], a.num_compute_heads), dim3(THREADS),
                                     (size_t)SMEM_BYTES, st, p);
    if (e != cudaSuccess) { fprintf(stderr, "streaming_prefill: launch: %s\n", cudaGetErrorString(e)); return OB_ERR_CUDA; }
  }
  return 0;
}

int streaming_prefill_plan(const StreamingPrefillArgs& a, int launch, int cta_x, int cta_y, int* out, int* key_tiles,
                           int max_key_tiles) {
  using namespace sp;
  if (!out) return OB_ERR_ARG;
  Params p{};
  std::vector<std::pair<int, int>> launches;
  if (int e = plan(a, p, launches)) return e;
  out[0] = a.num_compute_heads ? (int)launches.size() : 0;
  if (launch < 0 || launch >= out[0]) return 0;
  fill(a, p, launches[launch].first, launches[launch].second);
  out[1] = p.tile_start[p.nseq];
  out[2] = a.num_compute_heads;
  if (cta_x < 0 || cta_x >= out[1] || cta_y < 0 || cta_y >= out[2]) return OB_ERR_ARG;
  const Cta c = locate(p, cta_x, out[1]);
  out[3] = launches[launch].first + c.seq;
  out[4] = c.q_lo; out[5] = c.q_hi;
  out[6] = p.kvh[cta_y];
  KeyTiles kt;
  kt.init(c.q_lo, c.q_hi, p.sink[cta_y], p.local[cta_y]);
  out[7] = kt.n;
  for (int i = 0; i < kt.n && i < max_key_tiles; ++i) key_tiles[i] = kt.tile(i);
  return 0;
}

}  // namespace ob
