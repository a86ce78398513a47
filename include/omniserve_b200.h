/* omniserve_b200 -- C ABI of the B200-native W4A8KV4 hot path.
 *
 * Drop-in boundary.  The reference (mit-han-lab/omniserve) has no C ABI: its boundary is 13 pybind11
 * torch extensions under the python package `omniserve_backend` (kernels/setup.py:156-333) whose
 * functions take torch::Tensor.  Every entry point below is what such an extension function does after it
 * has unwrapped its tensors: raw device pointers, sizes, and the CUDA stream.  `INTEGRATION.md` shows
 * the binding a maintainer of the reference would add for each; `omniserve_b200/backend/*.py` is that
 * binding done with ctypes (same module / function names and argument order as the reference).
 *
 * Conventions: all pointers are device pointers unless stated; `stream` is a cudaStream_t passed as
 * void*; every function is asynchronous w.r.t. the host and returns 0 or an OB_ERR_* code (reference:
 * TORCH_CHECK -> RuntimeError; the ctypes mirror raises RuntimeError on non-zero).  fp16 = IEEE half.
 * No torch types, no CPU fallback.
 */
#ifndef OMNISERVE_B200_H
#define OMNISERVE_B200_H
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

#define OB_OK 0
#define OB_ERR_SHAPE 1
#define OB_ERR_ALIGN 2
#define OB_ERR_CUDA 3
#define OB_ERR_DRIVER 4
#define OB_ERR_ARG 5

int ob_version(void);
const char* ob_error_string(int code);

/* ---- qgemm_w4a8_per_chn.gemm_forward_cuda   (kernels/csrc/qgemm/w4a8_per_chn/gemm_cuda.cu:601-657)
 * out[M,N] = (in[M,K] . Wu4[N,K]^T) * wscales[n] * ascales[m] - w_szs[n] * a_ssums[m]
 * kernel: int8 [N,K/2] in the reference tile layout (w4a8_linear.py:297-327); ldc = out row pitch (elements). */
int ob_w4a8_gemm_per_chn(const int8_t* in_feats, const int8_t* kernel, const void* wscales, const void* ascales,
                         const void* w_szs, const void* a_ssums, void* out_feats, int M, int N, int K, int ldc,
                         void* stream);

/* ---- qgemm_w4a8_per_group.gemm_forward_cuda (kernels/csrc/qgemm/w4a8_per_group/gemm_cuda.cu:635-707)
 * w8 = q4*s2 + z2 (bytewise mod 256); out = (in . w8^T) * (wscales[n]*ascales[m]);  group = 128. */
int ob_w4a8_gemm_per_group(const int8_t* in_feats, const int8_t* kernel, const int8_t* zeros,
                           const int8_t* scales_i8, const void* wscales, const void* ascales, void* out_feats,
                           int M, int N, int K, int ldc, void* stream);

/* ---- grouped W4A8 per-channel GEMM for mixture-of-experts layers.  Interface of the reference's UNRELEASED op
 * `moe_gemm_forward_cuda_api(x, qweight, s1_scales, input_scales, s1_szeros, input_sum, problem_sizes)`
 * (omniserve/modeling/layers/quantized_linear/w4a8_moe_linear.py:83-94, buffers :30-72): in_feats int8 [T, K] with token
 * rows sorted by expert; kernel int8 [E, N, K/2], each expert in the w4a8_linear.py:297-327 tile layout; wscales / w_szs
 * fp16 [E, N]; ascales / a_ssums fp16 [T]; problem_sizes_host[e] = rows routed to expert e (HOST array, sum == T);
 * out fp16 [T, ldc] = per row r of expert e: (in[r] . W_e^T) * wscales[e,n] * ascales[r] - w_szs[e,n] * a_ssums[r].
 * N % 128 == 0, K % 128 == 0. */
int ob_w4a8_moe_gemm(const int8_t* in_feats, const int8_t* kernel, const void* wscales, const void* ascales,
                     const void* w_szs, const void* a_ssums, void* out_feats, const int* problem_sizes_host, int num_experts,
                     int T, int N, int K, int ldc, void* stream);

/* ---- qgemm_w8a8.w8a8_gemm_forward_cuda (kernels/csrc/qgemm/w8a8/w8a8_gemm_cuda.cu:537-600, epilogue :515-530)
 * out[M, ldc] (fp16) = (in[M,K] int8 . kernel[N,K]^T int8, s32 accumulate) * (wscales[n] * ascales[m]); kernel is plain
 * row-major [N, K] (w8a8_linear.py:42-52).  N % 8 == 0, K % 128 == 0. */
int ob_w8a8_gemm(const int8_t* in_feats, const int8_t* kernel, const void* wscales, const void* ascales, void* out_feats,
                 int M, int N, int K, int ldc, void* stream);

/* Same two GEMMs with scheduling knobs exposed for tests: force_bn in {0,16,32,64,128}, force_mode
 * -1 auto / 0 data-parallel tiles / 1 stream-K / 2 cluster split-K / 3 decode kernel (M <= 64), force_ctas 0 = auto. */
int ob_w4a8_gemm_ex(int per_group, const int8_t* in_feats, const int8_t* kernel, const int8_t* zeros,
                    const int8_t* scales_i8, const void* wscales, const void* ascales, const void* w_szs,
                    const void* a_ssums, void* out_feats, int M, int N, int K, int ldc, int force_bn,
                    int force_mode, int force_ctas, void* stream);
/* Host-only (no CUDA call, usable without a GPU): the scheduling decision the decode kernel (M <= 64) takes for a shape on a
 * device with `sms` SMs -- token tile BN, K-blocks of 128 per CTA, CTAs, and the cluster size of an aligned 2 / 4 / 8-way
 * split-K (0 = whole tiles or the L2 reduction).  For tests and tooling. */
int ob_debug_w4a8_decode_plan(int M, int N, int K, int sms, int ctas_per_sm, int use_cluster, int* bn, int* units_per_cta,
                              int* grid, int* cluster_s);

/* Extension (decode-sized M): the W4A8 GEMM followed, in the same launch, by the residual add + norm + per-token quant
 * that consumes its output in the reference's layer (llama_w4a8_unpad.py:425-431: `residual + o_proj(...)` ->
 * post_attention_layernorm -> int8; :437 + next layer's :416-421 for down_proj): hidden_out = hidden_in + out_feats
 * (fp16), then as ob_rms_norm_general(_fuse_sum)(norm_out, hidden_out, norm_weight, ...).  out_feats is still written.
 * ascales / a_ssums (inputs of the GEMM) may alias norm_scale / norm_sum (outputs of the tail).  Bit-identical to the
 * three-op chain.  M <= 256, N <= 4096 (returns OB_ERR_SHAPE otherwise: call the ops separately). */
int ob_w4a8_gemm_add_norm_quant(int per_group, const int8_t* in_feats, const int8_t* kernel, const int8_t* zeros,
                                const int8_t* scales_i8, const void* wscales, const void* ascales, const void* w_szs,
                                const void* a_ssums, void* out_feats, int M, int N, int K, int ldc, const void* hidden_in,
                                void* hidden_out, const void* norm_weight, int8_t* norm_out, void* norm_sum,
                                void* norm_scale, float eps, void* stream);

/* ---- fused_kernels.invoke_quant / invoke_quant_fuse_sum (kernels/csrc/fused_kernels.cu:218-271), per-token */
int ob_invoke_quant(int8_t* out, const void* input, void* scale, int num_tokens, int hidden, void* stream);
int ob_invoke_quant_fuse_sum(int8_t* out, const void* input, void* input_sum, void* scale, int num_tokens,
                             int hidden, void* stream);

/* ---- layernorm_ops (kernels/csrc/layernorm_kernels.cu:409-513), per-token quant variants */
int ob_rms_norm(void* out, const void* input, const void* weight, float eps, int num_tokens, int hidden,
                void* stream);
int ob_rms_norm_general(int8_t* out, const void* input, const void* weight, void* scaling, float eps,
                        int num_tokens, int hidden, void* stream);
int ob_rms_norm_general_fuse_sum(int8_t* out, const void* input, const void* weight, void* input_sum,
                                 void* scaling, float eps, int num_tokens, int hidden, void* stream);

/* Extensions (not in the reference): the fp16 residual add of llama_w4a8_unpad.py:425,437 fused into the norm
 * that follows it.  x = hidden_in + delta (fp16); hidden_out = x; then as rms_norm_general(_fuse_sum) / rms_norm.
 * input_sum may be NULL.  Bit-identical to torch.add followed by the unfused op. */
int ob_add_rms_norm_general(int8_t* out, const void* hidden_in, const void* delta, void* hidden_out, const void* weight,
                            void* input_sum, void* scaling, float eps, int num_tokens, int hidden, void* stream);
int ob_add_rms_norm(void* out, const void* hidden_in, const void* delta, const void* weight, float eps, int num_tokens,
                    int hidden, void* stream);

/* Extensions for tensor parallelism (the reference has none): the all-reduce that follows the row-parallel o_proj /
 * down_proj is fused into the norm that consumes it.  Every rank's GEMM leaves its partial sums in a buffer that all
 * GPUs of the node map (CUDA peer / symmetric memory over NVLink); the kernel exchanges per-block epoch flags in peer
 * memory, sums the W partial rows in fp32 in rank order and continues as ob_add_rms_norm_general / ob_add_rms_norm.
 * bufs[p] / flags[p]: rank p's buffer / flag array as mapped in THIS process (flags: uint32 [max_blocks][8], zeroed once;
 * epoch: local uint32 [max_blocks], zeroed once).  num_tokens <= max_blocks; all ranks must call with the same shape. */
typedef struct ob_peer_ctx {
  const void* bufs[8];
  void* flags[8];
  void* epoch;
  int world, rank, max_blocks;
} ob_peer_ctx;
int ob_peer_add_rms_norm_general(int8_t* out, const void* hidden_in, const ob_peer_ctx* peer, void* hidden_out,
                                 const void* weight, void* input_sum, void* scaling, float eps, int num_tokens, int hidden,
                                 void* stream);
int ob_peer_add_rms_norm(void* out, const void* hidden_in, const ob_peer_ctx* peer, const void* weight, float eps,
                         int num_tokens, int hidden, void* stream);

/* ---- activation_ops.silu_and_mul (kernels/csrc/activation_kernels.cu:84-97); input [T,2d] -> out [T,d] */
int ob_silu_and_mul(void* out, const void* input, int num_tokens, int d, void* stream);
/* silu_and_mul fused with invoke_quant(_fuse_sum) (activation.py:54-77 runs them as two kernels);
 * input_sum may be NULL. */
int ob_silu_and_mul_quant(int8_t* out, const void* input, void* input_sum, void* scale, int num_tokens, int d,
                          void* stream);
/* fp16 elementwise add (llama_w4a8_unpad.py:425,437). n % 8 == 0. */
int ob_add_f16(void* out, const void* a, const void* b, long long n, void* stream);

/* ---- fused_attention_{pure_dense,fine_grained_dense,fine_grained_sparse}.single_query_attention
 * (fused_attention_pure_dense/fused_attention.cpp:150-240; fine_grained/sparse_attention/fused_attention.cpp:198-377) */
typedef struct ob_kv4_decode_args {
  const void* q; const void* k; const void* v;       /* fp16 views [B,Hq,128] / [B,Hkv,128], head stride 128 */
  long long q_batch_stride, k_batch_stride, v_batch_stride; /* elements */
  void* out;                                          /* fp16 [B,Hq,128] contiguous */
  const int64_t* retrieval_kv_pointers;               /* [B,2,r_max_pages] device addresses of K / V pages */
  const int64_t* streaming_kv_pointers;               /* [B,2,s_max_pages] or NULL */
  int r_max_pages, s_max_pages;
  const int32_t* length_per_sample;                   /* [B] context length incl. the new token, or NULL */
  const int32_t* retrieval_head_flags;                /* [Hkv] or NULL */
  const int32_t* head_rank_table;                     /* [Hkv] or NULL */
  const int32_t* dynamic_sparse_page_idxes;           /* [B,Hq,P] or NULL */
  int num_dynamic_sparse_pages;
  int batch, num_heads, num_kv_heads, head_dim, tokens_per_block;
  int num_retrieval_kv_heads, num_streaming_kv_heads;
  int sink_token_num, local_token_num, sink_block_num, local_block_num;
  int timestep;                                       /* max cached tokens over the batch */
  int rotary_embedding_dim; float rotary_base; float rotary_scale; /* scale = linear factor (1 = none) */
  int force_split;                                    /* 0 = auto */
  /* fused_attention_fine_grained_sparse only (sparse_attention/...Template.hpp:1414-1429): when
   * tokens_per_sub_chunk > 0 the K append of a retrieval head also folds the new post-RoPE key into the page's
   * kmax / kmin statistics of its sub-chunk (element-wise max / min with what is stored there). */
  int tokens_per_sub_chunk;
  int hidden_dim_per_retrieval_token;                 /* num_retrieval_kv_heads * head_dim */
  /* Extension (not in the reference): fuse the per-token INT8 quantisation that follows the attention in
   * llama_w4a8_unpad.py:354 (invoke_quant / invoke_quant_fuse_sum of the [B, Hq*128] output) into this call.  NULL =
   * off.  quant_out int8 [B, Hq*128], quant_scale fp16 [B], quant_sum fp16 [B] or NULL; bit-identical to the two-op
   * chain. */
  void* quant_out; void* quant_scale; void* quant_sum;
  /* Extension: 1 = the caller guarantees that length_per_sample, the head / page tables, dynamic_sparse_page_idxes and
   * every page except the newest were last written before the kernel that PRECEDES this call in the stream (true inside
   * a decode loop); the kernel then streams those pages while its predecessor is still draining (programmatic dependent
   * launch).  0 = read nothing before the stream dependency has resolved (safe right after a prefill write). */
  int history_is_stable;
  /* Per-tensor KV8 mode (fused_attention_per_tensor/{dense,sparse}_attention/fused_attention.cpp: single_query_attention
   * takes kv_scale_quant_orig / kv_scale_orig_quant, float[2] = K, V): both non-NULL = the pages hold INT8 codes
   * [H_pool][64][128] (size_per_token = H_pool * 128) with static per-tensor scales; NULL = the KV4 pages above. */
  const float* kv_scale_quant_orig; const float* kv_scale_orig_quant;
} ob_kv4_decode_args;
int ob_kv4_single_query_attention(const ob_kv4_decode_args* args, void* stream);

/* ---- apply_bias_rope_update_kv_cache (fine_grained_common/update_kv_cache.cu:27-136), no bias */
typedef struct ob_kv4_prefill_args {
  void* qkv;                                          /* fp16 [T,(Hq+2Hkv)*128], RoPE applied in place to q,k */
  const int32_t* seq_lens;                            /* [B] */
  const int32_t* padding_offset;                      /* [T] */
  int max_seq_len;
  const int64_t* retrieval_kv_pointers; const int64_t* streaming_kv_pointers;
  int r_max_pages, s_max_pages;
  const int32_t* retrieval_head_flags; const int32_t* head_rank_table;
  int num_tokens, batch, num_heads, num_kv_heads;
  int num_retrieval_kv_heads, num_streaming_kv_heads;
  int sink_token_num, local_token_num, sink_block_num, local_block_num;
  int rotary_embedding_dim; float rotary_base; float rotary_scale;
  /* Per-tensor KV8 mode (per_tensor_common/update_kv_cache.cu:27-): non-NULL float[2] (K, V) = write INT8 pages
   * cvt.rni.sat(x * scale) instead of KV4; NULL = KV4.  Not supported by the _pool variant (OB_ERR_ARG). */
  const float* kv_scale_orig_quant;
} ob_kv4_prefill_args;
int ob_kv4_apply_rope_update_kv_cache(const ob_kv4_prefill_args* args, void* stream);
/* Extension (SURVEY.md section 8 row f2): the call above FUSED with fused_attention_ctx_pool.paged_min_max_pool of the
 * rotated keys (ctx_update_kv.py:104-178 runs the two back to back): one pass rotates q / k in place, writes the KV4 pages
 * and the kmax / kmin statistics of every `tokens_per_sub_chunk`-token sub-chunk of the retrieval heads (statistics row of a
 * head = head_rank_table[head]).  Page bytes and statistics are bit-identical to the two-op chain.  tokens_per_sub_chunk
 * must be 16, num_retrieval_kv_heads <= 8. */
int ob_kv4_apply_rope_update_kv_cache_pool(const ob_kv4_prefill_args* args, int tokens_per_sub_chunk, void* stream);

/* ---- compute_padding_offsets (common/input_metadata_helper.cu:16-49) */
int ob_compute_padding_offsets(int32_t* out, const int32_t* cu_seqlens, int batch, int max_seqlen, void* stream);

/* ---- fused_attention_ctx_pool.paged_min_max_pool (sparse_utils/ContextPool/context_pool_kernel.cu:145-213)
 * keys: fp16 [T, H_in, 128] post-RoPE (row / head strides in elements); for every sequence b, pooled head j
 * (input head pooling_heads_idx[j]) and `pooling_size`-token sub-chunk, the channel-wise max / min over the
 * sub-chunk's valid tokens is written to the kmax / kmin area of the K page that holds the sub-chunk. */
int ob_paged_min_max_pool(const void* keys, const int64_t* retrieval_kv_pointers, const int32_t* cu_seqlens,
                          const int32_t* pooling_heads_idx, long long row_stride, long long head_stride,
                          int r_max_pages, int batch, int num_pooling_heads, int head_dim, int max_seqlen,
                          int pooling_size, int page_size, int size_per_retrieval_token, int kv_cache_with_zeros,
                          void* stream);

/* ---- fused_attention_selector.single_query_page_selector
 * (sparse_utils/KVPageSelector/fused_kv_page_selector.cpp:171-334, KVPageSelectorTemplate.hpp:786-1290)
 * out: fp16 [B, Hq, padded] with padded = roundup(ceil(timestep / tokens_per_sub_chunk), sub-chunks per page);
 * zeroed by this call, rows of streaming heads stay zero.  score[sub] = sum_d max(q_d*kmax_d, q_d*kmin_d)
 * with q rotated to position length-1, fp16 arithmetic as in the reference. */
typedef struct ob_page_selector_args {
  const void* q; long long q_batch_stride;            /* fp16 [B,Hq,128] view, head stride 128 */
  void* out;
  const int64_t* retrieval_kv_pointers; int r_max_pages;
  const int32_t* length_per_sample;                   /* [B] incl. the new token, or NULL (= timestep + 1) */
  const int32_t* retrieval_head_flags; const int32_t* head_rank_table;   /* [Hkv] or NULL */
  int batch, num_heads, num_kv_heads, head_dim, tokens_per_block;
  int size_per_retrieval_token, num_retrieval_kv_heads;
  int timestep;
  int rotary_embedding_dim; float rotary_base; float rotary_scale;
  int tokens_per_sub_chunk, hidden_dim_per_retrieval_token;
} ob_page_selector_args;
int ob_kv4_page_selector(const ob_page_selector_args* args, void* stream);

/* Extension (SURVEY.md section 8 row f2): the page choice the reference makes with torch ops after the selector
 * (omniserve/modeling/layers/decoding_attention.py:132-141: view [B,Hq,pages,4] -> max -> topk(k-1) over all but the newest
 * page -> cat newest -> int32) as one kernel.  scores: the selector output, fp16 [rows = B*Hq, pitch] sub-chunk scores;
 * out int32 [rows, k_out]: the k_out-1 best of pages 0..total_pages-2 (ties at the threshold broken by page order; torch's
 * tie order is unspecified), then page total_pages-1.  The order within the first k_out-1 entries is ascending page index
 * per class (above threshold, ties), not score order -- the sparse attention only needs the set and the newest page last. */
int ob_kv4_page_topk(const void* scores, int32_t* out, int rows, int pitch_sub_chunks, int sub_chunks_per_page,
                     int total_pages, int k_out, void* stream);

/* ---- block_sparse_attn.token_streaming_attn_func for LServe's streaming heads (caller: ctx_attn_func.py:62-73; masks
 * ctx_attn_init.py:11-52).  fp16 causal prefill attention over variable-length sequences with the token-streaming mask:
 * query position i of a sequence attends key position j  iff  j <= i  and  (j < sink  or  i - j < local), which is the
 * window the streaming-head decode attention keeps (the sink plus the last `local` tokens, the current one included).
 * q [T, Hq, 128], k / v [T, Hkv, 128]: strided views (head stride 128, token strides below, e.g. into the qkv activation;
 * k / v 16-byte aligned, token strides multiples of 8).  out: fp16 [T, Hq, 128] contiguous; only the q-heads of the
 * kv heads listed in kv_heads are written.  cu_seqlens, kv_heads, sink, local are HOST arrays.  Hq / Hkv must divide
 * 128; at most 64 kv heads per call; sink >= 0, local >= 1.  Deterministic (no atomics). */
typedef struct ob_streaming_prefill_args {
  const void* q; const void* k; const void* v;
  long long q_row_stride, k_row_stride, v_row_stride; /* elements */
  void* out;
  const int32_t* cu_seqlens;                          /* HOST [batch + 1] */
  int batch, num_tokens, num_heads, num_kv_heads, head_dim;
  int num_compute_kv_heads;
  const int32_t* kv_heads;                            /* HOST [num_compute_kv_heads] */
  const int32_t* sink; const int32_t* local;          /* HOST [num_compute_kv_heads]: the (sink, local) of each kv group */
} ob_streaming_prefill_args;
int ob_token_streaming_prefill_attention(const ob_streaming_prefill_args* args, void* stream);
/* Host-only (no CUDA call, usable without a GPU): the launch plan of the call above.  out[0] = launches, out[1] / out[2] =
 * grid x / y of launch `launch`, out[3] = sequence, out[4] / out[5] = first / last query position (within the sequence) of
 * CTA (cta_x, cta_y), out[6] = its kv head, out[7] = number of 64-key tiles it visits, whose indices are written to
 * key_tiles (at most max_key_tiles).  Device pointers in args may be NULL. */
int ob_debug_streaming_prefill_plan(const ob_streaming_prefill_args* args, int launch, int cta_x, int cta_y, int* out,
                                    int* key_tiles, int max_key_tiles);

/* ==== Mixture-of-experts block (Mixtral).  The reference's MixtralSparseMoeBlockOurs.forward calls these ops but never released
 * them (omniserve/modeling/models/mixtral_w4a8_unpad.py:300-395, raises NotImplementedError at :309); oracle/moe.py pins the
 * semantics.  All are deterministic and row-independent; E <= 64 experts, 1 <= k <= min(E, 8) experts per token. */

/* ---- router logits (`router_logits = self.gate(hidden_states).float()`, :277,305): logits fp32 [T, E] = fp16-rounded
 * sum_h x[t,h] * gate_weight[e,h]; x fp16 [T, H] (the post_attention_layernorm output), gate_weight fp16 [E, H].  H % 8 == 0. */
int ob_moe_router_logits(const void* x, const void* gate_weight, float* logits, int T, int H, int E, void* stream);

/* ---- moe_helpers.moe_topk_gating_softmax (:315) + the expert histogram the caller builds with torch.bincount (:320), on the
 * device in one CTA: p = softmax(logits) (fp32), the k most probable experts (ties -> lower index; slots in descending p),
 * routing_weights fp32 [T, k] = p_sel / sum(p_sel); expert_indices int32 [T*k] token-major; rows sorted by expert, stably by
 * (token, slot): permuted_loc_to_unpermuted_loc int32 [T*k] (value t*k + j); expert_offsets int32 [E+1] (cumulative). */
int ob_moe_topk_sort(const float* logits, float* routing_weights, int32_t* expert_indices, int32_t* permuted_loc_to_unpermuted_loc,
                     int32_t* expert_offsets, int T, int E, int k, void* stream);

/* ---- moe_helpers.moe_expand_inputs_and_scales (:345): row r of q_out / ssums_out / scales_out = row (perm[r] / k) of the
 * per-token INT8 activations (invoke_quant_fuse_sum output, :334) / sums / scales; unpermuted_loc_to_permuted_loc[perm[r]] = r.
 * q_input_ssums / ssums_out may both be NULL.  H % 16 == 0. */
int ob_moe_expand(const int8_t* q_hidden_states, const void* q_input_ssums, const void* q_input_scales,
                  const int32_t* permuted_loc_to_unpermuted_loc, int8_t* q_out, void* ssums_out, void* scales_out,
                  int32_t* unpermuted_loc_to_permuted_loc, int T, int k, int H, void* stream);

/* ---- moe_helpers.moe_finalize_routing (:388): out fp16 [T, H] = fp16(sum_j routing_weights[t,j] * q_w2_out[inv[t*k+j]]),
 * fp32, j ascending; q_w2_out fp16 [T*k, ldy]. */
int ob_moe_finalize(const void* q_w2_out, const float* routing_weights, const int32_t* unpermuted_loc_to_permuted_loc, void* out,
                    int T, int k, int H, int ldy, void* stream);

/* ---- the w1_w3 / w2 grouped GEMMs of the block (:354,382) with the expert row ranges in DEVICE memory: as ob_w4a8_moe_gemm, but
 * expert e owns rows [expert_offsets[e], expert_offsets[e+1]) of the total_rows rows (the ob_moe_topk_sort output) and gets at
 * most 64 of them -- which holds whenever the layer has <= 64 tokens, since a token routes to distinct experts.  No host
 * read-back: capturable in a CUDA graph.  Rows are clamped to [0, total_rows] and cut at 64, so a malformed table cannot
 * address outside in_feats / out.  num_experts <= 64. */
int ob_w4a8_moe_gemm_dev(const int8_t* in_feats, const int8_t* kernel, const void* wscales, const void* ascales,
                         const void* w_szs, const void* a_ssums, void* out_feats, const int32_t* expert_offsets, int num_experts,
                         int total_rows, int N, int K, int ldc, void* stream);
/* Host-only (no CUDA call, usable without a GPU): the schedule of the call above on a device with `sms` SMs for the HOST table
 * offsets_host [E+1].  grid / tiles_per_cta depend on (E, N, K, sms) only.  If entries is not NULL it receives, per 128-row
 * weight tile in tile order (E * N / 128 entries, max_entries >= that), six ints: CTA, slot, expert, n-tile, row0, rows. */
int ob_debug_moe_device_plan(int num_experts, int N, int K, int sms, const int32_t* offsets_host, int total_rows, int* grid,
                             int* tiles_per_cta, int* entries, int max_entries);

#ifdef __cplusplus
}
#endif
#endif
