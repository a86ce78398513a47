// extern "C" entry points declared in include/omniserve_b200.h.
#include "../../include/omniserve_b200.h"
#include "kv4_attention.h"
#include "lserve_ops.h"
#include "moe_ops.h"
#include "prefill_attention.h"
#include "small_ops.h"
#include "w4a8_gemm.h"

using namespace ob;

#define H(p) reinterpret_cast<const __half*>(p)
#define HM(p) reinterpret_cast<__half*>(p)
#define ST(s) reinterpret_cast<cudaStream_t>(s)

extern "C" {

int ob_version(void) { return 100; }

const char* ob_error_string(int code) {
  switch (code) {
    case OB_OK: return "ok";
    case OB_ERR_SHAPE: return "unsupported shape";
    case OB_ERR_ALIGN: return "misaligned pointer or pitch";
    case OB_ERR_CUDA: return "CUDA runtime error";
    case OB_ERR_DRIVER: return "CUDA driver / tensor-map error";
    case OB_ERR_ARG: return "bad argument";
  }
  return "unknown";
}

int ob_w4a8_gemm_ex(int per_group, const int8_t* in_feats, const int8_t* kernel, const int8_t* zeros,
                    const int8_t* scales_i8, const void* wscales, const void* ascales, const void* w_szs,
                    const void* a_ssums, void* out_feats, int M, int N, int K, int ldc, int force_bn,
                    int force_mode, int force_ctas, void* stream) {
  if (!in_feats || !kernel || !wscales || !ascales || !out_feats) return OB_ERR_ARG;
  if (per_group ? (!zeros || !scales_i8) : (!w_szs || !a_ssums)) return OB_ERR_ARG;
  W4A8GemmArgs a{};
  a.in_feats = in_feats; a.qweight = kernel; a.s2_scales = scales_i8; a.s2_zeros = zeros;
  a.wscales = H(wscales); a.ascales = H(ascales); a.w_szs = H(w_szs); a.a_ssums = H(a_ssums);
  a.out_feats = HM(out_feats); a.M = M; a.N = N; a.K = K; a.ldc = ldc;
  a.force_bn = force_bn; a.force_mode = force_mode; a.force_ctas = force_ctas;
  return w4a8_gemm_run(a, per_group != 0, ST(stream));
}

int ob_w4a8_gemm_add_norm_quant(int per_group, const int8_t* in_feats, const int8_t* kernel, const int8_t* zeros,
                                const int8_t* scales_i8, const void* wscales, const void* ascales, const void* w_szs,
                                const void* a_ssums, void* out_feats, int M, int N, int K, int ldc, const void* hidden_in,
                                void* hidden_out, const void* norm_weight, int8_t* norm_out, void* norm_sum,
                                void* norm_scale, float eps, void* stream) {
  if (!in_feats || !kernel || !wscales || !ascales || !out_feats) return OB_ERR_ARG;
  if (per_group ? (!zeros || !scales_i8) : (!w_szs || !a_ssums)) return OB_ERR_ARG;
  if (!hidden_in || !hidden_out || !norm_weight || !norm_out || !norm_scale) return OB_ERR_ARG;
  W4A8GemmArgs a{};
  a.in_feats = in_feats; a.qweight = kernel; a.s2_scales = scales_i8; a.s2_zeros = zeros;
  a.wscales = H(wscales); a.ascales = H(ascales); a.w_szs = H(w_szs); a.a_ssums = H(a_ssums);
  a.out_feats = HM(out_feats); a.M = M; a.N = N; a.K = K; a.ldc = ldc;
  a.tail_hidden_in = H(hidden_in); a.tail_hidden_out = HM(hidden_out); a.tail_gamma = H(norm_weight);
  a.tail_q = norm_out; a.tail_scale = HM(norm_scale); a.tail_sum = HM(norm_sum); a.tail_eps = eps;
  return w4a8_gemm_run(a, per_group != 0, ST(stream));
}

int ob_w4a8_gemm_per_chn(const int8_t* in_feats, const int8_t* kernel, const void* wscales, const void* ascales,
                         const void* w_szs, const void* a_ssums, void* out_feats, int M, int N, int K, int ldc,
                         void* stream) {
  return ob_w4a8_gemm_ex(0, in_feats, kernel, nullptr, nullptr, wscales, ascales, w_szs, a_ssums, out_feats, M, N, K,
                         ldc, 0, -1, 0, stream);
}

int ob_w4a8_gemm_per_group(const int8_t* in_feats, const int8_t* kernel, const int8_t* zeros,
                           const int8_t* scales_i8, const void* wscales, const void* ascales, void* out_feats,
                           int M, int N, int K, int ldc, void* stream) {
  return ob_w4a8_gemm_ex(1, in_feats, kernel, zeros, scales_i8, wscales, ascales, nullptr, nullptr, out_feats, M, N, K,
                         ldc, 0, -1, 0, stream);
}

int ob_debug_w4a8_decode_plan(int M, int N, int K, int sms, int ctas_per_sm, int use_cluster, int* bn, int* units_per_cta,
                              int* grid, int* cluster_s) {
  return w4a8_gemm_decode_plan(M, N, K, sms, ctas_per_sm, use_cluster, bn, units_per_cta, grid, cluster_s);
}

int ob_w4a8_moe_gemm(const int8_t* in_feats, const int8_t* kernel, const void* wscales, const void* ascales,
                     const void* w_szs, const void* a_ssums, void* out_feats, const int* problem_sizes_host, int num_experts,
                     int T, int N, int K, int ldc, void* stream) {
  if (!in_feats || !kernel || !wscales || !ascales || !w_szs || !a_ssums || !out_feats || !problem_sizes_host) return OB_ERR_ARG;
  return w4a8_moe_gemm_run(in_feats, kernel, H(wscales), H(ascales), H(w_szs), H(a_ssums), HM(out_feats), problem_sizes_host,
                           num_experts, T, N, K, ldc, ST(stream));
}

int ob_w4a8_moe_gemm_dev(const int8_t* in_feats, const int8_t* kernel, const void* wscales, const void* ascales,
                         const void* w_szs, const void* a_ssums, void* out_feats, const int32_t* expert_offsets, int num_experts,
                         int total_rows, int N, int K, int ldc, void* stream) {
  if (!in_feats || !kernel || !wscales || !ascales || !w_szs || !a_ssums || !out_feats || !expert_offsets) return OB_ERR_ARG;
  return w4a8_moe_gemm_dev_run(in_feats, kernel, H(wscales), H(ascales), H(w_szs), H(a_ssums), HM(out_feats), expert_offsets,
                               num_experts, total_rows, N, K, ldc, ST(stream));
}

int ob_debug_moe_device_plan(int num_experts, int N, int K, int sms, const int32_t* offsets_host, int total_rows, int* grid,
                             int* tiles_per_cta, int* entries, int max_entries) {
  return w4a8_moe_dev_plan(num_experts, N, K, sms, offsets_host, total_rows, grid, tiles_per_cta, entries, max_entries);
}

int ob_moe_router_logits(const void* x, const void* gate_weight, float* logits, int T, int H, int E, void* stream) {
  if (T > 0 && (!x || !gate_weight || !logits)) return OB_ERR_ARG;
  return moe_router_logits_run(H(x), H(gate_weight), logits, T, H, E, ST(stream));
}

int ob_moe_topk_sort(const float* logits, float* routing_weights, int32_t* expert_indices, int32_t* permuted_loc_to_unpermuted_loc,
                     int32_t* expert_offsets, int T, int E, int k, void* stream) {
  if (!expert_offsets || (T > 0 && (!logits || !routing_weights || !expert_indices || !permuted_loc_to_unpermuted_loc)))
    return OB_ERR_ARG;
  return moe_topk_sort_run(logits, routing_weights, expert_indices, permuted_loc_to_unpermuted_loc, expert_offsets, T, E, k,
                           ST(stream));
}

int ob_moe_expand(const int8_t* q_hidden_states, const void* q_input_ssums, const void* q_input_scales,
                  const int32_t* permuted_loc_to_unpermuted_loc, int8_t* q_out, void* ssums_out, void* scales_out,
                  int32_t* unpermuted_loc_to_permuted_loc, int T, int k, int H, void* stream) {
  if (T > 0 && (!q_hidden_states || !q_input_scales || !permuted_loc_to_unpermuted_loc || !q_out || !scales_out ||
                !unpermuted_loc_to_permuted_loc))
    return OB_ERR_ARG;
  return moe_expand_run(q_hidden_states, H(q_input_ssums), H(q_input_scales), permuted_loc_to_unpermuted_loc, q_out, HM(ssums_out),
                        HM(scales_out), unpermuted_loc_to_permuted_loc, T, k, H, ST(stream));
}

int ob_moe_finalize(const void* q_w2_out, const float* routing_weights, const int32_t* unpermuted_loc_to_permuted_loc, void* out,
                    int T, int k, int H, int ldy, void* stream) {
  if (T > 0 && (!q_w2_out || !routing_weights || !unpermuted_loc_to_permuted_loc || !out)) return OB_ERR_ARG;
  return moe_finalize_run(H(q_w2_out), routing_weights, unpermuted_loc_to_permuted_loc, HM(out), T, k, H, ldy, ST(stream));
}

int ob_w8a8_gemm(const int8_t* in_feats, const int8_t* kernel, const void* wscales, const void* ascales, void* out_feats,
                 int M, int N, int K, int ldc, void* stream) {
  if (!in_feats || !kernel || !wscales || !ascales || !out_feats) return OB_ERR_ARG;
  return w8a8_gemm_run(in_feats, kernel, H(wscales), H(ascales), HM(out_feats), M, N, K, ldc, ST(stream));
}

int ob_invoke_quant(int8_t* out, const void* input, void* scale, int T, int Hd, void* stream) {
  if (T <= 0) return 0;
  if (!out || !input || !scale) return OB_ERR_ARG;
  return quant_run(H(input), out, HM(scale), nullptr, T, Hd, ST(stream));
}
int ob_invoke_quant_fuse_sum(int8_t* out, const void* input, void* input_sum, void* scale, int T, int Hd,
                             void* stream) {
  if (T <= 0) return 0;
  if (!out || !input || !scale || !input_sum) return OB_ERR_ARG;
  return quant_run(H(input), out, HM(scale), HM(input_sum), T, Hd, ST(stream));
}
int ob_rms_norm(void* out, const void* input, const void* weight, float eps, int T, int Hd, void* stream) {
  if (T <= 0) return 0;
  if (!out || !input || !weight) return OB_ERR_ARG;
  return rmsnorm_f16_run(H(input), nullptr, H(weight), HM(out), T, Hd, eps, ST(stream));
}
int ob_rms_norm_general(int8_t* out, const void* input, const void* weight, void* scaling, float eps, int T, int Hd,
                        void* stream) {
  if (T <= 0) return 0;
  if (!out || !input || !weight || !scaling) return OB_ERR_ARG;
  return rmsnorm_quant_run(H(input), nullptr, nullptr, H(weight), out, HM(scaling), nullptr, T, Hd, eps, ST(stream));
}
int ob_rms_norm_general_fuse_sum(int8_t* out, const void* input, const void* weight, void* input_sum, void* scaling,
                                 float eps, int T, int Hd, void* stream) {
  if (T <= 0) return 0;
  if (!out || !input || !weight || !scaling || !input_sum) return OB_ERR_ARG;
  return rmsnorm_quant_run(H(input), nullptr, nullptr, H(weight), out, HM(scaling), HM(input_sum), T, Hd, eps, ST(stream));
}
int ob_add_rms_norm_general(int8_t* out, const void* hidden_in, const void* delta, void* hidden_out, const void* weight,
                            void* input_sum, void* scaling, float eps, int T, int Hd, void* stream) {
  if (T <= 0) return 0;
  if (!out || !hidden_in || !delta || !hidden_out || !weight || !scaling) return OB_ERR_ARG;
  return rmsnorm_quant_run(H(hidden_in), H(delta), HM(hidden_out), H(weight), out, HM(scaling), HM(input_sum), T, Hd, eps,
                           ST(stream));
}
int ob_add_rms_norm(void* out, const void* hidden_in, const void* delta, const void* weight, float eps, int T, int Hd,
                    void* stream) {
  if (T <= 0) return 0;
  if (!out || !hidden_in || !delta || !weight) return OB_ERR_ARG;
  return rmsnorm_f16_run(H(hidden_in), H(delta), H(weight), HM(out), T, Hd, eps, ST(stream));
}
static PeerArgs to_peer(const ob_peer_ctx* x) {
  PeerArgs a{};
  for (int p = 0; p < 8; ++p) { a.bufs[p] = H(x->bufs[p]); a.flags[p] = reinterpret_cast<uint32_t*>(x->flags[p]); }
  a.epoch = reinterpret_cast<uint32_t*>(x->epoch); a.world = x->world; a.rank = x->rank; a.max_blocks = x->max_blocks;
  return a;
}
int ob_peer_add_rms_norm_general(int8_t* out, const void* hidden_in, const ob_peer_ctx* peer, void* hidden_out,
                                 const void* weight, void* input_sum, void* scaling, float eps, int T, int Hd, void* stream) {
  if (T <= 0) return 0;
  if (!out || !hidden_in || !peer || !hidden_out || !weight || !scaling) return OB_ERR_ARG;
  return peer_rmsnorm_quant_run(H(hidden_in), to_peer(peer), HM(hidden_out), H(weight), out, HM(scaling), HM(input_sum), T, Hd,
                                eps, ST(stream));
}
int ob_peer_add_rms_norm(void* out, const void* hidden_in, const ob_peer_ctx* peer, const void* weight, float eps, int T,
                         int Hd, void* stream) {
  if (T <= 0) return 0;
  if (!out || !hidden_in || !peer || !weight) return OB_ERR_ARG;
  return peer_rmsnorm_f16_run(H(hidden_in), to_peer(peer), H(weight), HM(out), T, Hd, eps, ST(stream));
}
int ob_silu_and_mul(void* out, const void* input, int T, int d, void* stream) {
  if (T <= 0) return 0;
  if (!out || !input) return OB_ERR_ARG;
  return silu_and_mul_run(H(input), HM(out), T, d, ST(stream));
}
int ob_silu_and_mul_quant(int8_t* out, const void* input, void* input_sum, void* scale, int T, int d, void* stream) {
  if (T <= 0) return 0;
  if (!out || !input || !scale) return OB_ERR_ARG;
  return silu_mul_quant_run(H(input), out, HM(scale), HM(input_sum), T, d, ST(stream));
}
int ob_add_f16(void* out, const void* a, const void* b, long long n, void* stream) {
  if (!out || !a || !b) return OB_ERR_ARG;
  return add_run(H(a), H(b), HM(out), (size_t)n, ST(stream));
}

int ob_kv4_single_query_attention(const ob_kv4_decode_args* x, void* stream) {
  if (!x || !x->q || !x->k || !x->v || !x->out) return OB_ERR_ARG;
  if (!x->retrieval_kv_pointers && !x->streaming_kv_pointers) return OB_ERR_ARG;
  KV4DecodeArgs a{};
  a.q = H(x->q); a.k = H(x->k); a.v = H(x->v);
  a.q_bs = x->q_batch_stride; a.k_bs = x->k_batch_stride; a.v_bs = x->v_batch_stride;
  a.out = HM(x->out);
  a.retrieval_kv_pointers = x->retrieval_kv_pointers; a.streaming_kv_pointers = x->streaming_kv_pointers;
  a.r_max_pages = x->r_max_pages; a.s_max_pages = x->s_max_pages;
  a.lengths = x->length_per_sample; a.retrieval_head_flags = x->retrieval_head_flags;
  a.head_rank_table = x->head_rank_table;
  a.dyn_idx = x->dynamic_sparse_page_idxes; a.dyn_pages = x->num_dynamic_sparse_pages;
  a.B = x->batch; a.Hq = x->num_heads; a.Hkv = x->num_kv_heads; a.head_dim = x->head_dim;
  a.tokens_per_block = x->tokens_per_block;
  a.num_retrieval_kv_heads = x->num_retrieval_kv_heads; a.num_streaming_kv_heads = x->num_streaming_kv_heads;
  a.sink_tokens = x->sink_token_num; a.local_tokens = x->local_token_num;
  a.sink_blocks = x->sink_block_num; a.local_blocks = x->local_block_num;
  a.timestep = x->timestep;
  a.max_attended = x->dynamic_sparse_page_idxes ? x->num_dynamic_sparse_pages * 64 : x->timestep;
  a.rotary_dim = x->rotary_embedding_dim; a.rotary_base = x->rotary_base;
  a.rotary_scale = x->rotary_scale != 0.f ? 1.0f / x->rotary_scale : 1.0f;
  a.force_split = x->force_split;
  a.tokens_per_sub_chunk = x->tokens_per_sub_chunk;
  a.hidden_dim_per_retrieval_token = x->hidden_dim_per_retrieval_token;
  a.q_out = reinterpret_cast<int8_t*>(x->quant_out); a.q_scale = HM(x->quant_scale); a.q_sum = HM(x->quant_sum);
  a.stable_history = x->history_is_stable;
  if ((x->kv_scale_quant_orig == nullptr) != (x->kv_scale_orig_quant == nullptr)) return OB_ERR_ARG;
  a.kv_scale_quant_orig = x->kv_scale_quant_orig; a.kv_scale_orig_quant = x->kv_scale_orig_quant;
  return kv4_decode_run(a, ST(stream));
}

int ob_kv4_apply_rope_update_kv_cache(const ob_kv4_prefill_args* x, void* stream) {
  if (!x || !x->qkv || !x->seq_lens || !x->padding_offset) return OB_ERR_ARG;
  KV4PrefillArgs a{};
  a.qkv = HM(x->qkv); a.seq_lens = x->seq_lens; a.padding_offset = x->padding_offset; a.max_seq_len = x->max_seq_len;
  a.retrieval_kv_pointers = x->retrieval_kv_pointers; a.streaming_kv_pointers = x->streaming_kv_pointers;
  a.r_max_pages = x->r_max_pages; a.s_max_pages = x->s_max_pages;
  a.retrieval_head_flags = x->retrieval_head_flags; a.head_rank_table = x->head_rank_table;
  a.T = x->num_tokens; a.B = x->batch; a.Hq = x->num_heads; a.Hkv = x->num_kv_heads;
  a.num_retrieval_kv_heads = x->num_retrieval_kv_heads; a.num_streaming_kv_heads = x->num_streaming_kv_heads;
  a.sink_tokens = x->sink_token_num; a.local_tokens = x->local_token_num;
  a.sink_blocks = x->sink_block_num; a.local_blocks = x->local_block_num;
  a.rotary_dim = x->rotary_embedding_dim; a.rotary_base = x->rotary_base;
  a.rotary_scale = x->rotary_scale != 0.f ? 1.0f / x->rotary_scale : 1.0f;
  a.kv_scale_orig_quant = x->kv_scale_orig_quant;
  return kv4_prefill_write_run(a, ST(stream));
}

int ob_kv4_apply_rope_update_kv_cache_pool(const ob_kv4_prefill_args* x, int tokens_per_sub_chunk, void* stream) {
  if (!x || !x->qkv || !x->seq_lens || !x->padding_offset) return OB_ERR_ARG;
  KV4PrefillArgs a{};
  a.qkv = HM(x->qkv); a.seq_lens = x->seq_lens; a.padding_offset = x->padding_offset; a.max_seq_len = x->max_seq_len;
  a.retrieval_kv_pointers = x->retrieval_kv_pointers; a.streaming_kv_pointers = x->streaming_kv_pointers;
  a.r_max_pages = x->r_max_pages; a.s_max_pages = x->s_max_pages;
  a.retrieval_head_flags = x->retrieval_head_flags; a.head_rank_table = x->head_rank_table;
  a.T = x->num_tokens; a.B = x->batch; a.Hq = x->num_heads; a.Hkv = x->num_kv_heads;
  a.num_retrieval_kv_heads = x->num_retrieval_kv_heads; a.num_streaming_kv_heads = x->num_streaming_kv_heads;
  a.sink_tokens = x->sink_token_num; a.local_tokens = x->local_token_num;
  a.sink_blocks = x->sink_block_num; a.local_blocks = x->local_block_num;
  a.rotary_dim = x->rotary_embedding_dim; a.rotary_base = x->rotary_base;
  a.rotary_scale = x->rotary_scale != 0.f ? 1.0f / x->rotary_scale : 1.0f;
  return kv4_prefill_write_pool_run(a, tokens_per_sub_chunk, ST(stream));
}

int ob_compute_padding_offsets(int32_t* out, const int32_t* cu_seqlens, int batch, int max_seqlen, void* stream) {
  if (!out || !cu_seqlens) return OB_ERR_ARG;
  return padding_offsets_run(out, cu_seqlens, batch, max_seqlen, ST(stream));
}

int ob_paged_min_max_pool(const void* keys, const int64_t* retrieval_kv_pointers, const int32_t* cu_seqlens,
                          const int32_t* pooling_heads_idx, long long row_stride, long long head_stride,
                          int r_max_pages, int batch, int num_pooling_heads, int head_dim, int max_seqlen,
                          int pooling_size, int page_size, int size_per_retrieval_token, int kv_cache_with_zeros,
                          void* stream) {
  if (!keys || !retrieval_kv_pointers || !cu_seqlens || !pooling_heads_idx) return OB_ERR_ARG;
  PoolArgs a{};
  a.keys = H(keys); a.row_stride = row_stride; a.head_stride = head_stride;
  a.retrieval_kv_pointers = retrieval_kv_pointers; a.r_max_pages = r_max_pages;
  a.cu_seqlens = cu_seqlens; a.pooling_heads_idx = pooling_heads_idx;
  a.batch = batch; a.num_pooling_heads = num_pooling_heads; a.head_dim = head_dim;
  a.max_seqlen = max_seqlen; a.pooling_size = pooling_size; a.page_size = page_size;
  a.size_per_retrieval_token = size_per_retrieval_token; a.kv_cache_with_zeros = kv_cache_with_zeros;
  return paged_min_max_pool_run(a, ST(stream));
}

int ob_kv4_page_selector(const ob_page_selector_args* x, void* stream) {
  if (!x || !x->q || !x->out || !x->retrieval_kv_pointers) return OB_ERR_ARG;
  SelectorArgs a{};
  a.q = H(x->q); a.q_bs = x->q_batch_stride; a.out = HM(x->out);
  a.retrieval_kv_pointers = x->retrieval_kv_pointers; a.r_max_pages = x->r_max_pages;
  a.lengths = x->length_per_sample;
  a.retrieval_head_flags = x->retrieval_head_flags; a.head_rank_table = x->head_rank_table;
  a.B = x->batch; a.Hq = x->num_heads; a.Hkv = x->num_kv_heads; a.head_dim = x->head_dim;
  a.tokens_per_block = x->tokens_per_block;
  a.size_per_retrieval_token = x->size_per_retrieval_token; a.num_retrieval_kv_heads = x->num_retrieval_kv_heads;
  a.timestep = x->timestep;
  a.rotary_dim = x->rotary_embedding_dim; a.rotary_base = x->rotary_base;
  a.rotary_scale = x->rotary_scale != 0.f ? 1.0f / x->rotary_scale : 1.0f;
  a.tokens_per_sub_chunk = x->tokens_per_sub_chunk;
  a.hidden_dim_per_retrieval_token = x->hidden_dim_per_retrieval_token;
  return page_selector_run(a, ST(stream));
}

static StreamingPrefillArgs to_streaming(const ob_streaming_prefill_args* x) {
  StreamingPrefillArgs a{};
  a.q = H(x->q); a.k = H(x->k); a.v = H(x->v);
  a.q_row_stride = x->q_row_stride; a.k_row_stride = x->k_row_stride; a.v_row_stride = x->v_row_stride;
  a.out = HM(x->out); a.cu_seqlens_host = x->cu_seqlens;
  a.B = x->batch; a.T = x->num_tokens; a.Hq = x->num_heads; a.Hkv = x->num_kv_heads; a.head_dim = x->head_dim;
  a.num_compute_heads = x->num_compute_kv_heads; a.kv_heads_host = x->kv_heads;
  a.sink_host = x->sink; a.local_host = x->local;
  return a;
}

int ob_token_streaming_prefill_attention(const ob_streaming_prefill_args* x, void* stream) {
  if (!x) return OB_ERR_ARG;
  return streaming_prefill_run(to_streaming(x), ST(stream));
}

int ob_debug_streaming_prefill_plan(const ob_streaming_prefill_args* x, int launch, int cta_x, int cta_y, int* out,
                                    int* key_tiles, int max_key_tiles) {
  if (!x) return OB_ERR_ARG;
  return streaming_prefill_plan(to_streaming(x), launch, cta_x, cta_y, out, key_tiles, max_key_tiles);
}

int ob_kv4_page_topk(const void* scores, int32_t* out, int rows, int pitch_sub_chunks, int sub_chunks_per_page,
                     int total_pages, int k_out, void* stream) {
  if (!scores || !out) return OB_ERR_ARG;
  return page_topk_run(H(scores), out, rows, pitch_sub_chunks, sub_chunks_per_page, total_pages, k_out, ST(stream));
}

}  // extern "C"
