// Composite entry points: whole transformer stacks behind ONE C-ABI call each, so the host does a single ctypes
// call per tower pass / prompt / decode step instead of ~8 per layer (the Python launch path costs ~15 us per
// kernel, more than several of the kernels themselves).  Pure sequencing of the kernels in this library on the
// caller's stream; no allocation (workspaces are passed in), no synchronisation.
#include "common.cuh"
#include "srgpt_b200.h"

using namespace srgpt;

#define SRGPT_TRY(call)            \
  do {                             \
    int _rc = (call);              \
    if (_rc != SRGPT_OK) return _rc; \
  } while (0)

static inline const char* cptr(const void* p, size_t byte_off) { return reinterpret_cast<const char*>(p) + byte_off; }
static inline char* mptr(void* p, size_t byte_off) { return reinterpret_cast<char*>(p) + byte_off; }

extern "C" __attribute__((visibility("default"))) int srgpt_vit_layers_bf16(void* x, const srgpt_siglip_layer_weights* layers, int n_layers, void* ws_h, void* ws_qkv,
                                                                              void* ws_attn, void* ws_mlp, int n_img, int T, int D, int heads, int I, float eps,
                                                                              int fc1_epilogue, void* stream) {
  SRGPT_CHECK_ARG(x && layers && ws_h && ws_qkv && ws_attn && ws_mlp && n_layers >= 0 && n_img > 0 && T > 0 && D > 0 && heads > 0 && I > 0);
  SRGPT_CHECK_ARG(D % heads == 0);
  SRGPT_CHECK_ARG(fc1_epilogue == SRGPT_EPI_BIAS_GELU_TANH || fc1_epilogue == SRGPT_EPI_BIAS_GELU_ERF || fc1_epilogue == SRGPT_EPI_BIAS_QUICK_GELU);
  const int M = n_img * T, hd = D / heads;
  const float scale = 1.0f / sqrtf((float)hd);
  for (int l = 0; l < n_layers; ++l) {
    const srgpt_siglip_layer_weights& w = layers[l];
    SRGPT_TRY(srgpt_layernorm_bf16(x, D, w.ln1_w, w.ln1_b, ws_h, D, M, D, eps, 0, stream));
    SRGPT_TRY(srgpt_gemm_bf16(ws_h, D, w.qkv_w, D, ws_qkv, 3 * D, M, 3 * D, D, w.qkv_b, nullptr, 0, 0, SRGPT_EPI_BIAS, 0, stream));
    SRGPT_TRY(srgpt_attention_prefill_bf16(ws_qkv, cptr(ws_qkv, (size_t)D * 2), cptr(ws_qkv, (size_t)2 * D * 2), ws_attn, 3 * D, 3 * D, D, n_img, T,
                                           heads, heads, hd, scale, 0, stream));
    SRGPT_TRY(srgpt_gemm_bf16(ws_attn, D, w.out_w, D, x, D, M, D, D, w.out_b, x, D, 0, SRGPT_EPI_BIAS_RESIDUAL, 0, stream));
    SRGPT_TRY(srgpt_layernorm_bf16(x, D, w.ln2_w, w.ln2_b, ws_h, D, M, D, eps, 0, stream));
    SRGPT_TRY(srgpt_gemm_bf16(ws_h, D, w.fc1_w, D, ws_mlp, I, M, I, D, w.fc1_b, nullptr, 0, 0, fc1_epilogue, 0, stream));
    SRGPT_TRY(srgpt_gemm_bf16(ws_mlp, I, w.fc2_w, I, x, D, M, D, I, w.fc2_b, x, D, 0, SRGPT_EPI_BIAS_RESIDUAL, 0, stream));
  }
  return SRGPT_OK;
}

extern "C" __attribute__((visibility("default"))) int srgpt_siglip_layers_bf16(void* x, const srgpt_siglip_layer_weights* layers, int n_layers, void* ws_h, void* ws_qkv,
                                                                                 void* ws_attn, void* ws_mlp, int n_img, int T, int D, int heads, int I, float eps,
                                                                                 void* stream) {
  return srgpt_vit_layers_bf16(x, layers, n_layers, ws_h, ws_qkv, ws_attn, ws_mlp, n_img, T, D, heads, I, eps, SRGPT_EPI_BIAS_GELU_TANH, stream);
}

extern "C" __attribute__((visibility("default"))) int srgpt_llama_prefill_layers_bf16(void* x, const srgpt_llama_layer_weights* layers, int n_layers, void* ws_h, void* ws_qkv,
                                                                                        void* ws_attn, void* ws_act, int S, int H, int n_heads, int n_kv_heads,
                                                                                        int head_dim, int I, float eps, const void* cos_tab, const void* sin_tab,
                                                                                        const int* start_pos, const int* page_table, int page_size, int n_seqs, const int* cu_seqlens,
                                                                                        int max_seqlen, int page_table_stride, void* stream) {
  SRGPT_CHECK_ARG(x && layers && ws_h && ws_qkv && ws_attn && ws_act && n_layers >= 0 && S > 0 && H > 0 && n_heads > 0 && n_kv_heads > 0 && head_dim > 0 && I > 0);
  const bool packed = cu_seqlens != nullptr;
  SRGPT_CHECK_ARG(packed ? (n_seqs >= 1 && max_seqlen >= 1 && max_seqlen <= S && page_table_stride > 0) : (n_seqs == 1));
  const int qd = n_heads * head_dim, kd = n_kv_heads * head_dim, nqkv = qd + 2 * kd;
  const float scale = 1.0f / sqrtf((float)head_dim);
  for (int l = 0; l < n_layers; ++l) {
    const srgpt_llama_layer_weights& w = layers[l];
    SRGPT_TRY(srgpt_rmsnorm_bf16(x, H, w.in_norm, ws_h, H, S, H, eps, stream));
    SRGPT_TRY(srgpt_gemm_bf16(ws_h, H, w.qkv_w, H, ws_qkv, nqkv, S, nqkv, H, nullptr, nullptr, 0, 0, SRGPT_EPI_NONE, 0, stream));
    if (packed) {
      SRGPT_TRY(srgpt_rope_kv_append_varlen_bf16(ws_qkv, S, n_heads, n_kv_heads, head_dim, cos_tab, sin_tab, start_pos, w.kv_pages, page_table, page_table_stride,
                                                 page_size, n_seqs, cu_seqlens, stream));
      SRGPT_TRY(srgpt_attention_prefill_varlen_bf16(ws_qkv, cptr(ws_qkv, (size_t)qd * 2), cptr(ws_qkv, (size_t)(qd + kd) * 2), ws_attn, nqkv, nqkv, qd, n_seqs,
                                                    cu_seqlens, max_seqlen, S, n_heads, n_kv_heads, head_dim, scale, 1, stream));
    } else {
      SRGPT_TRY(srgpt_rope_kv_append_bf16(ws_qkv, S, n_heads, n_kv_heads, head_dim, cos_tab, sin_tab, start_pos, w.kv_pages, page_table, page_size, stream));
      SRGPT_TRY(srgpt_attention_prefill_bf16(ws_qkv, cptr(ws_qkv, (size_t)qd * 2), cptr(ws_qkv, (size_t)(qd + kd) * 2), ws_attn, nqkv, nqkv, qd, 1, S, n_heads,
                                             n_kv_heads, head_dim, scale, 1, stream));
    }
    SRGPT_TRY(srgpt_gemm_bf16(ws_attn, qd, w.o_w, qd, x, H, S, H, qd, nullptr, x, H, 0, SRGPT_EPI_BIAS_RESIDUAL, 0, stream));
    SRGPT_TRY(srgpt_rmsnorm_bf16(x, H, w.post_norm, ws_h, H, S, H, eps, stream));
    SRGPT_TRY(srgpt_gemm_bf16(ws_h, H, w.gateup_w, H, ws_act, I, S, 2 * I, H, nullptr, nullptr, 0, 0, SRGPT_EPI_SWIGLU, 0, stream));
    SRGPT_TRY(srgpt_gemm_bf16(ws_act, I, w.down_w, I, x, H, S, H, I, nullptr, x, H, 0, SRGPT_EPI_BIAS_RESIDUAL, 0, stream));
  }
  return SRGPT_OK;
}

// The same layer sequence for new rows that continue sequences already in the cache (chunked prefill, a follow-up turn): RoPE
// and the KV append at start_pos[b] + i, then attention of the new rows over ALL cached positions of their sequence through
// the page tables (srgpt_attention_prefill_paged_bf16; modeling_llama.py:451-456 + 564-566 with q_len < kv_len).
extern "C" __attribute__((visibility("default"))) int srgpt_llama_prefill_layers_paged_bf16(
    void* x, const srgpt_llama_layer_weights* layers, int n_layers, void* ws_h, void* ws_qkv, void* ws_attn, void* ws_act, void* ws_split,
    long long ws_split_bytes, int S, int H, int n_heads, int n_kv_heads, int head_dim, int I, float eps, const void* cos_tab, const void* sin_tab,
    const int* start_pos, const int* page_tables, int page_table_stride, int page_size, int n_seqs, const int* cu_seqlens, int max_seqlen,
    int max_ctx_len, void* stream) {
  SRGPT_CHECK_ARG(x && layers && ws_h && ws_qkv && ws_attn && ws_act && start_pos && page_tables && cu_seqlens);
  SRGPT_CHECK_ARG(n_layers >= 0 && S > 0 && H > 0 && n_heads > 0 && n_kv_heads > 0 && head_dim > 0 && I > 0);
  SRGPT_CHECK_ARG(n_seqs >= 1 && max_seqlen >= 1 && max_seqlen <= S && max_ctx_len >= max_seqlen && page_table_stride > 0);
  const int qd = n_heads * head_dim, kd = n_kv_heads * head_dim, nqkv = qd + 2 * kd;
  const float scale = 1.0f / sqrtf((float)head_dim);
  for (int l = 0; l < n_layers; ++l) {
    const srgpt_llama_layer_weights& w = layers[l];
    SRGPT_TRY(srgpt_rmsnorm_bf16(x, H, w.in_norm, ws_h, H, S, H, eps, stream));
    SRGPT_TRY(srgpt_gemm_bf16(ws_h, H, w.qkv_w, H, ws_qkv, nqkv, S, nqkv, H, nullptr, nullptr, 0, 0, SRGPT_EPI_NONE, 0, stream));
    SRGPT_TRY(srgpt_rope_kv_append_varlen_bf16(ws_qkv, S, n_heads, n_kv_heads, head_dim, cos_tab, sin_tab, start_pos, w.kv_pages, page_tables,
                                               page_table_stride, page_size, n_seqs, cu_seqlens, stream));
    SRGPT_TRY(srgpt_attention_prefill_paged_bf16(ws_qkv, nqkv, ws_attn, qd, w.kv_pages, page_tables, page_table_stride, page_size, n_seqs, cu_seqlens,
                                                 start_pos, max_seqlen, max_ctx_len, n_heads, n_kv_heads, head_dim, scale, ws_split, ws_split_bytes,
                                                 stream));
    SRGPT_TRY(srgpt_gemm_bf16(ws_attn, qd, w.o_w, qd, x, H, S, H, qd, nullptr, x, H, 0, SRGPT_EPI_BIAS_RESIDUAL, 0, stream));
    SRGPT_TRY(srgpt_rmsnorm_bf16(x, H, w.post_norm, ws_h, H, S, H, eps, stream));
    SRGPT_TRY(srgpt_gemm_bf16(ws_h, H, w.gateup_w, H, ws_act, I, S, 2 * I, H, nullptr, nullptr, 0, 0, SRGPT_EPI_SWIGLU, 0, stream));
    SRGPT_TRY(srgpt_gemm_bf16(ws_act, I, w.down_w, I, x, H, S, H, I, nullptr, x, H, 0, SRGPT_EPI_BIAS_RESIDUAL, 0, stream));
  }
  return SRGPT_OK;
}

extern "C" __attribute__((visibility("default"))) int srgpt_llama_decode_step_bf16(void* h, const srgpt_llama_layer_weights* layers, int n_layers, void* q_buf, void* attn_buf,
                                                                                     void* act_buf, int H, int n_heads, int n_kv_heads, int head_dim, int I, float eps,
                                                                                     const void* cos_tab, const void* sin_tab, int* pos, const int* page_table,
                                                                                     int page_size, const void* final_norm, const void* lm_head, int V,
                                                                                     const void* embed_table, void* lm_workspace, float* logits_out,
                                                                                     long long* out_ids, int* step, void* stream) {
  SRGPT_CHECK_ARG(h && layers && q_buf && attn_buf && act_buf && pos && page_table && final_norm && lm_head && lm_workspace && out_ids && step);
  const int qd = n_heads * head_dim, nqkv = (n_heads + 2 * n_kv_heads) * head_dim;
  const float scale = 1.0f / sqrtf((float)head_dim);
  for (int l = 0; l < n_layers; ++l) {
    const srgpt_llama_layer_weights& w = layers[l];
    SRGPT_TRY(srgpt_gemv_bf16(h, w.qkv_w, H, q_buf, nqkv, H, w.in_norm, eps, nullptr, SRGPT_GEMV_QKV_ROPE, n_heads, n_kv_heads, head_dim, cos_tab, sin_tab, pos,
                              w.kv_pages, page_table, page_size, stream));
    SRGPT_TRY(srgpt_attention_decode_bf16(q_buf, attn_buf, w.kv_pages, page_table, page_size, pos, n_heads, n_kv_heads, head_dim, scale, stream));
    SRGPT_TRY(srgpt_gemv_bf16(attn_buf, w.o_w, qd, h, H, qd, nullptr, 0.f, h, SRGPT_GEMV_PLAIN, 0, 0, 0, nullptr, nullptr, nullptr, nullptr, nullptr, 0, stream));
    SRGPT_TRY(srgpt_gemv_bf16(h, w.gateup_w, H, act_buf, 2 * I, H, w.post_norm, eps, nullptr, SRGPT_GEMV_SWIGLU, 0, 0, 0, nullptr, nullptr, nullptr, nullptr, nullptr, 0,
                              stream));
    SRGPT_TRY(srgpt_gemv_bf16(act_buf, w.down_w, I, h, H, I, nullptr, 0.f, h, SRGPT_GEMV_PLAIN, 0, 0, 0, nullptr, nullptr, nullptr, nullptr, nullptr, 0, stream));
  }
  return srgpt_lm_head_argmax_bf16(h, lm_head, H, V, H, final_norm, eps, logits_out, lm_workspace, embed_table, h, out_ids, step, pos, stream);
}
