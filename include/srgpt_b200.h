/* srgpt_b200 — C-ABI of the B200 (sm_100a) kernels behind SpatialRGPT's multimodal generate() path.
 *
 * The reference (AnjieCheng/SpatialRGPT) has no FFI / plugin layer: every op below replaces a
 * PyTorch library call on the path  LlavaLlamaModel.generate -> prepare_inputs_labels_for_multimodal
 * -> llm.generate  (llava/model/language_model/llava_llama.py:194-213).  Each entry cites the
 * reference call site it replaces (paths relative to the reference checkout;
 * "modeling_llama.py" = llava/train/transformers_replace/models/llama/modeling_llama.py).
 *
 * Conventions
 *   - plain C: device pointers as void*, sizes as int / long long, CUDA stream as void* (cudaStream_t).
 *   - all tensors are row-major; strides (ld*) are in ELEMENTS.
 *   - element type: the library is built twice from the same sources.  libsrgpt_b200.so computes in bfloat16 (the dtype the
 *     reference's eval scripts load the model in, llava/eval/eval_spatial.py:206-212); libsrgpt_b200_f16.so (-DSRGPT_ELEM_F16) in
 *     IEEE half, the reference loader's default (llava/model/builder.py:62, llava/eval/eval_region_cls.py:316-317).  Both export the
 *     SAME entry points: in the names and comments below "bf16" stands for "the 16-bit element type of the build" - __nv_bfloat16
 *     or __half - and srgpt_elem_type() says which.  Accumulation is fp32 and the rounding points are identical in both builds.
 *   - every function is asynchronous on `stream`, allocates nothing, and returns 0 on success or a
 *     negative srgpt error code; the message is available from srgpt_last_error().  Nothing throws.
 *   - callable from any host thread; no global state except the last-error string (thread-local).
 */
#ifndef SRGPT_B200_H_
#define SRGPT_B200_H_

#ifdef __cplusplus
extern "C" {
#endif

#define SRGPT_ABI_VERSION 1

/* ---- library -------------------------------------------------------------------------------- */
int srgpt_abi_version(void);
/* 0 = bfloat16 build, 1 = IEEE half build (see "element type" above). */
int srgpt_elem_type(void);
const char* srgpt_last_error(void);
/* sm count + compute capability of the current device; fails (<0) unless it is sm_100. */
int srgpt_device_info(int* sm_count, int* cc_major, int* cc_minor);

/* Optional in-kernel timeline for the decode-step kernels (debug / profiling aid; nsys is not available on
 * the target boxes).  Between trace_begin and trace_end every traced launch (gemv / lm_head / decode attention)
 * takes the next 4-u64 record of device_buf: {min CTA-start ns, min after-dependency-wait ns, max CTA-end ns,
 * CTA count} from %globaltimer.  The caller pre-fills records with {~0, ~0, 0, 0}.  trace_end returns the
 * number of records used.  Not thread-safe; launches captured into a CUDA graph keep their record. */
int srgpt_trace_begin(void* device_buf, int capacity_records);
int srgpt_trace_end(void);

/* ---- dense GEMM on tcgen05/TMEM (gemm_tcgen05.cu) --------------------------------------------
 * C[M,N] = epilogue(A[M,K] · W[N,K]^T), bf16 in, fp32 accumulate.  W is the nn.Linear weight as
 * stored ([out, in]).  Replaces every F.linear / Conv2d(k=s) / ConvTranspose2d(k=s) on the path:
 * SigLIP q/k/v/out/fc1/fc2 (HF SiglipVisionModel, call site vision_encoder.py:119-130),
 * deconv refinement (base_extractor.py:92-97), rgb/depth projectors (base_extractor.py:158),
 * mm_projector (base_projector.py:76-79), Llama q/k/v/o/gate/up/down at prefill
 * (modeling_llama.py:429-431,498,221). */
enum {
  SRGPT_EPI_NONE = 0,           /* C = acc                                                        */
  SRGPT_EPI_BIAS = 1,           /* C = acc + bias[n]                                              */
  SRGPT_EPI_BIAS_GELU_TANH = 2, /* C = gelu_tanh(bf16(acc + bias))   (SigLIP fc1)                 */
  SRGPT_EPI_BIAS_GELU_ERF = 3,  /* C = gelu_erf(bf16(acc + bias))    (deconv #2, mm_projector)    */
  SRGPT_EPI_BIAS_RESIDUAL = 4,  /* C = bf16(acc + bias) + residual[row (% res_row_mod), n]        */
  SRGPT_EPI_SWIGLU = 5,         /* W rows interleaved (gate_i, up_i): C[:, i] = silu(g) * u; C has N/2 cols */
  SRGPT_EPI_BIAS_QUICK_GELU = 6 /* C = x * sigmoid(1.702 x), x = bf16(acc + bias)   (CLIP fc1, HF QuickGELUActivation) */
};
/* Optional workspace of the short-prompt ("tall stream-K") configuration: M <= 384 rows, all rows in one CTA, the (n-tile,
 * k-block) units balanced over the SMs, split tiles combined through fp32 partials in this buffer.  The caller owns the memory
 * (no hidden allocation): srgpt_gemm_workspace_bytes() bytes, 1024-byte aligned, ZEROED when registered, used by one stream at a
 * time, alive until unregistered with (NULL, 0).  Without a workspace short prompts run on the default 128-row tiles. */
long long srgpt_gemm_workspace_bytes(void);
int srgpt_gemm_set_workspace(void* workspace, long long bytes);
int srgpt_gemm_bf16(const void* A, int lda, const void* W, int ldw, void* C, int ldc, int M, int N, int K,
                    const void* bias /*bf16[N] or NULL*/, const void* residual /*bf16 or NULL*/, int ldr,
                    int res_row_mod /*0 = none*/, int epilogue, int out_fp32, void* stream);

/* ---- row-wise normalisation / elementwise (rowops.cu) ----------------------------------------
 * LayerNorm over the last dim, fp32 statistics, bf16 in/out.  act: 0 none, 1 GELU(erf) applied to
 * the bf16-rounded LN output.  Replaces nn.LayerNorm in SigLIP (eps 1e-6) and LayerNorm2d + GELU
 * (base_extractor.py:12-24,93-95; our activations are pixel-major so LN2d is a row LayerNorm). */
int srgpt_layernorm_bf16(const void* x, int ldx, const void* weight, const void* bias, void* y, int ldy, int rows,
                         int cols, float eps, int act, void* stream);
/* mm_projector front end (base_projector.py:32-52,75): DownSampleBlock (zero-pad side->even,
 * 2x2 token merge, the reference's transposed output order) fused with LayerNorm(4C).
 * x: [n_img, side*side, C] -> y: [n_img, ceil(side/2)^2, 4C]. */
int srgpt_downsample_layernorm_bf16(const void* x, const void* weight, const void* bias, void* y, int n_img, int side,
                                    int C, float eps, void* stream);
/* LlamaRMSNorm (modeling_llama.py:70-75): y = weight * bf16(x * rsqrt(mean(x^2) + eps)). */
int srgpt_rmsnorm_bf16(const void* x, int ldx, const void* weight, void* y, int ldy, int rows, int cols, float eps,
                       void* stream);
/* SigLIP patch embedding front end: Conv2d(3, D, k=14, s=14) == GEMM over this im2col
 * (HF SiglipVisionEmbeddings; call site siglip_encoder.py:11-16).  images: [n, 3, R, R] fp32 or
 * bf16 (src_is_bf16) -> A: [n*(R/ps)^2, ldk] bf16, column = c*ps*ps + ky*ps + kx, zero padded to ldk. */
int srgpt_patchify_bf16(const void* images, int src_is_bf16, void* A, int n, int R, int ps, int ldk, void* stream);
/* CLIP embeddings (HF CLIPVisionEmbeddings.forward; call site clip_encoder.py:11): out [n_img, T + 1, D] =
 * cat([class_embedding, patch_embeds[n]]) + position_embedding, one element-type add per value like torch's. */
int srgpt_clip_embed_bf16(const void* patch_embeds, const void* class_embedding, const void* position_embedding, void* out,
                          int n_img, int T, int D, void* stream);
/* Embedding splice (llava_arch.py:434-539): out[r,:] = src[src_id[r]][src_row[r],:] for the four
 * sources (0 = token embedding table, 1 = image features, 2 = mask embeds, 3 = depth embeds).
 * The (src_id,src_row) plan is built on the host from input_ids. */
int srgpt_splice_rows_bf16(const void* src0, const void* src1, const void* src2, const void* src3, const int* src_id,
                           const int* src_row, void* out, int rows, int cols, void* stream);

/* ---- region extractor HBM kernels (region.cu) -------------------------------------------------
 * MaskPooling weights (base_extractor.py:52-72): bilinear (align_corners=False, no antialias)
 * resample of masks [n_img, M, IH, IW] to the feature grid (side x side), cast to bf16, divide by
 * bf16(sum + 1e-8).  w: [n_img, M, side*side] bf16 (the reference's `mask / denorm`) in the feature
 * tensor's row order: order = 0 row-major (y*side+x); order = 2 the 2-level 2x2-nested order the deconv
 * GEMMs produce (see DESIGN.md "hres layout").  rscale = (float)(1.0 / scale_factor) exactly as ATen
 * computes it.  workspace: srgpt_mask_weights_workspace(n_img, M, side) bytes. */
long long srgpt_mask_weights_workspace(int n_img, int M, int side);
/* Layout of w (here and in srgpt_mask_pool_bf16): [n_img, M, ld] bf16 with ld = L rounded up to a multiple of 8 elements (16-byte
 * rows for the TMA view of the pooling kernel; L = side^2 is odd for odd sides); the pad elements are never read. */
int srgpt_mask_weights(const void* masks, int mask_is_bf16, void* w, void* workspace, int n_img, int M, int IH, int IW,
                       int side, float rscale, int order, void* stream);
/* Mask pooling proper (base_extractor.py:74-78): out[i,m,:] = sum_l w[i,m,l] * x[i,l,:] — bf16 tensor-core
 * product with fp32 accumulation like the reference's einsum.  x: [n_img, L, C] bf16 streamed once;
 * workspace: fp32 partials, srgpt_mask_pool_workspace() bytes. */
long long srgpt_mask_pool_workspace(int n_img, int M, int L, int C);
int srgpt_mask_pool_bf16(const void* x, const void* w, void* out, void* workspace, int n_img, int M, int L, int C,
                         void* stream);
/* AdaptiveAvgPool2d(out_side) over the (side x side) feature map (base_extractor.py:123,145).
 * x: [n_img, side*side, C] in `order` (as above) -> y: [n_img, out_side*out_side, C] row-major. */
int srgpt_adaptive_avgpool_bf16(const void* x, void* y, int n_img, int side, int out_side, int C, int order,
                                void* stream);
/* Row permutation between the nested order and row-major (tests / API parity for `hres`). */
int srgpt_reorder_rows_bf16(const void* x, void* y, int n_img, int side, int C, int from_order, int to_order,
                            void* stream);
/* Depth map preparation (llava/eval/eval_spatial.py:99-105): bilinear resize of depth [h, w] fp32 to
 * (H, W), min-max normalise * 255, truncate to u8, replicate to 3 channels -> out [H, W, 3] u8.
 * workspace: (H*W + 2) floats. */
int srgpt_depth_to_u8x3(const void* depth, int h, int w, void* out, int H, int W, void* workspace, void* stream);

/* ---- attention (attention.cu) ------------------------------------------------------------------
 * Prefill attention, softmax in fp32, flash-style (no S x S matrix in HBM).  head_dim 72 / 128 run on the
 * tcgen05 tensor cores (attention_tc.cu: TMA boxes out of the fused qkv buffer, S and P.V accumulators in TMEM,
 * warp-specialised softmax); other head sizes use the mma.sync kernel.
 * Replaces SigLIP's eager attention (non-causal, head_dim 72) and flash_attn_func(causal=True) with
 * GQA (modeling_llama.py:564-566).  q/k/v/out rows are tokens; head h of a row starts at h*head_dim.
 * Sequences are `batch` equal-length segments of `seqlen` consecutive rows. */
int srgpt_attention_prefill_bf16(const void* q, const void* k, const void* v, void* out, int q_ld, int kv_ld, int o_ld,
                                 int batch, int seqlen, int n_heads, int n_kv_heads, int head_dim, float scale,
                                 int causal, void* stream);
/* Same, for `n_seqs` variable-length sequences packed back to back: sequence b owns rows
 * [cu_seqlens[b], cu_seqlens[b+1]) (device int32 [n_seqs+1]); max_seqlen bounds the grid, total_rows =
 * cu_seqlens[n_seqs] bounds the TMA views (host value).  This is the varlen form of modeling_llama.py:540-562
 * (flash_attn_varlen_func over unpadded rows). */
int srgpt_attention_prefill_varlen_bf16(const void* q, const void* k, const void* v, void* out, int q_ld, int kv_ld,
                                        int o_ld, int n_seqs, const int* cu_seqlens, int max_seqlen, int total_rows,
                                        int n_heads, int n_kv_heads, int head_dim, float scale, int causal, void* stream);
/* RoPE + KV-cache append for `rows` new tokens of one sequence (modeling_llama.py:448-456):
 * rotates q and k in place inside the fused qkv buffer [rows, (nh + 2*nkv)*hd] using the bf16
 * cos/sin tables [max_pos, hd/2], and writes k, v into the paged cache.
 * Cache layout: pages [n_pages, 2 (k,v), page_size, nkv, hd] bf16 for ONE layer; page_table[i] =
 * physical page of logical page i of this sequence.  start_pos: device int (position of row 0). */
int srgpt_rope_kv_append_bf16(void* qkv, int rows, int n_heads, int n_kv_heads, int head_dim, const void* cos_tab,
                              const void* sin_tab, const int* start_pos, void* kv_pages, const int* page_table,
                              int page_size, void* stream);
/* Packed-sequence form: row r belongs to sequence b with cu_seqlens[b] <= r < cu_seqlens[b+1], its position is
 * start_pos[b] + r - cu_seqlens[b], and its page table is page_tables + b * page_table_stride. */
int srgpt_rope_kv_append_varlen_bf16(void* qkv, int rows, int n_heads, int n_kv_heads, int head_dim, const void* cos_tab,
                                     const void* sin_tab, const int* start_pos, void* kv_pages, const int* page_tables,
                                     int page_table_stride, int page_size, int n_seqs, const int* cu_seqlens, void* stream);
/* Prefill attention of NEW rows over the paged cache (chunked prefill, continuing a cached sequence): replaces torch.cat of the
 * past K/V (modeling_llama.py:451-456) + flash_attn_func(causal=True) with q_len < kv_len, whose causal mask is aligned
 * bottom-right (:564-566), for the rows prepare_inputs_for_generation keeps after dropping the cached prefix (:1112-1149).
 * Rows [cu_q[b], cu_q[b+1]) of q (device int32 [n_seqs+1]) are sequence b's new rows at positions start_pos[b] + i (device
 * int32 [n_seqs]); the row at position p attends to positions 0..p of its sequence, read from ONE layer's kv_pages
 * ([n_pages, 2, page_size, nkv, hd], as srgpt_rope_kv_append_bf16 describes) through page_tables + b * page_table_stride.
 * The new rows' own K/V must already be appended (srgpt_rope_kv_append_varlen_bf16).  max_q_len (longest chunk) and
 * max_ctx_len (largest start_pos[b] + chunk length) are host bounds used for the grid only.  head_dim 128, page_size 16,
 * n_heads / n_kv_heads <= 8.  q / out: rows [.., q_ld] / [.., o_ld] (e.g. the q columns of the fused qkv buffer).
 * workspace: fp32 partials of the context split, srgpt_attention_prefill_paged_workspace() bytes (0 = no split for this shape),
 * 16-byte aligned; NULL runs without a split. */
long long srgpt_attention_prefill_paged_workspace(int n_seqs, int max_q_len, int max_ctx_len, int n_heads, int n_kv_heads);
int srgpt_attention_prefill_paged_bf16(const void* q, int q_ld, void* out, int o_ld, const void* kv_pages, const int* page_tables,
                                       int page_table_stride, int page_size, int n_seqs, const int* cu_q, const int* start_pos,
                                       int max_q_len, int max_ctx_len, int n_heads, int n_kv_heads, int head_dim, float scale,
                                       void* workspace, long long workspace_bytes, void* stream);
/* Decode attention for ONE new token over the paged cache (replaces torch.cat of the cache +
 * flash_attn_func with q_len 1, modeling_llama.py:451-456,564).  q: [nh*hd] bf16 (already rotated),
 * kv_len_minus1: device int = position of the new token (its k/v are already in the cache). */
int srgpt_attention_decode_bf16(const void* q, void* out, const void* kv_pages, const int* page_table, int page_size,
                                const int* kv_len_minus1, int n_heads, int n_kv_heads, int head_dim, float scale,
                                void* stream);

/* ---- decode-time weight-streaming kernels (gemv.cu) -------------------------------------------
 * One token: y = W · x with W [N, K] bf16 streamed once from HBM (the decode roofline).
 *   norm_weight != NULL : x is first RMS-normalised (LlamaRMSNorm) inside the kernel.
 *   mode SRGPT_GEMV_PLAIN    : y[n] = bf16(acc) (+ residual[n])            (o_proj, down_proj)
 *   mode SRGPT_GEMV_SWIGLU   : W rows interleaved (gate_i, up_i); y[i] = silu(g)*u   (gate/up)
 *   mode SRGPT_GEMV_QKV_ROPE : W = fused [q;k;v]; rotates q,k at *pos with the cos/sin tables, writes
 *                              q to y [nh*hd] and appends k,v to the paged cache      (q/k/v_proj + RoPE)
 * Replaces modeling_llama.py:429-431,448-456,498,221 at q_len == 1. */
enum { SRGPT_GEMV_PLAIN = 0, SRGPT_GEMV_SWIGLU = 1, SRGPT_GEMV_QKV_ROPE = 2 };
int srgpt_gemv_bf16(const void* x, const void* W, int ldw, void* y, int N, int K, const void* norm_weight, float eps,
                    const void* residual, int mode,
                    /* QKV_ROPE only: */ int n_heads, int n_kv_heads, int head_dim, const void* cos_tab,
                    const void* sin_tab, const int* pos, void* kv_pages, const int* page_table, int page_size,
                    void* stream);
/* Final norm + lm_head + greedy argmax (modeling_llama.py:922,1044-1045 + HF greedy search):
 * logits = float(bf16(W · rmsnorm(x))); writes argmax (lowest index on ties) to out_ids[*step],
 * copies the chosen token's embedding row to next_x, then ++*step and ++*pos.
 * logits_out (fp32 [V]) may be NULL.  workspace: srgpt_lm_head_workspace(V) bytes. */
long long srgpt_lm_head_workspace(int V);
int srgpt_lm_head_argmax_bf16(const void* x, const void* W, int ldw, int V, int K, const void* norm_weight, float eps,
                              float* logits_out, void* workspace, const void* embed_table, void* next_x,
                              long long* out_ids, int* step, int* pos, void* stream);
/* Plain argmax over fp32 rows (first index on ties), e.g. first token after prefill. */
int srgpt_argmax_f32(const float* x, int rows, int cols, long long* out, void* stream);
/* Same over bf16 rows [rows, ldx] (the bf16-rounded logits of a batched lm_head GEMM, modeling_llama.py:1044). */
int srgpt_argmax_bf16(const void* x, int ldx, int rows, int cols, long long* out, void* stream);
/* Beam-search candidates (rowops.cu): replaces log_softmax + the [num_beams x vocab] torch.topk of HF GenerationMixin.beam_search
 * (transformers 4.37.2; reached from llava_llama.py:212 when the eval scripts pass --num_beams > 1).  logits: [n_beams, ldx] in the
 * element type (the rounded lm_head output, modeling_llama.py:1044-1045).  Per row the n_cand best
 * (log_softmax(logits.float())[token] + beam_scores[row], token) in (score desc, token asc) order -> cand_scores / cand_tokens
 * [n_beams, n_cand] (token -1 / score -inf when a row has fewer finite logits). */
int srgpt_beam_candidates_bf16(const void* logits, int ldx, int n_beams, int V, const float* beam_scores, int n_cand,
                               float* cand_scores, int* cand_tokens, void* stream);
/* Temperature + nucleus (top-p) sampling of one token from fp32 logits [V] (sampling.cu): replaces HF's TemperatureLogitsWarper /
 * TopKLogitsWarper / TopPLogitsWarper / multinomial behind do_sample=True (llava/eval/eval_spatial.py:231-236, llava/eval/model_vqa.py:72-78).
 * params = device float[3] {temperature, top_p, top_k (0 = off)}; seed = device u64; the draw is a counter-based generator of
 * (*seed, *step + step_offset) - both read at run time, so a captured decode graph serves every request.
 * Writes out_ids[*step + step_offset] and, when given, next_x[K] = embed_table[token].  Call it right after
 * srgpt_lm_head_argmax_bf16 / srgpt_llama_decode_step_bf16 (which advanced *step) with step_offset = -1. */
int srgpt_sample_top_p_f32(const float* logits, int V, const float* params, const unsigned long long* seed, const int* step, int step_offset,
                           long long* out_ids, const void* embed_table, void* next_x, int K, void* stream);

/* ---- host preprocessing on the GPU (preprocess.cu; llava/mm_utils.py:421-542: process_images / process_regions) ----------
 * The pinned image processor (transformers 4.37.2 SiglipImageProcessor) = Pillow BICUBIC resize of the uint8 image + rescale +
 * normalise; masks = cv2 INTER_NEAREST.  Pillow's resampler is integer arithmetic over host-built coefficient tables
 * (spatialrgpt_b200/preprocess.py, same double arithmetic as libImaging/Resample.c), so the results are bit-exact. */
int srgpt_resample_u8(const void* in, void* out, int H, int W, int C, int axis, int out_size, const int* kk, const int* bounds, int ksize,
                      void* stream);
/* mean3 / std3: HOST arrays of 3 floats (passed by value to the kernel) */
int srgpt_u8_to_normalized_chw(const void* in, float* out, int H, int W, int C, double scale, const float* mean3, const float* std3,
                               int do_normalize, void* stream);
int srgpt_resize_nearest_u8(const void* in, float* out, int H, int W, int Hout, int Wout, const int* ys, const int* xs, void* stream);

/* ---- batched decode (B sequences, one new token each; llava_arch.py:549-611 pads, modeling_llama.py:540-562 un-pads: here
 * the rows are never padded).  The projections are srgpt_gemm_bf16 over the B rows (tall stream-K configuration: every weight is
 * streamed once for the whole batch), RoPE / KV append is srgpt_rope_kv_append_varlen_bf16 with one row per sequence. */
int srgpt_attention_decode_batched_bf16(const void* q, int q_ld, void* out, int o_ld, const void* kv_pages, const int* page_tables,
                                        int pt_stride, int page_size, const int* kv_len_minus1, int batch, int n_heads, int n_kv_heads,
                                        int head_dim, float scale, void* stream);
/* ids [B] (the step's arg max per sequence) -> out_ids[*step * B + b], h[b, :] = embed_table[ids[b], :], ++pos[b], ++*step. */
int srgpt_decode_batch_advance(const long long* ids, const void* embed_table, void* h, int H, long long* out_ids, int* step, int* pos,
                               int B, void* ticket, void* stream);

/* ---- tensor-parallel decode (SURVEY.md §8e "optional TP", BASELINE config c5; no reference counterpart, parity = TP-1) ----------
 * Megatron-style sharding of the Llama decoder over `world` ranks: column-parallel fused QKV (a rank owns n_heads/world query
 * heads and their kv heads) and gate/up, row-parallel o_proj / down_proj whose fp32 partial sums are all-reduced, vocabulary-
 * parallel lm_head with an (value, index) all-gather.  The KV cache keeps the FULL layout on every rank (a rank only ever reads
 * and writes its own kv heads), so prefill stays the replicated path. */
int srgpt_gemv_tp_bf16(const void* x, const void* W, int ldw, void* y, int N, int K, const void* norm_weight, float eps, int mode,
                       int n_heads, int n_kv_heads, int head_dim, const void* cos_tab, const void* sin_tab, const int* pos, void* kv_pages,
                       const int* page_table, int page_size, int kv_heads_total, int kv_head_off, float* partial_f32, void* stream);
int srgpt_attention_decode_tp_bf16(const void* q, void* out, const void* kv_pages, const int* page_table, int page_size,
                                   const int* kv_len_minus1, int n_heads_local, int group, int n_kv_total, int kv_head_off, int head_dim,
                                   float scale, void* stream);
/* h[n] = bf16(bf16(partial[n]) + h[n]) after the all-reduce of the row-parallel partial sums (modeling_llama.py:668,682). */
int srgpt_tp_residual_add_bf16(void* h, const float* partial, int n, void* stream);
/* rows [index_base, index_base + V_local) of lm_head: best = device int[2] {best bf16-rounded logit (float bits), GLOBAL index}. */
int srgpt_lm_head_local_best_bf16(const void* x, const void* W_local, int ldw, int V_local, int K, const void* norm_weight, float eps,
                                  void* workspace, int index_base, int* best, void* stream);
/* best_all = the all-gathered int[world][2]; writes out_ids[*step], next_x = embed_table[token], ++*step, ++*pos. */
int srgpt_tp_pick_token(const int* best_all, int world, const void* embed_table, void* next_x, int K, long long* out_ids, int* step,
                        int* pos, void* stream);

/* Fused collectives over NVLink peer memory (tp_comm.cu): every rank's partial sums / arg-max candidates live in a SYMMETRIC buffer
 * (srgpt_tp_comm_bytes bytes, zeroed, same layout on every GPU, peer-mapped by the caller - torch symmetric memory); one kernel
 * signals the peers, waits for all of them, pulls their 16 KB partials through NVLink, reduces in rank order and applies the residual
 * add (or picks the token).  peer_bases = HOST array [world] of peer-mapped base addresses; idx < 128 numbers the collectives of a
 * step; epoch / step are device ints (request counter, the decoder's step counter), so CUDA-graph replays need no host values. */
long long srgpt_tp_comm_bytes(int world, int n_slots, int slot_floats);
long long srgpt_tp_comm_slot_offset(int world, int slot, int slot_floats);
int srgpt_tp_allreduce_residual_bf16(const unsigned long long* peer_bases, int rank, int world, long long slot_off_bytes, int idx,
                                     const int* epoch, const int* step, void* h, int n, void* stream);
int srgpt_tp_allgather_pick_token(const unsigned long long* peer_bases, int rank, int world, long long slot_off_bytes, int idx,
                                  const int* epoch, const void* embed_table, void* next_x, int K, long long* out_ids, int* step, int* pos,
                                  void* stream);

/* ---- composite entry points (layers.cu): one call per tower pass / prompt / decode step -------------------
 * Pure sequencing of the kernels above on `stream` (no allocation, no sync); they exist because a Python-side
 * launch costs more host time than several of these kernels take on the device.  Weights are the re-laid-out
 * tensors described in DESIGN.md §3 (fused qkv, interleaved gate/up).  Workspaces (bf16): ws_h [M, D|H],
 * ws_qkv [M, 3D | (nh+2nkv)hd], ws_attn [M, D | nh*hd], ws_mlp [M, I] / ws_act [S, I]. */
typedef struct {
  const void *ln1_w, *ln1_b, *qkv_w, *qkv_b, *out_w, *out_b, *ln2_w, *ln2_b, *fc1_w, *fc1_b, *fc2_w, *fc2_b;
} srgpt_siglip_layer_weights;
typedef struct {
  const void *in_norm, *qkv_w, *o_w, *post_norm, *gateup_w, *down_w;
  void* kv_pages; /* this layer's KV pages [n_pages, 2, page_size, nkv, hd] */
} srgpt_llama_layer_weights;
/* n_layers SigLIP encoder layers in place on x [n_img*T, D] (HF SiglipEncoderLayer; call site vision_encoder.py:119-130). */
int srgpt_siglip_layers_bf16(void* x, const srgpt_siglip_layer_weights* layers, int n_layers, void* ws_h, void* ws_qkv,
                             void* ws_attn, void* ws_mlp, int n_img, int T, int D, int heads, int I, float eps, void* stream);
/* The same pre-LN encoder layer with the MLP activation as a parameter (fc1_epilogue = SRGPT_EPI_BIAS_GELU_TANH: SigLIP,
 * SRGPT_EPI_BIAS_QUICK_GELU: CLIP (HF CLIPEncoderLayer; call site clip_encoder.py:11, vision_encoder.py:119-130),
 * SRGPT_EPI_BIAS_GELU_ERF: hidden_act "gelu").  T counts ALL rows of an image (CLIP: patches + the class token). */
int srgpt_vit_layers_bf16(void* x, const srgpt_siglip_layer_weights* layers, int n_layers, void* ws_h, void* ws_qkv, void* ws_attn,
                          void* ws_mlp, int n_img, int T, int D, int heads, int I, float eps, int fc1_epilogue, void* stream);
/* n_layers Llama decoder layers over the prompt rows x [S, H] in place, appending K/V to the paged cache
 * (LlamaDecoderLayer.forward, modeling_llama.py:623-684).  n_seqs == 1, cu_seqlens == NULL: one prompt of S rows.
 * Otherwise S is the total row count of n_seqs prompts packed back to back (cu_seqlens int32 [n_seqs+1] on the
 * device, max_seqlen = longest prompt, start_pos [n_seqs], page_tables [n_seqs, page_table_stride]): every GEMM
 * runs once over all S rows (batch 32 x 259 rows = the c3 workload), attention and the KV append per sequence. */
int srgpt_llama_prefill_layers_bf16(void* x, const srgpt_llama_layer_weights* layers, int n_layers, void* ws_h, void* ws_qkv,
                                    void* ws_attn, void* ws_act, int S, int H, int n_heads, int n_kv_heads, int head_dim, int I,
                                    float eps, const void* cos_tab, const void* sin_tab, const int* start_pos,
                                    const int* page_tables, int page_size, int n_seqs, const int* cu_seqlens, int max_seqlen,
                                    int page_table_stride, void* stream);
/* The same layers over new rows that CONTINUE sequences already in the cache (chunked prefill, a follow-up turn): S rows of
 * n_seqs chunks packed back to back (cu_seqlens, max_seqlen as above), chunk b at positions start_pos[b].., attention over all
 * cached positions through srgpt_attention_prefill_paged_bf16 (max_ctx_len, ws_split / ws_split_bytes = its bound and workspace). */
int srgpt_llama_prefill_layers_paged_bf16(void* x, const srgpt_llama_layer_weights* layers, int n_layers, void* ws_h, void* ws_qkv,
                                          void* ws_attn, void* ws_act, void* ws_split, long long ws_split_bytes, int S, int H, int n_heads,
                                          int n_kv_heads, int head_dim, int I, float eps, const void* cos_tab, const void* sin_tab,
                                          const int* start_pos, const int* page_tables, int page_table_stride, int page_size, int n_seqs,
                                          const int* cu_seqlens, int max_seqlen, int max_ctx_len, void* stream);
/* One whole decode step (5 kernels per layer + lm_head + argmax), h [H] in/out = residual stream of the new token. */
int srgpt_llama_decode_step_bf16(void* h, const srgpt_llama_layer_weights* layers, int n_layers, void* q_buf, void* attn_buf,
                                 void* act_buf, int H, int n_heads, int n_kv_heads, int head_dim, int I, float eps,
                                 const void* cos_tab, const void* sin_tab, int* pos, const int* page_table, int page_size,
                                 const void* final_norm, const void* lm_head, int V, const void* embed_table, void* lm_workspace,
                                 float* logits_out, long long* out_ids, int* step, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* SRGPT_B200_H_ */
