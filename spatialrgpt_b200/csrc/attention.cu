// Attention kernels for the generate() path.
//   * attn_prefill_kernel : flash-style (online softmax, no SxS matrix in HBM) forward attention for
//     SigLIP (non-causal, head_dim 72) and Llama prefill (causal, GQA, head_dim 128).  Round-1
//     implementation: warp-level mma.sync m16n8k16 tiles with a cp.async double-buffered K/V ring.
//     (The tcgen05/TMEM version of this kernel is the next step; attention is ~13 % of the ViT FLOPs
//     and <1 % of the Llama prefill FLOPs at S~260, the GEMMs are on tcgen05 already.)
//   * rope_kv_append_kernel : RoPE on q,k + paged KV-cache append for the prompt tokens.
//   * attn_decode_kernel    : one-token attention over the paged KV cache.
//   * attn_prefill_paged_kernel : new prompt rows over the paged KV cache (chunked prefill / continuing a cached
//     sequence); mma.sync, chosen over tcgen05 for its latency / bytes-bound shapes (see the comment above the kernel).
// Reference: modeling_llama.py:405-566 (LlamaFlashAttention2), :160-191 (RoPE); HF SiglipAttention.
#include <algorithm>

#include "common.cuh"
#include "srgpt_b200.h"

namespace srgpt {
namespace attn {

constexpr int BM = 64, BN = 64, NTHREADS = 128;

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gsrc) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_u32(smem_dst)), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

__device__ __forceinline__ void ldmatrix_x4(uint32_t* r, const void* p) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3])
               : "r"(smem_u32(p)));
}
__device__ __forceinline__ void ldmatrix_x4_trans(uint32_t* r, const void* p) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3])
               : "r"(smem_u32(p)));
}
__device__ __forceinline__ void mma_bf16_16816(float* d, const uint32_t* a, uint32_t b0, uint32_t b1) {
  asm volatile(
      "mma.sync.aligned.m16n8k16.row.col.f32." SRGPT_ELEM_PTX "." SRGPT_ELEM_PTX ".f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
      : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}

template <int HD, int HDP>
struct Smem {
  static constexpr int LD = HDP + 8;  // +16 bytes per row: conflict-free ldmatrix
  bf16 q[BM][LD];
  bf16 k[2][BN][LD];
  bf16 v[2][BN][LD];
};

// cooperative load of a [64 x HD] tile (rows row0.. of one sequence) into smem; rows >= seqlen -> 0
template <int HD, int LD>
__device__ __forceinline__ void load_tile(bf16 (*dst)[LD], const bf16* __restrict__ src, int ld, int row0, int seqlen) {
  constexpr int CH = HD / 8;
  for (int i = threadIdx.x; i < 64 * CH; i += NTHREADS) {
    const int r = i / CH, c = i % CH;
    if (row0 + r < seqlen)
      cp_async16(&dst[r][c * 8], src + (size_t)(row0 + r) * ld + c * 8);
    else
      *reinterpret_cast<uint4*>(&dst[r][c * 8]) = make_uint4(0, 0, 0, 0);
  }
}

template <int HD, int HDP, bool CAUSAL>
__global__ void __launch_bounds__(NTHREADS)
attn_prefill_kernel(const bf16* __restrict__ q, const bf16* __restrict__ k, const bf16* __restrict__ v, bf16* __restrict__ out,
                    int q_ld, int kv_ld, int o_ld, int seqlen_fixed, const int* __restrict__ cu_seqlens, int group, float scale_log2) {
  using S = Smem<HD, HDP>;
  constexpr int LD = S::LD;
  extern __shared__ __align__(16) uint8_t smem_raw[];
  S& sm = *reinterpret_cast<S*>(smem_raw);

  const int qt = blockIdx.x, head = blockIdx.y, b = blockIdx.z;
  const int kvh = head / group;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int q0 = qt * BM;
  // sequences are either equal-length (row base b * seqlen) or packed back to back with cu_seqlens[b] as row base
  int row_base = b * seqlen_fixed, seqlen = seqlen_fixed;
  if (cu_seqlens != nullptr) {
    row_base = cu_seqlens[b];
    seqlen = cu_seqlens[b + 1] - row_base;
    if (q0 >= seqlen) return;  // grid.x covers the longest sequence
  }
  const bf16* qb = q + (size_t)row_base * q_ld + head * HD;
  const bf16* kb = k + (size_t)row_base * kv_ld + kvh * HD;
  const bf16* vb = v + (size_t)row_base * kv_ld + kvh * HD;

  // zero the padding columns [HD, LD) of every buffer once (never overwritten by the tile loads)
  if (HDP + 8 > HD) {
    constexpr int PADC = LD - HD;  // multiple of 8
    for (int i = threadIdx.x; i < 5 * 64 * (PADC / 8); i += NTHREADS) {
      const int buf = i / (64 * (PADC / 8)), rem = i % (64 * (PADC / 8));
      const int r = rem / (PADC / 8), c = rem % (PADC / 8);
      bf16* base = buf == 0 ? &sm.q[0][0] : (buf <= 2 ? &sm.k[buf - 1][0][0] : &sm.v[buf - 3][0][0]);
      *reinterpret_cast<uint4*>(base + r * LD + HD + c * 8) = make_uint4(0, 0, 0, 0);
    }
  }

  int ntiles = (seqlen + BN - 1) / BN;
  if (CAUSAL) ntiles = min(ntiles, qt + 1);

  load_tile<HD, LD>(sm.q, qb, q_ld, q0, seqlen);
  load_tile<HD, LD>(sm.k[0], kb, kv_ld, 0, seqlen);
  load_tile<HD, LD>(sm.v[0], vb, kv_ld, 0, seqlen);
  cp_async_commit();

  float o[HDP / 8][4];
#pragma unroll
  for (int i = 0; i < HDP / 8; ++i) o[i][0] = o[i][1] = o[i][2] = o[i][3] = 0.f;
  float m_run[2] = {-INFINITY, -INFINITY}, l_run[2] = {0.f, 0.f};
  uint32_t qf[HDP / 16][4];

  const int lr = lane & 7, lmat = lane >> 3;
  const int g = lane >> 2, t4 = lane & 3;

  for (int j = 0; j < ntiles; ++j) {
    const int cur = j & 1;
    if (j + 1 < ntiles) {
      load_tile<HD, LD>(sm.k[cur ^ 1], kb, kv_ld, (j + 1) * BN, seqlen);
      load_tile<HD, LD>(sm.v[cur ^ 1], vb, kv_ld, (j + 1) * BN, seqlen);
      cp_async_commit();
      cp_async_wait<1>();
    } else {
      cp_async_wait<0>();
    }
    __syncthreads();
    if (j == 0) {
#pragma unroll
      for (int kk = 0; kk < HDP / 16; ++kk)
        ldmatrix_x4(qf[kk], &sm.q[warp * 16 + lr + (lmat & 1) * 8][kk * 16 + (lmat >> 1) * 8]);
    }
    // ---- S = Q K^T (16 x 64 per warp)
    float s[BN / 8][4];
#pragma unroll
    for (int i = 0; i < BN / 8; ++i) s[i][0] = s[i][1] = s[i][2] = s[i][3] = 0.f;
#pragma unroll
    for (int np = 0; np < BN / 16; ++np) {
#pragma unroll
      for (int kk = 0; kk < HDP / 16; ++kk) {
        uint32_t bfr[4];
        ldmatrix_x4(bfr, &sm.k[cur][np * 16 + lr + (lmat >> 1) * 8][kk * 16 + (lmat & 1) * 8]);
        mma_bf16_16816(s[2 * np], qf[kk], bfr[0], bfr[1]);
        mma_bf16_16816(s[2 * np + 1], qf[kk], bfr[2], bfr[3]);
      }
    }
    // ---- scale, mask, online softmax
    const int qi0 = q0 + warp * 16 + g;  // rows qi0 and qi0 + 8
    float mx[2] = {-INFINITY, -INFINITY};
#pragma unroll
    for (int nb = 0; nb < BN / 8; ++nb) {
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const int kv = j * BN + nb * 8 + 2 * t4 + (e & 1);
        const int qi = qi0 + (e >> 1) * 8;
        float val = s[nb][e] * scale_log2;
        if (kv >= seqlen || (CAUSAL && kv > qi)) val = -INFINITY;
        s[nb][e] = val;
        mx[e >> 1] = fmaxf(mx[e >> 1], val);
      }
    }
    float alpha[2], m_new[2];
#pragma unroll
    for (int r = 0; r < 2; ++r) {
      mx[r] = fmaxf(mx[r], __shfl_xor_sync(0xffffffffu, mx[r], 1));
      mx[r] = fmaxf(mx[r], __shfl_xor_sync(0xffffffffu, mx[r], 2));
      m_new[r] = fmaxf(m_run[r], mx[r]);
      const float m_use = (m_new[r] == -INFINITY) ? 0.f : m_new[r];
      alpha[r] = exp2f(m_run[r] - m_use);  // m_run = -inf -> 0
      m_run[r] = m_new[r];
      m_new[r] = m_use;
    }
    float rs[2] = {0.f, 0.f};
#pragma unroll
    for (int nb = 0; nb < BN / 8; ++nb) {
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const float p = exp2f(s[nb][e] - m_new[e >> 1]);
        s[nb][e] = p;
        rs[e >> 1] += p;
      }
    }
#pragma unroll
    for (int r = 0; r < 2; ++r) l_run[r] = l_run[r] * alpha[r] + rs[r];
#pragma unroll
    for (int i = 0; i < HDP / 8; ++i) {
      o[i][0] *= alpha[0]; o[i][1] *= alpha[0];
      o[i][2] *= alpha[1]; o[i][3] *= alpha[1];
    }
    // ---- O += P V
#pragma unroll
    for (int kk = 0; kk < BN / 16; ++kk) {
      uint32_t a[4];
      a[0] = pack_bf16x2(s[2 * kk][0], s[2 * kk][1]);
      a[1] = pack_bf16x2(s[2 * kk][2], s[2 * kk][3]);
      a[2] = pack_bf16x2(s[2 * kk + 1][0], s[2 * kk + 1][1]);
      a[3] = pack_bf16x2(s[2 * kk + 1][2], s[2 * kk + 1][3]);
#pragma unroll
      for (int dp = 0; dp < HDP / 16; ++dp) {
        uint32_t bfr[4];
        ldmatrix_x4_trans(bfr, &sm.v[cur][kk * 16 + lr + (lmat & 1) * 8][dp * 16 + (lmat >> 1) * 8]);
        mma_bf16_16816(o[2 * dp], a, bfr[0], bfr[1]);
        mma_bf16_16816(o[2 * dp + 1], a, bfr[2], bfr[3]);
      }
    }
    __syncthreads();  // all warps done with buffer `cur` before it is refilled
  }

  // ---- finalize: O / l
#pragma unroll
  for (int r = 0; r < 2; ++r) {
    l_run[r] += __shfl_xor_sync(0xffffffffu, l_run[r], 1);
    l_run[r] += __shfl_xor_sync(0xffffffffu, l_run[r], 2);
  }
  const float inv0 = l_run[0] > 0.f ? 1.f / l_run[0] : 0.f;
  const float inv1 = l_run[1] > 0.f ? 1.f / l_run[1] : 0.f;
  bf16* ob = out + (size_t)row_base * o_ld + head * HD;
  const int r0 = q0 + warp * 16 + g, r1 = r0 + 8;
#pragma unroll
  for (int db = 0; db < HDP / 8; ++db) {
    const int d = db * 8 + 2 * t4;
    if (d < HD) {
      if (r0 < seqlen) *reinterpret_cast<uint32_t*>(ob + (size_t)r0 * o_ld + d) = pack_bf16x2(o[db][0] * inv0, o[db][1] * inv0);
      if (r1 < seqlen) *reinterpret_cast<uint32_t*>(ob + (size_t)r1 * o_ld + d) = pack_bf16x2(o[db][2] * inv1, o[db][3] * inv1);
    }
  }
}

// ---------------------------------------------------------------------------------------------
// RoPE (bf16 rounding points of modeling_llama.py:186-191) + paged KV append, prompt tokens
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void rope_pair(float x1, float x2, float c, float s, float& o1, float& o2) {
  // q_embed = q*cos + rotate_half(q)*sin, every product and the sum rounded to bf16
  o1 = bf16_round(bf16_round(x1 * c) + bf16_round(-x2 * s));
  o2 = bf16_round(bf16_round(x2 * c) + bf16_round(x1 * s));
}

__global__ void __launch_bounds__(128)
rope_kv_append_kernel(bf16* __restrict__ qkv, int n_heads, int n_kv_heads, int hd, const bf16* __restrict__ cos_tab,
                      const bf16* __restrict__ sin_tab, const int* __restrict__ start_pos, bf16* __restrict__ kv_pages,
                      const int* __restrict__ page_table, int page_size, const int* __restrict__ cu_seqlens, int n_seqs,
                      int pt_stride) {
  const int row = blockIdx.x;
  int seq = 0, local = row;
  if (cu_seqlens != nullptr) {  // packed sequences: largest s with cu_seqlens[s] <= row
    int lo = 0, hi = n_seqs - 1;
    while (lo < hi) {
      const int mid = (lo + hi + 1) >> 1;
      if (cu_seqlens[mid] <= row) lo = mid; else hi = mid - 1;
    }
    seq = lo;
    local = row - cu_seqlens[seq];
    page_table += (size_t)seq * pt_stride;
  }
  const int pos = start_pos[seq] + local;
  const int half = hd >> 1;
  const int ld = (n_heads + 2 * n_kv_heads) * hd;
  bf16* r = qkv + (size_t)row * ld;
  const bf16* ct = cos_tab + (size_t)pos * half;
  const bf16* st = sin_tab + (size_t)pos * half;
  const int page = page_table[pos / page_size], slot = pos % page_size;
  bf16* kdst = kv_pages + (((size_t)page * 2 + 0) * page_size + slot) * n_kv_heads * hd;
  bf16* vdst = kv_pages + (((size_t)page * 2 + 1) * page_size + slot) * n_kv_heads * hd;
  // 16-byte units: 8 channels of the first half of a head together with the matching 8 of the second half
  const int upc = half >> 3;  // units per head
  const int nunits = (n_heads + n_kv_heads) * upc;
  for (int i = threadIdx.x; i < nunits; i += blockDim.x) {
    const int h = i / upc, d = (i % upc) << 3;
    bf16* p = r + h * hd;
    float x1[8], x2[8], c[8], sn[8], o1[8], o2[8];
    unpack8(*reinterpret_cast<const uint4*>(p + d), x1);
    unpack8(*reinterpret_cast<const uint4*>(p + d + half), x2);
    unpack8(*reinterpret_cast<const uint4*>(ct + d), c);
    unpack8(*reinterpret_cast<const uint4*>(st + d), sn);
#pragma unroll
    for (int t = 0; t < 8; ++t) rope_pair(x1[t], x2[t], c[t], sn[t], o1[t], o2[t]);
    const uint4 b1 = pack8(o1), b2 = pack8(o2);
    *reinterpret_cast<uint4*>(p + d) = b1;
    *reinterpret_cast<uint4*>(p + d + half) = b2;
    if (h >= n_heads) {
      const int kh = h - n_heads;
      *reinterpret_cast<uint4*>(kdst + kh * hd + d) = b1;
      *reinterpret_cast<uint4*>(kdst + kh * hd + d + half) = b2;
    }
  }
  const bf16* vsrc = r + (n_heads + n_kv_heads) * hd;
  for (int i = threadIdx.x; i < (n_kv_heads * hd) >> 3; i += blockDim.x)
    reinterpret_cast<uint4*>(vdst)[i] = reinterpret_cast<const uint4*>(vsrc)[i];
}

// ---------------------------------------------------------------------------------------------
// decode attention: one CTA per query head, 32 half-warps; half-warp hw owns kv positions
// j = hw, hw+32, ...; every lane holds 8 of the 128 head dims (one 16-byte load per K/V row).
//
// The kernel is a pure latency chain (a few hundred KB per head), and the in-graph timeline
// (profiles/r01_decode_trace_gemv_v3.txt) showed 7 us of exposed time per layer.  K/V rows of PAST positions
// are immutable, so the first DEC_PRE*32 = 256 of them are requested BEFORE griddepcontrol.wait, i.e. while the
// QKV kernel of this layer is still streaming its weights; only q, the true position and the newest row(s)
// are read after the dependency resolves.  `*kv_len_minus1` read before the wait may be one step stale, which
// is a valid lower bound (positions only grow and rows below it are final).
// Two further ideas were built and measured on the in-graph timeline, then dropped (profiles/
// r01_decode_trace_attn_smemwindow.txt): a 128 KB shared-memory prefetch window for rows [256, 512) (the kernel no longer
// co-resides with the QKV GEMV CTAs, starts late: 7.8 us exposed) and speculative loads of the newest row(s) right after
// the wait (6.3 us).  This version measures 4.1-5.1 us.
// ---------------------------------------------------------------------------------------------
constexpr int DEC_THREADS = 512;
constexpr int DEC_HW = DEC_THREADS / 16;
constexpr int DEC_PRE = 8;
constexpr int DEC_UNROLL = 4;

__device__ __forceinline__ void dec_load_kv(const bf16* __restrict__ kv_pages, const int* __restrict__ page_table, int page_size,
                                            size_t row_stride, int kvh, int hl, int j, uint4& ku, uint4& vu) {
  const int pg = j / page_size;
  const int page = __ldg(page_table + pg);
  const int slot = j - pg * page_size;
  const bf16* kp = kv_pages + (((size_t)page * 2 + 0) * page_size + slot) * row_stride + kvh * 128 + hl * 8;
  ku = *reinterpret_cast<const uint4*>(kp);
  vu = *reinterpret_cast<const uint4*>(kp + (size_t)page_size * row_stride);
}

__global__ void __launch_bounds__(DEC_THREADS)
attn_decode_kernel(const bf16* __restrict__ q, bf16* __restrict__ out, const bf16* __restrict__ kv_pages,
                   const int* __restrict__ page_table, int page_size, const int* __restrict__ kv_len_minus1, int n_kv_heads,
                   int group, float scale_log2, unsigned long long* trace, int prefetch, int kv_head_off, int q_ld, int o_ld, int pt_stride) {
  constexpr int HD = 128;
  // batched decode (gridDim.y sequences, one new token each): row b of q / out, page table b, position b
  q += (size_t)blockIdx.y * q_ld;
  out += (size_t)blockIdx.y * o_ld;
  page_table += (size_t)blockIdx.y * pt_stride;
  kv_len_minus1 += blockIdx.y;
  __shared__ float s_m[DEC_HW], s_l[DEC_HW];
  __shared__ float s_acc[DEC_HW][HD];
  // tensor parallelism: q / out hold this rank's heads only, the cache keeps the full layout (n_kv_heads = heads per cache row)
  const int head = blockIdx.x, kvh = head / group + kv_head_off;
  const int hw = threadIdx.x >> 4, hl = threadIdx.x & 15;
  const size_t row_stride = (size_t)n_kv_heads * HD;
  trace_mark(trace, 0);

  // ---- before the dependency wait: immutable rows only
  const int pos_early = prefetch ? *reinterpret_cast<const volatile int*>(kv_len_minus1) : 0;  // rows [0, pos_early) are final
  uint4 kpre[DEC_PRE], vpre[DEC_PRE];
#pragma unroll
  for (int u = 0; u < DEC_PRE; ++u) {
    const int j = u * DEC_HW + hw;
    kpre[u] = make_uint4(0, 0, 0, 0);
    vpre[u] = make_uint4(0, 0, 0, 0);
    if (j < pos_early) dec_load_kv(kv_pages, page_table, page_size, row_stride, kvh, hl, j, kpre[u], vpre[u]);
  }
  // immutable rows beyond the register window (prompts longer than DEC_PRE * 32 = 256 tokens): requested into L2 now, so the
  // loop after the wait pays an L2 hit instead of an HBM round trip (one 128-byte line per 8 lanes of a half-warp)
  if (prefetch && (hl & 7) == 0) {
    for (int j = DEC_PRE * DEC_HW + hw; j < pos_early; j += DEC_HW) {
      const int pg = j / page_size;
      const int page = __ldg(page_table + pg);
      const bf16* kp = kv_pages + (((size_t)page * 2 + 0) * page_size + (j - pg * page_size)) * row_stride + kvh * 128 + hl * 8;
      asm volatile("prefetch.global.L2 [%0];" ::"l"(kp));
      asm volatile("prefetch.global.L2 [%0];" ::"l"(kp + (size_t)page_size * row_stride));
    }
  }
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  asm volatile("griddepcontrol.wait;" ::: "memory");
  trace_mark(trace, 1);

  const int kv_len = *reinterpret_cast<const volatile int*>(kv_len_minus1) + 1;
  float qf[8];
  unpack8(*reinterpret_cast<const uint4*>(q + head * HD + hl * 8), qf);
  float m = -INFINITY, l = 0.f, acc[8] = {0, 0, 0, 0, 0, 0, 0, 0};

  auto consume = [&](const uint4* ku, const uint4* vu, const bool* valid, int n) {
    float d[DEC_PRE];
#pragma unroll
    for (int u = 0; u < DEC_PRE; ++u) {
      if (u < n) {
        float kf[8];
        unpack8(ku[u], kf);
        d[u] = 0.f;
#pragma unroll
        for (int t = 0; t < 8; ++t) d[u] = fmaf(qf[t], kf[t], d[u]);
      }
    }
#pragma unroll
    for (int o = 8; o > 0; o >>= 1) {
#pragma unroll
      for (int u = 0; u < DEC_PRE; ++u)
        if (u < n) d[u] += __shfl_xor_sync(0xffffffffu, d[u], o);  // stays inside the half-warp; n is warp-uniform
    }
#pragma unroll
    for (int u = 0; u < DEC_PRE; ++u) {
      if (u < n && valid[u]) {
        float vf[8];
        unpack8(vu[u], vf);
        const float dd = d[u] * scale_log2;
        const float m_new = fmaxf(m, dd);
        const float a = exp2f(m - m_new), p = exp2f(dd - m_new);
        l = l * a + p;
#pragma unroll
        for (int t = 0; t < 8; ++t) acc[t] = acc[t] * a + p * vf[t];
        m = m_new;
      }
    }
  };

  {  // prefetched window
    bool valid[DEC_PRE];
#pragma unroll
    for (int u = 0; u < DEC_PRE; ++u) valid[u] = (u * DEC_HW + hw) < pos_early;
    consume(kpre, vpre, valid, DEC_PRE);
  }
  // ---- everything the prefetch did not cover: the newest row(s) and positions >= DEC_PRE*32
  const int done_upto = pos_early < DEC_PRE * DEC_HW ? pos_early : DEC_PRE * DEC_HW;  // positions [0, done_upto) are consumed
  for (int j0 = (done_upto / DEC_HW) * DEC_HW; j0 < kv_len; j0 += DEC_HW * DEC_UNROLL) {  // warp-uniform trip count
    uint4 ku[DEC_UNROLL], vu[DEC_UNROLL];
    bool valid[DEC_UNROLL];
#pragma unroll
    for (int u = 0; u < DEC_UNROLL; ++u) {
      const int j = j0 + u * DEC_HW + hw;
      valid[u] = j < kv_len && j >= done_upto;
      ku[u] = make_uint4(0, 0, 0, 0);
      vu[u] = make_uint4(0, 0, 0, 0);
      if (valid[u]) dec_load_kv(kv_pages, page_table, page_size, row_stride, kvh, hl, j, ku[u], vu[u]);
    }
    consume(ku, vu, valid, DEC_UNROLL);
  }

  if (hl == 0) { s_m[hw] = m; s_l[hw] = l; }
#pragma unroll
  for (int t = 0; t < 8; ++t) s_acc[hw][hl * 8 + t] = acc[t];
  __syncthreads();
  if (threadIdx.x < HD) {
    float mt = -INFINITY;
#pragma unroll
    for (int i = 0; i < DEC_HW; ++i) mt = fmaxf(mt, s_m[i]);
    float lt = 0.f, at = 0.f;
#pragma unroll
    for (int i = 0; i < DEC_HW; ++i) {
      const float w = (s_m[i] == -INFINITY) ? 0.f : exp2f(s_m[i] - mt);
      lt += s_l[i] * w;
      at += s_acc[i][threadIdx.x] * w;
    }
    out[head * HD + threadIdx.x] = f2e(at / lt);
  }
  trace_mark(trace, 2);
}

// ---------------------------------------------------------------------------------------------
// Batched decode attention, one CTA per (kv head, sequence): the GROUP query heads that share a kv head (GQA) are served from ONE pass
// over that head's K / V rows.  With a CTA per (q head, sequence) a 32-sequence step of Llama-3-8B launched 1024 CTAs that each
// re-read their kv head's rows (48 us per layer in profiles/r02_launches_batched_decode.txt, against 6 us of bytes); here it is 256
// CTAs and a quarter of the reads.  Same arithmetic per head as attn_decode_kernel (half-warp per kv row, base-2 online softmax).
// ---------------------------------------------------------------------------------------------
template <int GROUP>
__global__ void __launch_bounds__(DEC_THREADS)
attn_decode_gqa_kernel(const bf16* __restrict__ q, int q_ld, bf16* __restrict__ out, int o_ld, const bf16* __restrict__ kv_pages,
                       const int* __restrict__ page_tables, int pt_stride, int page_size, const int* __restrict__ kv_len_minus1, int n_kv_heads,
                       float scale_log2) {
  constexpr int HD = 128;
  __shared__ float s_m[DEC_HW], s_l[DEC_HW];
  __shared__ float s_acc[DEC_HW][HD];
  const int kvh = blockIdx.x, b = blockIdx.y;
  const int hw = threadIdx.x >> 4, hl = threadIdx.x & 15;
  const size_t row_stride = (size_t)n_kv_heads * HD;
  const int* page_table = page_tables + (size_t)b * pt_stride;
  const int kv_len = kv_len_minus1[b] + 1;
  float qf[GROUP][8];
#pragma unroll
  for (int g = 0; g < GROUP; ++g) unpack8(*reinterpret_cast<const uint4*>(q + (size_t)b * q_ld + (kvh * GROUP + g) * HD + hl * 8), qf[g]);
  float m[GROUP], l[GROUP], acc[GROUP][8];
#pragma unroll
  for (int g = 0; g < GROUP; ++g) {
    m[g] = -INFINITY;
    l[g] = 0.f;
#pragma unroll
    for (int t = 0; t < 8; ++t) acc[g][t] = 0.f;
  }
  for (int j0 = 0; j0 < kv_len; j0 += DEC_HW * DEC_UNROLL) {  // warp-uniform trip count
    uint4 ku[DEC_UNROLL], vu[DEC_UNROLL];
    bool valid[DEC_UNROLL];
#pragma unroll
    for (int u = 0; u < DEC_UNROLL; ++u) {
      const int j = j0 + u * DEC_HW + hw;
      valid[u] = j < kv_len;
      ku[u] = make_uint4(0, 0, 0, 0);
      vu[u] = make_uint4(0, 0, 0, 0);
      if (valid[u]) dec_load_kv(kv_pages, page_table, page_size, row_stride, kvh, hl, j, ku[u], vu[u]);
    }
#pragma unroll
    for (int u = 0; u < DEC_UNROLL; ++u) {
      float kf[8], vf[8], d[GROUP];
      unpack8(ku[u], kf);
      unpack8(vu[u], vf);
#pragma unroll
      for (int g = 0; g < GROUP; ++g) {
        d[g] = 0.f;
#pragma unroll
        for (int t = 0; t < 8; ++t) d[g] = fmaf(qf[g][t], kf[t], d[g]);
      }
#pragma unroll
      for (int o = 8; o > 0; o >>= 1) {
#pragma unroll
        for (int g = 0; g < GROUP; ++g) d[g] += __shfl_xor_sync(0xffffffffu, d[g], o);  // stays inside the half-warp
      }
      if (valid[u]) {
#pragma unroll
        for (int g = 0; g < GROUP; ++g) {
          const float dd = d[g] * scale_log2;
          const float m_new = fmaxf(m[g], dd);
          const float a = exp2f(m[g] - m_new), pp = exp2f(dd - m_new);
          l[g] = l[g] * a + pp;
#pragma unroll
          for (int t = 0; t < 8; ++t) acc[g][t] = acc[g][t] * a + pp * vf[t];
          m[g] = m_new;
        }
      }
    }
  }
  // cross-half-warp reduction, one head at a time through the same 16 KB of shared memory
#pragma unroll
  for (int g = 0; g < GROUP; ++g) {
    __syncthreads();
    if (hl == 0) { s_m[hw] = m[g]; s_l[hw] = l[g]; }
#pragma unroll
    for (int t = 0; t < 8; ++t) s_acc[hw][hl * 8 + t] = acc[g][t];
    __syncthreads();
    if (threadIdx.x < HD) {
      float mt = -INFINITY;
#pragma unroll
      for (int i = 0; i < DEC_HW; ++i) mt = fmaxf(mt, s_m[i]);
      float lt = 0.f, at = 0.f;
#pragma unroll
      for (int i = 0; i < DEC_HW; ++i) {
        const float w = (s_m[i] == -INFINITY) ? 0.f : exp2f(s_m[i] - mt);
        lt += s_l[i] * w;
        at += s_acc[i][threadIdx.x] * w;
      }
      out[(size_t)b * o_ld + (kvh * GROUP + g) * HD + threadIdx.x] = f2e(at / lt);
    }
  }
}

// ---------------------------------------------------------------------------------------------
// Prefill attention over the PAGED cache: new prompt rows of a sequence attend to every earlier position, whether it was
// written by this chunk or by an earlier prefill / decode (chunked prefill, continuing a cached conversation).  The reference
// concatenates the past K/V (modeling_llama.py:451-456) and calls flash_attn_func(causal=True) with q_len < kv_len, i.e. the
// causal mask aligned bottom-right (:564-566); prepare_inputs_for_generation drops the cached prefix (:1112-1149).
//
// Rows [cu_q[b], cu_q[b+1]) of q are sequence b's new rows at positions start_pos[b] + i; their K/V are already in the pages
// (srgpt_rope_kv_append_varlen_bf16).  Row at position p attends to positions 0..p, read through page_tables[b].
//
// Work split.  One CTA serves all G query heads of a kv head: the 64 rows of the MMA tile are G x (64 / G) (query row, head)
// pairs, packed row pr = (row q0 + pr / G, head kvh * G + pr % G), so every K/V tile is read once per group and q tile (GQA
// shares the pass like attn_decode_gqa_kernel).  When seqs x kv heads x q tiles is far below one wave (a 40-row follow-up turn
// of Llama-3-8B is 24 CTAs) the context is split over CTAs; each split writes fp32 (O, m, l) and attn_paged_combine_kernel
// merges them in split order (deterministic, no atomics, graph-safe).
// mma.sync m16n8k16 + cp.async page loads, same rounding as attn_prefill_kernel (fp32 scores and online softmax, P rounded to
// the element type before P.V, the output rounded once).  tcgen05 is not used: the follow-up shape is ~0.3 GFLOP and 2 MB of
// K/V per layer (latency / bytes bound, and page-granular gathers do not map onto one TMA box), and a 512-row chunk at the end of
// a 4k context (~32 GFLOP per layer) is a rare shape next to the GEMMs of the same chunk.
// ---------------------------------------------------------------------------------------------
constexpr int PG_PAGE = 16;
constexpr int PG_SPLIT_BELOW = 74;   // split the context when the grid has at most half a wave of CTAs...
constexpr int PG_SPLIT_TARGET = 148; // ...up to about one wave (the B200's SM count; fixed so the workspace size is host arithmetic)

using PagedSmem = Smem<128, 128>;

// K (which = 0) or V (which = 1) rows of positions [kv0, kv0 + 64) of kv head kvh; positions >= kv_len are zero-filled (no
// page-table read past the sequence's reserved pages)
__device__ __forceinline__ void load_kv_paged(bf16 (*dst)[PagedSmem::LD], const bf16* __restrict__ kv_pages, const int* __restrict__ pt,
                                              size_t row_stride, int kvh, int which, int kv0, int kv_len) {
  for (int i = threadIdx.x; i < BN * 16; i += NTHREADS) {
    const int r = i >> 4, c = i & 15;
    const int j = kv0 + r;
    if (j < kv_len) {
      const int page = __ldg(pt + j / PG_PAGE);
      cp_async16(&dst[r][c * 8], kv_pages + (((size_t)page * 2 + which) * PG_PAGE + (j % PG_PAGE)) * row_stride + kvh * 128 + c * 8);
    } else {
      *reinterpret_cast<uint4*>(&dst[r][c * 8]) = make_uint4(0, 0, 0, 0);
    }
  }
}

__global__ void __launch_bounds__(NTHREADS)
attn_prefill_paged_kernel(const bf16* __restrict__ q, int q_ld, bf16* __restrict__ out, int o_ld, const bf16* __restrict__ kv_pages,
                          const int* __restrict__ page_tables, int pt_stride, const int* __restrict__ cu_q, const int* __restrict__ start_pos,
                          int n_heads, int n_kv_heads, int group, int n_split, int tiles_per_split, float* __restrict__ ws_o,
                          float* __restrict__ ws_ml, int ws_rows, float scale_log2) {
  constexpr int HD = 128;
  using S = PagedSmem;
  extern __shared__ __align__(16) uint8_t smem_raw[];
  S& sm = *reinterpret_cast<S*>(smem_raw);

  const int qt = blockIdx.x, kvh = blockIdx.y, b = blockIdx.z / n_split, split = blockIdx.z % n_split;
  const int QR = BM / group;  // query rows per tile
  const int row_base = cu_q[b], q_len = cu_q[b + 1] - row_base;
  const int q0 = qt * QR;
  if (q0 >= q_len) return;  // grid.x covers the longest chunk
  const int sp = start_pos[b];
  const int kv_len = sp + min(q0 + QR, q_len);  // positions [0, kv_len) are visible to some row of this tile
  const int ntiles = (kv_len + BN - 1) / BN;
  const int t_begin = min(split * tiles_per_split, ntiles);
  const int t_end = split == n_split - 1 ? ntiles : min(ntiles, t_begin + tiles_per_split);
  const int* pt = page_tables + (size_t)b * pt_stride;
  const size_t row_stride = (size_t)n_kv_heads * HD;

  for (int i = threadIdx.x; i < BM * 16; i += NTHREADS) {
    const int pr = i >> 4, c = i & 15, qi = pr / group;
    if (pr < QR * group && q0 + qi < q_len)
      cp_async16(&sm.q[pr][c * 8], q + (size_t)(row_base + q0 + qi) * q_ld + (kvh * group + pr % group) * HD + c * 8);
    else
      *reinterpret_cast<uint4*>(&sm.q[pr][c * 8]) = make_uint4(0, 0, 0, 0);
  }
  if (t_begin < t_end) {
    load_kv_paged(sm.k[0], kv_pages, pt, row_stride, kvh, 0, t_begin * BN, kv_len);
    load_kv_paged(sm.v[0], kv_pages, pt, row_stride, kvh, 1, t_begin * BN, kv_len);
  }
  cp_async_commit();

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int lr = lane & 7, lmat = lane >> 3;
  const int g = lane >> 2, t4 = lane & 3;
  // this thread's two packed rows (pr, pr + 8): query position, or -1 for a padding row (everything masked)
  int prow[2], ppos[2];
#pragma unroll
  for (int r = 0; r < 2; ++r) {
    const int pr = warp * 16 + g + r * 8, qi = pr / group;
    const bool ok = pr < QR * group && q0 + qi < q_len;
    prow[r] = pr;
    ppos[r] = ok ? sp + q0 + qi : -1;
  }

  float o[HD / 8][4];
#pragma unroll
  for (int i = 0; i < HD / 8; ++i) o[i][0] = o[i][1] = o[i][2] = o[i][3] = 0.f;
  float m_run[2] = {-INFINITY, -INFINITY}, l_run[2] = {0.f, 0.f};
  uint32_t qf[HD / 16][4];

  if (t_begin == t_end) cp_async_wait<0>();
  for (int j = t_begin; j < t_end; ++j) {
    const int cur = (j - t_begin) & 1;
    if (j + 1 < t_end) {
      load_kv_paged(sm.k[cur ^ 1], kv_pages, pt, row_stride, kvh, 0, (j + 1) * BN, kv_len);
      load_kv_paged(sm.v[cur ^ 1], kv_pages, pt, row_stride, kvh, 1, (j + 1) * BN, kv_len);
      cp_async_commit();
      cp_async_wait<1>();
    } else {
      cp_async_wait<0>();
    }
    __syncthreads();
    if (j == t_begin) {
#pragma unroll
      for (int kk = 0; kk < HD / 16; ++kk)
        ldmatrix_x4(qf[kk], &sm.q[warp * 16 + lr + (lmat & 1) * 8][kk * 16 + (lmat >> 1) * 8]);
    }
    // ---- S = Q K^T (16 packed rows x 64 positions per warp)
    float s[BN / 8][4];
#pragma unroll
    for (int i = 0; i < BN / 8; ++i) s[i][0] = s[i][1] = s[i][2] = s[i][3] = 0.f;
#pragma unroll
    for (int np = 0; np < BN / 16; ++np) {
#pragma unroll
      for (int kk = 0; kk < HD / 16; ++kk) {
        uint32_t bfr[4];
        ldmatrix_x4(bfr, &sm.k[cur][np * 16 + lr + (lmat >> 1) * 8][kk * 16 + (lmat & 1) * 8]);
        mma_bf16_16816(s[2 * np], qf[kk], bfr[0], bfr[1]);
        mma_bf16_16816(s[2 * np + 1], qf[kk], bfr[2], bfr[3]);
      }
    }
    // ---- scale, causal mask (bottom-right aligned: position p sees 0..p), online softmax
    float mx[2] = {-INFINITY, -INFINITY};
#pragma unroll
    for (int nb = 0; nb < BN / 8; ++nb) {
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const int kv = j * BN + nb * 8 + 2 * t4 + (e & 1);
        float val = s[nb][e] * scale_log2;
        if (kv > ppos[e >> 1]) val = -INFINITY;
        s[nb][e] = val;
        mx[e >> 1] = fmaxf(mx[e >> 1], val);
      }
    }
    float alpha[2], m_new[2];
#pragma unroll
    for (int r = 0; r < 2; ++r) {
      mx[r] = fmaxf(mx[r], __shfl_xor_sync(0xffffffffu, mx[r], 1));
      mx[r] = fmaxf(mx[r], __shfl_xor_sync(0xffffffffu, mx[r], 2));
      m_new[r] = fmaxf(m_run[r], mx[r]);
      const float m_use = (m_new[r] == -INFINITY) ? 0.f : m_new[r];
      alpha[r] = exp2f(m_run[r] - m_use);
      m_run[r] = m_new[r];
      m_new[r] = m_use;
    }
    float rs[2] = {0.f, 0.f};
#pragma unroll
    for (int nb = 0; nb < BN / 8; ++nb) {
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const float p = exp2f(s[nb][e] - m_new[e >> 1]);
        s[nb][e] = p;
        rs[e >> 1] += p;
      }
    }
#pragma unroll
    for (int r = 0; r < 2; ++r) l_run[r] = l_run[r] * alpha[r] + rs[r];
#pragma unroll
    for (int i = 0; i < HD / 8; ++i) {
      o[i][0] *= alpha[0]; o[i][1] *= alpha[0];
      o[i][2] *= alpha[1]; o[i][3] *= alpha[1];
    }
    // ---- O += P V
#pragma unroll
    for (int kk = 0; kk < BN / 16; ++kk) {
      uint32_t a[4];
      a[0] = pack_bf16x2(s[2 * kk][0], s[2 * kk][1]);
      a[1] = pack_bf16x2(s[2 * kk][2], s[2 * kk][3]);
      a[2] = pack_bf16x2(s[2 * kk + 1][0], s[2 * kk + 1][1]);
      a[3] = pack_bf16x2(s[2 * kk + 1][2], s[2 * kk + 1][3]);
#pragma unroll
      for (int dp = 0; dp < HD / 16; ++dp) {
        uint32_t bfr[4];
        ldmatrix_x4_trans(bfr, &sm.v[cur][kk * 16 + lr + (lmat & 1) * 8][dp * 16 + (lmat >> 1) * 8]);
        mma_bf16_16816(o[2 * dp], a, bfr[0], bfr[1]);
        mma_bf16_16816(o[2 * dp + 1], a, bfr[2], bfr[3]);
      }
    }
    __syncthreads();  // all warps done with buffer `cur` before it is refilled
  }

#pragma unroll
  for (int r = 0; r < 2; ++r) {
    l_run[r] += __shfl_xor_sync(0xffffffffu, l_run[r], 1);
    l_run[r] += __shfl_xor_sync(0xffffffffu, l_run[r], 2);
  }
#pragma unroll
  for (int r = 0; r < 2; ++r) {
    if (ppos[r] < 0) continue;
    const int row = row_base + q0 + prow[r] / group, head = kvh * group + prow[r] % group;
    if (n_split == 1) {
      const float inv = l_run[r] > 0.f ? 1.f / l_run[r] : 0.f;
      bf16* ob = out + (size_t)row * o_ld + head * HD;
#pragma unroll
      for (int db = 0; db < HD / 8; ++db)
        *reinterpret_cast<uint32_t*>(ob + db * 8 + 2 * t4) = pack_bf16x2(o[db][2 * r] * inv, o[db][2 * r + 1] * inv);
    } else if (row < ws_rows) {
      const size_t slot = ((size_t)split * ws_rows + row) * n_heads + head;
      float* wo = ws_o + slot * HD;
#pragma unroll
      for (int db = 0; db < HD / 8; ++db) *reinterpret_cast<float2*>(wo + db * 8 + 2 * t4) = make_float2(o[db][2 * r], o[db][2 * r + 1]);
      if (t4 == 0) *reinterpret_cast<float2*>(ws_ml + slot * 2) = make_float2(m_run[r], l_run[r]);
    }
  }
}

// merges the n_split partial results of a row and head in split order: O = sum_s o_s 2^(m_s - M) / sum_s l_s 2^(m_s - M)
__global__ void __launch_bounds__(128)
attn_paged_combine_kernel(const float* __restrict__ ws_o, const float* __restrict__ ws_ml, bf16* __restrict__ out, int o_ld,
                          const int* __restrict__ cu_q, int n_seqs, int n_split, int ws_rows, int n_heads) {
  const int row = blockIdx.x, head = blockIdx.y, d = threadIdx.x;
  if (row >= cu_q[n_seqs]) return;
  float mt = -INFINITY;
  for (int s = 0; s < n_split; ++s) mt = fmaxf(mt, ws_ml[(((size_t)s * ws_rows + row) * n_heads + head) * 2]);
  float lt = 0.f, at = 0.f;
  for (int s = 0; s < n_split; ++s) {
    const size_t slot = ((size_t)s * ws_rows + row) * n_heads + head;
    const float m = ws_ml[slot * 2];
    const float w = m == -INFINITY ? 0.f : exp2f(m - mt);
    lt += ws_ml[slot * 2 + 1] * w;
    at += ws_o[slot * 128 + d] * w;
  }
  out[(size_t)row * o_ld + head * 128 + d] = f2e(lt > 0.f ? at / lt : 0.f);
}

// context split of the paged kernel; pure host arithmetic (the workspace size must not need a device)
static int paged_split(int n_seqs, int max_q_len, int max_ctx_len, int n_heads, int n_kv_heads, int* tiles_per_split) {
  const int group = n_heads / n_kv_heads;
  const int ctas = n_seqs * n_kv_heads * ceil_div(max_q_len, BM / group);
  const int kv_tiles = ceil_div(max_ctx_len, BN);
  int n_split = 1;
  if (ctas <= PG_SPLIT_BELOW) n_split = std::max(1, std::min(kv_tiles, ceil_div(PG_SPLIT_TARGET, ctas)));
  *tiles_per_split = ceil_div(kv_tiles, n_split);
  return ceil_div(kv_tiles, *tiles_per_split);  // no empty trailing split
}

template <int HD, int HDP, bool CAUSAL>
static int launch_prefill(const void* q, const void* k, const void* v, void* out, int q_ld, int kv_ld, int o_ld, int batch,
                          int seqlen, const int* cu_seqlens, int n_heads, int n_kv_heads, float scale, cudaStream_t st) {
  using S = Smem<HD, HDP>;
  static bool configured = false;
  if (!configured) {
    SRGPT_CHECK_CUDA(cudaFuncSetAttribute(attn_prefill_kernel<HD, HDP, CAUSAL>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(S)));
    configured = true;
  }
  dim3 grid(ceil_div(seqlen, BM), n_heads, batch);
  attn_prefill_kernel<HD, HDP, CAUSAL><<<grid, NTHREADS, sizeof(S), st>>>(
      reinterpret_cast<const bf16*>(q), reinterpret_cast<const bf16*>(k), reinterpret_cast<const bf16*>(v),
      reinterpret_cast<bf16*>(out), q_ld, kv_ld, o_ld, seqlen, cu_seqlens, n_heads / n_kv_heads, scale * 1.4426950408889634f);
  SRGPT_CHECK_LAUNCH();
  return SRGPT_OK;
}

}  // namespace attn
}  // namespace srgpt

using namespace srgpt;

static bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

namespace srgpt {
namespace attn_tc {  // attention_tc.cu: tcgen05 / TMEM / TMA kernel (head_dim 72 and 128)
int prefill(const void* q, const void* k, const void* v, void* out, int q_ld, int kv_ld, int o_ld, int batch, int seqlen, const int* cu, long long total_rows,
            int n_heads, int n_kv_heads, int head_dim, float scale, int causal, cudaStream_t st);
}
}  // namespace srgpt

static int attention_prefill_any(const void* q, const void* k, const void* v, void* out, int q_ld, int kv_ld, int o_ld, int batch, int seqlen,
                                 const int* cu, long long total_rows, int n_heads, int n_kv_heads, int head_dim, float scale, int causal, void* stream) {
  SRGPT_CHECK_ARG(q && k && v && out && batch > 0 && seqlen > 0 && n_heads > 0 && n_kv_heads > 0);
  SRGPT_CHECK_ARG((n_heads % n_kv_heads) == 0);
  SRGPT_CHECK_ARG((q_ld % 8) == 0 && (kv_ld % 8) == 0 && (o_ld % 2) == 0);
  SRGPT_CHECK_ARG(aligned16(q) && aligned16(k) && aligned16(v) && (reinterpret_cast<uintptr_t>(out) & 3) == 0);
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  // tensor-memory kernel first; the mma.sync kernel below covers the remaining head sizes (and SRGPT_ATTN_MMA_SYNC=1)
  static const bool force_mma_sync = env_flag("SRGPT_ATTN_MMA_SYNC");
  if (!force_mma_sync) {
    const int rc = attn_tc::prefill(q, k, v, out, q_ld, kv_ld, o_ld, batch, seqlen, cu, total_rows, n_heads, n_kv_heads, head_dim, scale, causal, st);
    if (rc != SRGPT_ERR_UNSUPPORTED) return rc;
  }
  if (head_dim == 72 && !causal)
    return attn::launch_prefill<72, 80, false>(q, k, v, out, q_ld, kv_ld, o_ld, batch, seqlen, cu, n_heads, n_kv_heads, scale, st);
  if (head_dim == 72 && causal)
    return attn::launch_prefill<72, 80, true>(q, k, v, out, q_ld, kv_ld, o_ld, batch, seqlen, cu, n_heads, n_kv_heads, scale, st);
  if (head_dim == 128 && causal)
    return attn::launch_prefill<128, 128, true>(q, k, v, out, q_ld, kv_ld, o_ld, batch, seqlen, cu, n_heads, n_kv_heads, scale, st);
  if (head_dim == 128 && !causal)
    return attn::launch_prefill<128, 128, false>(q, k, v, out, q_ld, kv_ld, o_ld, batch, seqlen, cu, n_heads, n_kv_heads, scale, st);
  if (head_dim == 64)
    return causal ? attn::launch_prefill<64, 64, true>(q, k, v, out, q_ld, kv_ld, o_ld, batch, seqlen, cu, n_heads, n_kv_heads, scale, st)
                  : attn::launch_prefill<64, 64, false>(q, k, v, out, q_ld, kv_ld, o_ld, batch, seqlen, cu, n_heads, n_kv_heads, scale, st);
  set_last_error("srgpt_attention_prefill: unsupported head_dim %d (supported: 64, 72, 128)", head_dim);
  return SRGPT_ERR_UNSUPPORTED;
}

extern "C" __attribute__((visibility("default"))) int srgpt_attention_prefill_bf16(const void* q, const void* k, const void* v, void* out, int q_ld, int kv_ld, int o_ld,
                                            int batch, int seqlen, int n_heads, int n_kv_heads, int head_dim, float scale,
                                            int causal, void* stream) {
  return attention_prefill_any(q, k, v, out, q_ld, kv_ld, o_ld, batch, seqlen, nullptr, (long long)batch * seqlen, n_heads, n_kv_heads, head_dim, scale, causal,
                               stream);
}

extern "C" __attribute__((visibility("default"))) int srgpt_attention_prefill_varlen_bf16(const void* q, const void* k, const void* v, void* out, int q_ld, int kv_ld,
                                                   int o_ld, int n_seqs, const int* cu_seqlens, int max_seqlen, int total_rows, int n_heads,
                                                   int n_kv_heads, int head_dim, float scale, int causal, void* stream) {
  SRGPT_CHECK_ARG(cu_seqlens != nullptr && total_rows >= max_seqlen);
  return attention_prefill_any(q, k, v, out, q_ld, kv_ld, o_ld, n_seqs, max_seqlen, cu_seqlens, total_rows, n_heads, n_kv_heads, head_dim, scale, causal, stream);
}

static int rope_kv_append_any(void* qkv, int rows, int n_heads, int n_kv_heads, int head_dim, const void* cos_tab, const void* sin_tab,
                              const int* start_pos, void* kv_pages, const int* page_table, int page_size, const int* cu, int n_seqs, int pt_stride,
                              void* stream) {
  SRGPT_CHECK_ARG(qkv && cos_tab && sin_tab && start_pos && kv_pages && page_table);
  SRGPT_CHECK_ARG(rows > 0 && n_heads > 0 && n_kv_heads > 0 && head_dim > 0 && (head_dim % 16) == 0 && page_size > 0);
  SRGPT_CHECK_ARG(aligned16(qkv) && aligned16(kv_pages));
  attn::rope_kv_append_kernel<<<rows, 128, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
      reinterpret_cast<bf16*>(qkv), n_heads, n_kv_heads, head_dim, reinterpret_cast<const bf16*>(cos_tab),
      reinterpret_cast<const bf16*>(sin_tab), start_pos, reinterpret_cast<bf16*>(kv_pages), page_table, page_size, cu, n_seqs, pt_stride);
  SRGPT_CHECK_LAUNCH();
  return SRGPT_OK;
}

extern "C" __attribute__((visibility("default"))) int srgpt_rope_kv_append_bf16(void* qkv, int rows, int n_heads, int n_kv_heads, int head_dim, const void* cos_tab,
                                         const void* sin_tab, const int* start_pos, void* kv_pages, const int* page_table,
                                         int page_size, void* stream) {
  return rope_kv_append_any(qkv, rows, n_heads, n_kv_heads, head_dim, cos_tab, sin_tab, start_pos, kv_pages, page_table, page_size, nullptr, 1, 0, stream);
}

extern "C" __attribute__((visibility("default"))) int srgpt_rope_kv_append_varlen_bf16(void* qkv, int rows, int n_heads, int n_kv_heads, int head_dim, const void* cos_tab,
                                                const void* sin_tab, const int* start_pos, void* kv_pages, const int* page_tables,
                                                int page_table_stride, int page_size, int n_seqs, const int* cu_seqlens, void* stream) {
  SRGPT_CHECK_ARG(cu_seqlens != nullptr && n_seqs > 0 && page_table_stride > 0);
  return rope_kv_append_any(qkv, rows, n_heads, n_kv_heads, head_dim, cos_tab, sin_tab, start_pos, kv_pages, page_tables, page_size, cu_seqlens, n_seqs,
                            page_table_stride, stream);
}

extern "C" __attribute__((visibility("default"))) int srgpt_attention_decode_bf16(const void* q, void* out, const void* kv_pages, const int* page_table, int page_size,
                                           const int* kv_len_minus1, int n_heads, int n_kv_heads, int head_dim, float scale,
                                           void* stream) {
  SRGPT_CHECK_ARG(q && out && kv_pages && page_table && kv_len_minus1);
  SRGPT_CHECK_ARG(n_heads > 0 && n_kv_heads > 0 && (n_heads % n_kv_heads) == 0 && page_size > 0);
  SRGPT_CHECK_ARG(aligned16(q) && aligned16(kv_pages));
  if (head_dim != 128) {
    set_last_error("srgpt_attention_decode_bf16: head_dim %d unsupported (128 only)", head_dim);
    return SRGPT_ERR_UNSUPPORTED;
  }
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(n_heads);
  cfg.blockDim = dim3(attn::DEC_THREADS);
  cfg.stream = reinterpret_cast<cudaStream_t>(stream);
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = pdl_enabled() ? 1 : 0;
  static const bool no_prefetch = env_flag("SRGPT_ATTN_NO_PREFETCH");
  SRGPT_CHECK_CUDA(cudaLaunchKernelEx(&cfg, attn::attn_decode_kernel, reinterpret_cast<const bf16*>(q), reinterpret_cast<bf16*>(out),
                                      reinterpret_cast<const bf16*>(kv_pages), page_table, page_size, kv_len_minus1, n_kv_heads,
                                      n_heads / n_kv_heads, scale * 1.4426950408889634f, trace_next_slot(), no_prefetch ? 0 : 1, 0, 0, 0, 0));
  return SRGPT_OK;
}

static bool paged_args_ok(int n_seqs, int max_q_len, int max_ctx_len, int n_heads, int n_kv_heads) {
  return n_seqs > 0 && n_seqs <= 65535 / attn::PG_SPLIT_TARGET && max_q_len > 0 && max_ctx_len >= max_q_len && n_heads > 0 && n_kv_heads > 0 &&
         (n_heads % n_kv_heads) == 0 && n_heads / n_kv_heads <= 8;
}

extern "C" __attribute__((visibility("default"))) long long srgpt_attention_prefill_paged_workspace(int n_seqs, int max_q_len, int max_ctx_len,
                                                                                                    int n_heads, int n_kv_heads) {
  if (!paged_args_ok(n_seqs, max_q_len, max_ctx_len, n_heads, n_kv_heads)) return -1;
  int tps = 0;
  const int n_split = attn::paged_split(n_seqs, max_q_len, max_ctx_len, n_heads, n_kv_heads, &tps);
  if (n_split == 1) return 0;
  return (long long)n_split * n_seqs * max_q_len * n_heads * (128 + 2) * (long long)sizeof(float);
}

extern "C" __attribute__((visibility("default"))) int srgpt_attention_prefill_paged_bf16(const void* q, int q_ld, void* out, int o_ld, const void* kv_pages,
                                                                                         const int* page_tables, int page_table_stride, int page_size, int n_seqs,
                                                                                         const int* cu_q, const int* start_pos, int max_q_len, int max_ctx_len,
                                                                                         int n_heads, int n_kv_heads, int head_dim, float scale, void* workspace,
                                                                                         long long workspace_bytes, void* stream) {
  SRGPT_CHECK_ARG(q && out && kv_pages && page_tables && cu_q && start_pos);
  SRGPT_CHECK_ARG(paged_args_ok(n_seqs, max_q_len, max_ctx_len, n_heads, n_kv_heads) && page_table_stride > 0);
  SRGPT_CHECK_ARG(aligned16(q) && aligned16(kv_pages) && (q_ld % 8) == 0 && q_ld >= n_heads * head_dim && o_ld >= n_heads * head_dim);
  SRGPT_CHECK_ARG((o_ld % 2) == 0 && (reinterpret_cast<uintptr_t>(out) & 3) == 0);
  if (head_dim != 128 || page_size != attn::PG_PAGE) {
    set_last_error("srgpt_attention_prefill_paged_bf16: head_dim %d / page_size %d unsupported (128 / 16 only)", head_dim, page_size);
    return SRGPT_ERR_UNSUPPORTED;
  }
  int tps = 0;
  int n_split = attn::paged_split(n_seqs, max_q_len, max_ctx_len, n_heads, n_kv_heads, &tps);
  const long long need = srgpt_attention_prefill_paged_workspace(n_seqs, max_q_len, max_ctx_len, n_heads, n_kv_heads);
  if (workspace == nullptr) {  // no workspace: one CTA walks the whole context
    n_split = 1;
    tps = ceil_div(max_ctx_len, attn::BN);
  } else {
    SRGPT_CHECK_ARG(workspace_bytes >= need && (reinterpret_cast<uintptr_t>(workspace) & 15) == 0);
  }
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  static bool configured = false;
  if (!configured) {
    SRGPT_CHECK_CUDA(cudaFuncSetAttribute(attn::attn_prefill_paged_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(attn::PagedSmem)));
    configured = true;
  }
  const int group = n_heads / n_kv_heads;
  const int ws_rows = n_seqs * max_q_len;
  float* ws_o = reinterpret_cast<float*>(workspace);
  float* ws_ml = ws_o == nullptr ? nullptr : ws_o + (size_t)n_split * ws_rows * n_heads * 128;
  const dim3 grid(ceil_div(max_q_len, attn::BM / group), n_kv_heads, n_seqs * n_split);
  attn::attn_prefill_paged_kernel<<<grid, attn::NTHREADS, sizeof(attn::PagedSmem), st>>>(
      reinterpret_cast<const bf16*>(q), q_ld, reinterpret_cast<bf16*>(out), o_ld, reinterpret_cast<const bf16*>(kv_pages), page_tables,
      page_table_stride, cu_q, start_pos, n_heads, n_kv_heads, group, n_split, tps, ws_o, ws_ml, ws_rows, scale * 1.4426950408889634f);
  SRGPT_CHECK_LAUNCH();
  if (n_split > 1) {
    attn::attn_paged_combine_kernel<<<dim3(ws_rows, n_heads), 128, 0, st>>>(ws_o, ws_ml, reinterpret_cast<bf16*>(out), o_ld, cu_q, n_seqs, n_split,
                                                                          ws_rows, n_heads);
    SRGPT_CHECK_LAUNCH();
  }
  return SRGPT_OK;
}

// B sequences, one new token each (batched decode): q rows [B, q_ld] (e.g. the q columns of a fused qkv buffer), out [B, o_ld],
// page_tables [B, pt_stride], kv_len_minus1 [B] (position of each sequence's newest row).
extern "C" __attribute__((visibility("default"))) int srgpt_attention_decode_batched_bf16(const void* q, int q_ld, void* out, int o_ld, const void* kv_pages,
                                                                                          const int* page_tables, int pt_stride, int page_size,
                                                                                          const int* kv_len_minus1, int batch, int n_heads, int n_kv_heads,
                                                                                          int head_dim, float scale, void* stream) {
  SRGPT_CHECK_ARG(q && out && kv_pages && page_tables && kv_len_minus1 && batch > 0 && batch <= 65535);
  SRGPT_CHECK_ARG(n_heads > 0 && n_kv_heads > 0 && (n_heads % n_kv_heads) == 0 && page_size > 0 && pt_stride > 0);
  SRGPT_CHECK_ARG(aligned16(q) && aligned16(kv_pages) && (q_ld % 8) == 0 && q_ld >= n_heads * head_dim && o_ld >= n_heads * head_dim);
  if (head_dim != 128) {
    set_last_error("srgpt_attention_decode_batched_bf16: head_dim %d unsupported (128 only)", head_dim);
    return SRGPT_ERR_UNSUPPORTED;
  }
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  const int group = n_heads / n_kv_heads;
  const float sl2 = scale * 1.4426950408889634f;
  const bf16* qp = reinterpret_cast<const bf16*>(q);
  bf16* op = reinterpret_cast<bf16*>(out);
  const bf16* kp = reinterpret_cast<const bf16*>(kv_pages);
  const dim3 grid(n_kv_heads, batch);
  switch (group) {  // one CTA per (kv head, sequence): the group's query heads share one pass over the K / V rows
    case 1: attn::attn_decode_gqa_kernel<1><<<grid, attn::DEC_THREADS, 0, st>>>(qp, q_ld, op, o_ld, kp, page_tables, pt_stride, page_size, kv_len_minus1, n_kv_heads, sl2); break;
    case 2: attn::attn_decode_gqa_kernel<2><<<grid, attn::DEC_THREADS, 0, st>>>(qp, q_ld, op, o_ld, kp, page_tables, pt_stride, page_size, kv_len_minus1, n_kv_heads, sl2); break;
    case 4: attn::attn_decode_gqa_kernel<4><<<grid, attn::DEC_THREADS, 0, st>>>(qp, q_ld, op, o_ld, kp, page_tables, pt_stride, page_size, kv_len_minus1, n_kv_heads, sl2); break;
    case 8: attn::attn_decode_gqa_kernel<8><<<grid, attn::DEC_THREADS, 0, st>>>(qp, q_ld, op, o_ld, kp, page_tables, pt_stride, page_size, kv_len_minus1, n_kv_heads, sl2); break;
    default:
      attn::attn_decode_kernel<<<dim3(n_heads, batch), attn::DEC_THREADS, 0, st>>>(qp, op, kp, page_tables, page_size, kv_len_minus1, n_kv_heads, group, sl2,
                                                                                 nullptr, 1, 0, q_ld, o_ld, pt_stride);
  }
  SRGPT_CHECK_LAUNCH();
  return SRGPT_OK;
}

// One rank of a tensor-parallel decoder: n_heads_local query heads (q / out are [n_heads_local * 128]) over kv heads
// [kv_head_off, kv_head_off + n_heads_local / group) of a cache whose rows hold n_kv_total heads.
extern "C" __attribute__((visibility("default"))) int srgpt_attention_decode_tp_bf16(const void* q, void* out, const void* kv_pages, const int* page_table, int page_size,
                                                                                     const int* kv_len_minus1, int n_heads_local, int group, int n_kv_total,
                                                                                     int kv_head_off, int head_dim, float scale, void* stream) {
  SRGPT_CHECK_ARG(q && out && kv_pages && page_table && kv_len_minus1);
  SRGPT_CHECK_ARG(n_heads_local > 0 && group > 0 && (n_heads_local % group) == 0 && page_size > 0);
  SRGPT_CHECK_ARG(kv_head_off >= 0 && kv_head_off + n_heads_local / group <= n_kv_total);
  SRGPT_CHECK_ARG(aligned16(q) && aligned16(kv_pages));
  if (head_dim != 128) {
    set_last_error("srgpt_attention_decode_tp_bf16: head_dim %d unsupported (128 only)", head_dim);
    return SRGPT_ERR_UNSUPPORTED;
  }
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(n_heads_local);
  cfg.blockDim = dim3(attn::DEC_THREADS);
  cfg.stream = reinterpret_cast<cudaStream_t>(stream);
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = pdl_enabled() ? 1 : 0;
  SRGPT_CHECK_CUDA(cudaLaunchKernelEx(&cfg, attn::attn_decode_kernel, reinterpret_cast<const bf16*>(q), reinterpret_cast<bf16*>(out),
                                      reinterpret_cast<const bf16*>(kv_pages), page_table, page_size, kv_len_minus1, n_kv_total, group,
                                      scale * 1.4426950408889634f, trace_next_slot(), 1, kv_head_off, 0, 0, 0));
  return SRGPT_OK;
}
