"""torch.Tensor-facing wrappers over the C-ABI (one function per exported kernel group).

torch is used for device memory and streams only; every computation below is a hand-written
sm_100a kernel in ``csrc/``.  All wrappers raise ``SrgptError`` on any failure (no fallbacks).
"""
from __future__ import annotations

from typing import Optional

import torch

from . import _lib
from ._lib import SrgptError
from ._lib import check as _check_rc

_KERNELS_PER_CALL = {"srgpt_lm_head_local_best_bf16": 2, "srgpt_mask_pool_bf16": 2, "srgpt_mask_weights": 2, "srgpt_lm_head_argmax_bf16": 2, "srgpt_depth_to_u8x3": 3}


def check(rc: int, what: str) -> None:
    global LAUNCHES
    _check_rc(rc, what)
    LAUNCHES += _KERNELS_PER_CALL.get(what, 1)

EPI_NONE, EPI_BIAS, EPI_BIAS_GELU_TANH, EPI_BIAS_GELU_ERF, EPI_BIAS_RESIDUAL, EPI_SWIGLU, EPI_BIAS_QUICK_GELU = range(7)
GEMV_PLAIN, GEMV_SWIGLU, GEMV_QKV_ROPE = range(3)
ORDER_ROWMAJOR, ORDER_NESTED = 0, 2

BF16 = torch.bfloat16
F16 = torch.float16
_ELEM_NAMES = {torch.bfloat16: "bf16", torch.float16: "f16"}
_ELEM_DTYPES = {v: k for k, v in _ELEM_NAMES.items()}


def ELEM() -> torch.dtype:
    """The 16-bit element type the ops currently compute in (which build of the library ``_lib.load()`` hands out)."""
    return _ELEM_DTYPES[_lib.current_elem()]


class elem_dtype:
    """``with ops.elem_dtype(torch.float16): ...`` - route the ops through the IEEE-half build of the kernels (the reference loader's
    default dtype, llava/model/builder.py:62) instead of the bfloat16 one.  The models wrap their public entry points in this with their
    own dtype, so a bf16 and an fp16 model can live in one process (one thread at a time: the setting is process-wide)."""

    def __init__(self, dtype: torch.dtype):
        if dtype not in _ELEM_NAMES:
            raise SrgptError(f"unsupported compute dtype {dtype}: the kernels are built for torch.bfloat16 and torch.float16")
        self.name = _ELEM_NAMES[dtype]

    def __enter__(self):
        self.prev = _lib.set_elem(self.name)
        return self

    def __exit__(self, *exc):
        _lib.set_elem(self.prev)
        return False


def in_own_dtype(fn):
    """Method decorator: run the method with the kernels of ``self.dtype`` (torch.bfloat16 / torch.float16)."""
    import functools

    @functools.wraps(fn)
    def wrapped(self, *a, **k):
        with elem_dtype(self.dtype):
            return fn(self, *a, **k)

    return wrapped


# number of OUR kernels launched through this module (bench.py's `gpu_launches`); CUDA-graph replays
# are added by the decoder (kernels_per_decode_step per replay)
LAUNCHES = 0


def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


def _p(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


def _need(t: torch.Tensor, dtype, name: str) -> None:
    if not t.is_cuda:
        raise SrgptError(f"{name}: expected a CUDA tensor (the sm_100a kernels have no CPU fallback)")
    if t.dtype != dtype:
        raise SrgptError(f"{name}: expected dtype {dtype}, got {t.dtype}")


def _rowmajor2d(t: torch.Tensor, name: str) -> int:
    if t.dim() != 2 or t.stride(1) != 1:
        raise SrgptError(f"{name}: expected a 2-D tensor with unit inner stride, got shape {tuple(t.shape)} strides {t.stride()}")
    return t.stride(0)


# workspace of the short-prompt GEMM configuration (include/srgpt_b200.h: srgpt_gemm_set_workspace): owned here, one per process,
# registered on the first GEMM call on a device (the library keeps only the pointer)
_GEMM_WS = {}  # element type -> buffer (each build of the library keeps its own registration)


def _ensure_gemm_workspace(device) -> None:
    elem = _lib.current_elem()
    if elem in _GEMM_WS:
        return
    lib = _lib.load()
    n = int(lib.srgpt_gemm_workspace_bytes())
    ws = _GEMM_WS[elem] = torch.zeros(n + 1024, dtype=torch.uint8, device=device)
    off = (-ws.data_ptr()) % 1024
    torch.cuda.synchronize(device)  # the zero fill is complete before any kernel polls the flags
    check(lib.srgpt_gemm_set_workspace(ws.data_ptr() + off, n), "srgpt_gemm_set_workspace")
    global LAUNCHES
    LAUNCHES -= 1


# ------------------------------------------------------------------------------------------------
def gemm(a: torch.Tensor, w: torch.Tensor, bias: Optional[torch.Tensor] = None, residual: Optional[torch.Tensor] = None,
         epilogue: int = EPI_NONE, out: Optional[torch.Tensor] = None, out_fp32: bool = False,
         res_row_mod: int = 0) -> torch.Tensor:
    """out[M,N] = epilogue(a[M,K] @ w[N,K]^T) on tcgen05 tensor cores."""
    _need(a, ELEM(), "gemm.a"); _need(w, ELEM(), "gemm.w")
    _ensure_gemm_workspace(a.device)
    lda, ldw = _rowmajor2d(a, "gemm.a"), _rowmajor2d(w, "gemm.w")
    M, K = a.shape
    N, K2 = w.shape
    if K != K2:
        raise SrgptError(f"gemm: K mismatch {K} vs {K2}")
    n_out = N // 2 if epilogue == EPI_SWIGLU else N
    if out is None:
        out = torch.empty((M, n_out), dtype=torch.float32 if out_fp32 else ELEM(), device=a.device)
    else:
        _need(out, torch.float32 if out_fp32 else ELEM(), "gemm.out")
        if out.shape != (M, n_out):
            raise SrgptError(f"gemm.out: expected {(M, n_out)}, got {tuple(out.shape)}")
    ldc = _rowmajor2d(out, "gemm.out")
    ldr = 0
    if residual is not None:
        _need(residual, ELEM(), "gemm.residual")
        ldr = _rowmajor2d(residual, "gemm.residual")
    if bias is not None:
        _need(bias, ELEM(), "gemm.bias")
    check(_lib.load().srgpt_gemm_bf16(_p(a), lda, _p(w), ldw, _p(out), ldc, M, N, K, _p(bias), _p(residual), ldr,
                                      res_row_mod, epilogue, 1 if out_fp32 else 0, _stream()), "srgpt_gemm_bf16")
    return out


def layernorm(x: torch.Tensor, weight: torch.Tensor, bias: torch.Tensor, eps: float, act: int = 0,
              out: Optional[torch.Tensor] = None) -> torch.Tensor:
    _need(x, ELEM(), "layernorm.x")
    ldx = _rowmajor2d(x, "layernorm.x")
    rows, cols = x.shape
    if out is None:
        out = torch.empty((rows, cols), dtype=ELEM(), device=x.device)
    check(_lib.load().srgpt_layernorm_bf16(_p(x), ldx, _p(weight), _p(bias), _p(out), _rowmajor2d(out, "layernorm.out"),
                                           rows, cols, eps, act, _stream()), "srgpt_layernorm_bf16")
    return out


def downsample_layernorm(x: torch.Tensor, weight: torch.Tensor, bias: torch.Tensor, eps: float) -> torch.Tensor:
    """x [n, side*side, C] -> [n, ceil(side/2)^2, 4C] (DownSampleBlock + LayerNorm)."""
    _need(x, ELEM(), "downsample_layernorm.x")
    if x.dim() != 3 or not x.is_contiguous():
        raise SrgptError("downsample_layernorm: expected contiguous [n, side*side, C]")
    n, hw, c = x.shape
    side = int(round(hw ** 0.5))
    if side * side != hw:
        raise SrgptError(f"downsample_layernorm: {hw} tokens is not a square grid")
    half = (side + 1) // 2
    out = torch.empty((n, half * half, 4 * c), dtype=ELEM(), device=x.device)
    check(_lib.load().srgpt_downsample_layernorm_bf16(_p(x), _p(weight), _p(bias), _p(out), n, side, c, eps, _stream()),
          "srgpt_downsample_layernorm_bf16")
    return out


def rmsnorm(x: torch.Tensor, weight: torch.Tensor, eps: float, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    _need(x, ELEM(), "rmsnorm.x")
    ldx = _rowmajor2d(x, "rmsnorm.x")
    rows, cols = x.shape
    if out is None:
        out = torch.empty((rows, cols), dtype=ELEM(), device=x.device)
    check(_lib.load().srgpt_rmsnorm_bf16(_p(x), ldx, _p(weight), _p(out), _rowmajor2d(out, "rmsnorm.out"), rows, cols, eps,
                                         _stream()), "srgpt_rmsnorm_bf16")
    return out


def patchify(images: torch.Tensor, patch: int, ldk: int) -> torch.Tensor:
    if not images.is_cuda or images.dim() != 4 or images.shape[1] != 3 or not images.is_contiguous():
        raise SrgptError("patchify: expected a contiguous CUDA tensor [n, 3, R, R]")
    if images.dtype not in (torch.float32, ELEM()):
        raise SrgptError(f"patchify: unsupported dtype {images.dtype}")
    n, _, R, R2 = images.shape
    if R != R2:
        raise SrgptError("patchify: square images only")
    P = R // patch
    out = torch.empty((n * P * P, ldk), dtype=ELEM(), device=images.device)
    check(_lib.load().srgpt_patchify_bf16(_p(images), 1 if images.dtype == ELEM() else 0, _p(out), n, R, patch, ldk, _stream()),
          "srgpt_patchify_bf16")
    return out


def splice_rows(src0: torch.Tensor, src1, src2, src3, src_id: torch.Tensor, src_row: torch.Tensor) -> torch.Tensor:
    _need(src0, ELEM(), "splice.src0"); _need(src_id, torch.int32, "splice.src_id"); _need(src_row, torch.int32, "splice.src_row")
    cols = src0.shape[-1]
    rows = src_id.numel()
    for s in (src1, src2, src3):
        if s is not None:
            _need(s, ELEM(), "splice.src")
            if s.shape[-1] != cols or not s.is_contiguous():
                raise SrgptError("splice: all sources must be contiguous with the same width")
    out = torch.empty((rows, cols), dtype=ELEM(), device=src0.device)
    check(_lib.load().srgpt_splice_rows_bf16(_p(src0), _p(src1), _p(src2), _p(src3), _p(src_id), _p(src_row), _p(out), rows,
                                             cols, _stream()), "srgpt_splice_rows_bf16")
    return out


# ------------------------------------------------------------------------------------------------
def mask_weights(masks: torch.Tensor, side: int, order: int) -> torch.Tensor:
    """masks [n_img, M, IH, IW] (fp32 or bf16) -> normalised bf16 pooling weights [n_img, M, side*side]."""
    if not masks.is_cuda or masks.dim() != 4 or not masks.is_contiguous():
        raise SrgptError("mask_weights: expected a contiguous CUDA tensor [n_img, M, IH, IW]")
    if masks.dtype not in (torch.float32, ELEM()):
        raise SrgptError(f"mask_weights: unsupported dtype {masks.dtype}")
    n, M, IH, IW = masks.shape
    # base_extractor.py:53-57: scale_factor = (L / (IH*IW)) ** 0.5 in Python doubles; ATen then uses
    # static_cast<float>(1.0 / scale_factor) as the source-index scale.
    scale_factor = ((side * side) / (IH * IW)) ** 0.5
    if int(IH * scale_factor) != side or int(IW * scale_factor) != side:
        raise SrgptError(f"mask_weights: floor({IH}x{IW} * {scale_factor}) != {side} (non-square masks are unsupported)")
    rscale = float(torch.tensor(1.0 / scale_factor, dtype=torch.float64).to(torch.float32))
    lib = _lib.load()
    L = side * side
    ld = (L + 7) // 8 * 8  # rows padded to 16 bytes (include/srgpt_b200.h); the returned view hides the pad
    w = torch.empty((n, M, ld), dtype=ELEM(), device=masks.device)[:, :, :L]
    ws = torch.empty(lib.srgpt_mask_weights_workspace(n, M, side), dtype=torch.uint8, device=masks.device)
    check(lib.srgpt_mask_weights(_p(masks), 1 if masks.dtype == ELEM() else 0, _p(w), _p(ws), n, M, IH, IW, side, rscale, order,
                                 _stream()), "srgpt_mask_weights")
    return w


def mask_pool(x: torch.Tensor, w: torch.Tensor, workspace: Optional[torch.Tensor] = None) -> torch.Tensor:
    """x [n_img, L, C] bf16, w [n_img, M, L] bf16 -> [n_img, M, C] bf16."""
    _need(x, ELEM(), "mask_pool.x"); _need(w, ELEM(), "mask_pool.w")
    if x.dim() != 3 or w.dim() != 3 or not x.is_contiguous():
        raise SrgptError("mask_pool: expected contiguous x [n, L, C] and w [n, M, L]")
    n, L, Cc = x.shape
    n2, M, L2 = w.shape
    ld = (L2 + 7) // 8 * 8
    if w.stride(2) != 1 or w.stride(1) != ld or w.stride(0) != M * ld:
        raise SrgptError("mask_pool: w must be the [n, M, L] view of a [n, M, round_up(L, 8)] buffer (what mask_weights returns)")
    if n != n2 or L != L2:
        raise SrgptError("mask_pool: shape mismatch between x and w")
    need = _lib.load().srgpt_mask_pool_workspace(n, M, L, Cc)
    if workspace is None or workspace.numel() * workspace.element_size() < need:
        workspace = torch.empty((need + 3) // 4, dtype=torch.float32, device=x.device)
    out = torch.empty((n, M, Cc), dtype=ELEM(), device=x.device)
    check(_lib.load().srgpt_mask_pool_bf16(_p(x), _p(w), _p(out), _p(workspace), n, M, L, Cc, _stream()), "srgpt_mask_pool_bf16")
    return out


def adaptive_avgpool(x: torch.Tensor, side: int, out_side: int, order: int) -> torch.Tensor:
    _need(x, ELEM(), "adaptive_avgpool.x")
    n, L, Cc = x.shape
    if L != side * side or not x.is_contiguous():
        raise SrgptError("adaptive_avgpool: expected contiguous [n, side*side, C]")
    y = torch.empty((n, out_side * out_side, Cc), dtype=ELEM(), device=x.device)
    check(_lib.load().srgpt_adaptive_avgpool_bf16(_p(x), _p(y), n, side, out_side, Cc, order, _stream()),
          "srgpt_adaptive_avgpool_bf16")
    return y


def reorder_rows(x: torch.Tensor, side: int, from_order: int, to_order: int) -> torch.Tensor:
    _need(x, ELEM(), "reorder_rows.x")
    n, L, Cc = x.shape
    if L != side * side or not x.is_contiguous():
        raise SrgptError("reorder_rows: expected contiguous [n, side*side, C]")
    y = torch.empty_like(x)
    check(_lib.load().srgpt_reorder_rows_bf16(_p(x), _p(y), n, side, Cc, from_order, to_order, _stream()), "srgpt_reorder_rows_bf16")
    return y


def depth_to_u8x3(depth: torch.Tensor, H: int, W: int) -> torch.Tensor:
    """depth [h, w] or [1, h, w] fp32 -> [H, W, 3] uint8 (eval_spatial.py:99-105)."""
    _need(depth, torch.float32, "depth_to_u8x3.depth")
    d = depth.reshape(depth.shape[-2], depth.shape[-1]).contiguous()
    out = torch.empty((H, W, 3), dtype=torch.uint8, device=depth.device)
    ws = torch.empty(H * W + 2, dtype=torch.float32, device=depth.device)
    check(_lib.load().srgpt_depth_to_u8x3(_p(d), d.shape[0], d.shape[1], _p(out), H, W, _p(ws), _stream()), "srgpt_depth_to_u8x3")
    return out


# ------------------------------------------------------------------------------------------------
def attention_prefill(q: torch.Tensor, k: torch.Tensor, v: torch.Tensor, batch: int, seqlen: int, n_heads: int,
                      n_kv_heads: int, head_dim: int, scale: float, causal: bool,
                      out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """q/k/v: 2-D row-major views [batch*seqlen, heads*head_dim] (may be column slices of a fused qkv buffer)."""
    for t, nm in ((q, "q"), (k, "k"), (v, "v")):
        _need(t, ELEM(), f"attention_prefill.{nm}")
    q_ld, k_ld, v_ld = _rowmajor2d(q, "q"), _rowmajor2d(k, "k"), _rowmajor2d(v, "v")
    if k_ld != v_ld:
        raise SrgptError("attention_prefill: k and v must share a row stride")
    if out is None:
        out = torch.empty((batch * seqlen, n_heads * head_dim), dtype=ELEM(), device=q.device)
    check(_lib.load().srgpt_attention_prefill_bf16(_p(q), _p(k), _p(v), _p(out), q_ld, k_ld, _rowmajor2d(out, "out"), batch,
                                                   seqlen, n_heads, n_kv_heads, head_dim, scale, 1 if causal else 0, _stream()),
          "srgpt_attention_prefill_bf16")
    return out


def attention_prefill_varlen(q: torch.Tensor, k: torch.Tensor, v: torch.Tensor, cu_seqlens: torch.Tensor, max_seqlen: int,
                             n_heads: int, n_kv_heads: int, head_dim: int, scale: float, causal: bool) -> torch.Tensor:
    """Packed sequences: rows [cu_seqlens[b], cu_seqlens[b+1]) belong to sequence b (modeling_llama.py:540-562)."""
    for t, nm in ((q, "q"), (k, "k"), (v, "v")):
        _need(t, ELEM(), f"attention_prefill_varlen.{nm}")
    _need(cu_seqlens, torch.int32, "attention_prefill_varlen.cu_seqlens")
    q_ld, k_ld, v_ld = _rowmajor2d(q, "q"), _rowmajor2d(k, "k"), _rowmajor2d(v, "v")
    if k_ld != v_ld:
        raise SrgptError("attention_prefill_varlen: k and v must share a row stride")
    out = torch.empty((q.shape[0], n_heads * head_dim), dtype=ELEM(), device=q.device)
    check(_lib.load().srgpt_attention_prefill_varlen_bf16(_p(q), _p(k), _p(v), _p(out), q_ld, k_ld, _rowmajor2d(out, "out"),
                                                          cu_seqlens.numel() - 1, _p(cu_seqlens), max_seqlen, q.shape[0], n_heads, n_kv_heads,
                                                          head_dim, scale, 1 if causal else 0, _stream()),
          "srgpt_attention_prefill_varlen_bf16")
    return out


def attention_prefill_paged_workspace(n_seqs: int, max_q_len: int, max_ctx_len: int, n_heads: int, n_kv_heads: int, device) -> Optional[torch.Tensor]:
    """fp32 partials of the paged kernel's context split for this shape (None when the shape runs unsplit)."""
    n = _lib.load().srgpt_attention_prefill_paged_workspace(n_seqs, max_q_len, max_ctx_len, n_heads, n_kv_heads)
    if n < 0:
        raise SrgptError(f"attention_prefill_paged: unsupported shape n_seqs={n_seqs} max_q_len={max_q_len} max_ctx_len={max_ctx_len} "
                         f"heads={n_heads}/{n_kv_heads}")
    return torch.empty(n // 4, dtype=torch.float32, device=device) if n else None


def attention_prefill_paged(q: torch.Tensor, kv_pages: torch.Tensor, page_tables: torch.Tensor, page_size: int, cu_q: torch.Tensor,
                            start_pos: torch.Tensor, max_q_len: int, max_ctx_len: int, n_heads: int, n_kv_heads: int, head_dim: int,
                            scale: float, out: Optional[torch.Tensor] = None, split: bool = True) -> torch.Tensor:
    """New rows over the paged cache of ONE layer (modeling_llama.py:451-456 + 564-566 with q_len < kv_len): rows
    [cu_q[b], cu_q[b+1]) of q [rows, >= n_heads*head_dim] are sequence b's rows at positions start_pos[b] + i, each attends to
    positions 0..p through page_tables[b].  The rows' own K/V must already be in the pages.  ``split=False`` runs without the
    context split (one CTA walks the whole context)."""
    _need(q, ELEM(), "attention_prefill_paged.q")
    _need(kv_pages, ELEM(), "attention_prefill_paged.kv_pages")
    for t, nm in ((page_tables, "page_tables"), (cu_q, "cu_q"), (start_pos, "start_pos")):
        _need(t, torch.int32, f"attention_prefill_paged.{nm}")
    n_seqs = cu_q.numel() - 1
    if page_tables.dim() != 2 or page_tables.shape[0] < n_seqs or page_tables.stride(1) != 1 or start_pos.numel() < n_seqs:
        raise SrgptError("attention_prefill_paged: page_tables [n_seqs, cap] / start_pos [n_seqs] expected")
    if out is None:
        out = torch.empty((q.shape[0], n_heads * head_dim), dtype=ELEM(), device=q.device)
    ws = attention_prefill_paged_workspace(n_seqs, max_q_len, max_ctx_len, n_heads, n_kv_heads, q.device) if split else None
    check(_lib.load().srgpt_attention_prefill_paged_bf16(_p(q), _rowmajor2d(q, "q"), _p(out), _rowmajor2d(out, "out"), _p(kv_pages), _p(page_tables),
                                                         page_tables.stride(0), page_size, n_seqs, _p(cu_q), _p(start_pos), max_q_len, max_ctx_len,
                                                         n_heads, n_kv_heads, head_dim, scale, _p(ws), 0 if ws is None else ws.numel() * 4, _stream()),
          "srgpt_attention_prefill_paged_bf16")
    if ws is not None:
        _count(2)
    return out


def rope_kv_append_varlen(qkv: torch.Tensor, n_heads: int, n_kv_heads: int, head_dim: int, cos_tab: torch.Tensor, sin_tab: torch.Tensor,
                          start_pos: torch.Tensor, kv_pages: torch.Tensor, page_tables: torch.Tensor, page_size: int,
                          cu_seqlens: torch.Tensor) -> None:
    _need(qkv, ELEM(), "rope_kv_append_varlen.qkv")
    if not qkv.is_contiguous() or qkv.shape[1] != (n_heads + 2 * n_kv_heads) * head_dim:
        raise SrgptError("rope_kv_append_varlen: qkv must be contiguous [rows, (nh + 2 nkv) * hd]")
    for t, nm in ((start_pos, "start_pos"), (page_tables, "page_tables"), (cu_seqlens, "cu_seqlens")):
        _need(t, torch.int32, f"rope_kv_append_varlen.{nm}")
    n_seqs = cu_seqlens.numel() - 1
    if page_tables.dim() != 2 or page_tables.shape[0] < n_seqs or page_tables.stride(1) != 1 or start_pos.numel() < n_seqs:
        raise SrgptError("rope_kv_append_varlen: page_tables [n_seqs, cap] / start_pos [n_seqs] expected")
    check(_lib.load().srgpt_rope_kv_append_varlen_bf16(_p(qkv), qkv.shape[0], n_heads, n_kv_heads, head_dim, _p(cos_tab), _p(sin_tab),
                                                       _p(start_pos), _p(kv_pages), _p(page_tables), page_tables.stride(0), page_size,
                                                       n_seqs, _p(cu_seqlens), _stream()), "srgpt_rope_kv_append_varlen_bf16")


def rope_kv_append(qkv: torch.Tensor, n_heads: int, n_kv_heads: int, head_dim: int, cos_tab: torch.Tensor,
                   sin_tab: torch.Tensor, start_pos: torch.Tensor, kv_pages: torch.Tensor, page_table: torch.Tensor,
                   page_size: int) -> None:
    _need(qkv, ELEM(), "rope_kv_append.qkv")
    if not qkv.is_contiguous() or qkv.shape[1] != (n_heads + 2 * n_kv_heads) * head_dim:
        raise SrgptError("rope_kv_append: qkv must be contiguous [rows, (nh + 2 nkv) * hd]")
    _need(start_pos, torch.int32, "rope_kv_append.start_pos"); _need(page_table, torch.int32, "rope_kv_append.page_table")
    check(_lib.load().srgpt_rope_kv_append_bf16(_p(qkv), qkv.shape[0], n_heads, n_kv_heads, head_dim, _p(cos_tab), _p(sin_tab),
                                                _p(start_pos), _p(kv_pages), _p(page_table), page_size, _stream()),
          "srgpt_rope_kv_append_bf16")


def attention_decode(q: torch.Tensor, out: torch.Tensor, kv_pages: torch.Tensor, page_table: torch.Tensor, page_size: int,
                     pos: torch.Tensor, n_heads: int, n_kv_heads: int, head_dim: int, scale: float) -> torch.Tensor:
    check(_lib.load().srgpt_attention_decode_bf16(_p(q), _p(out), _p(kv_pages), _p(page_table), page_size, _p(pos), n_heads,
                                                  n_kv_heads, head_dim, scale, _stream()), "srgpt_attention_decode_bf16")
    return out


def gemv(x: torch.Tensor, w: torch.Tensor, y: torch.Tensor, norm_weight: Optional[torch.Tensor] = None, eps: float = 0.0,
         residual: Optional[torch.Tensor] = None, mode: int = GEMV_PLAIN, n_heads: int = 0, n_kv_heads: int = 0,
         head_dim: int = 0, cos_tab=None, sin_tab=None, pos=None, kv_pages=None, page_table=None, page_size: int = 0) -> torch.Tensor:
    N, K = w.shape
    check(_lib.load().srgpt_gemv_bf16(_p(x), _p(w), w.stride(0), _p(y), N, K, _p(norm_weight), eps, _p(residual), mode, n_heads,
                                      n_kv_heads, head_dim, _p(cos_tab), _p(sin_tab), _p(pos), _p(kv_pages), _p(page_table),
                                      page_size, _stream()), "srgpt_gemv_bf16")
    return y


# ---- host preprocessing on the GPU (preprocess.py) ---------------------------------------------------------------
def resample_u8(img: torch.Tensor, axis: int, out_size: int, kk: torch.Tensor, bounds: torch.Tensor, ksize: int) -> torch.Tensor:
    _need(img, torch.uint8, "resample_u8.img"); _need(kk, torch.int32, "resample_u8.kk"); _need(bounds, torch.int32, "resample_u8.bounds")
    H, W, Cc = img.shape
    out = torch.empty((out_size, W, Cc) if axis == 0 else (H, out_size, Cc), dtype=torch.uint8, device=img.device)
    check(_lib.load().srgpt_resample_u8(_p(img), _p(out), H, W, Cc, axis, out_size, _p(kk), _p(bounds), ksize, _stream()), "srgpt_resample_u8")
    return out


def u8_to_normalized_chw(img: torch.Tensor, scale: float, mean, std, do_normalize: bool = True) -> torch.Tensor:
    import ctypes
    _need(img, torch.uint8, "u8_to_normalized_chw.img")
    H, W, Cc = img.shape
    out = torch.empty((Cc, H, W), dtype=torch.float32, device=img.device)
    m3 = (ctypes.c_float * 3)(*([float(v) for v in mean] + [0.0] * 3)[:3])
    s3 = (ctypes.c_float * 3)(*([float(v) for v in std] + [1.0] * 3)[:3])
    check(_lib.load().srgpt_u8_to_normalized_chw(_p(img), _p(out), H, W, Cc, float(scale), m3, s3, 1 if do_normalize else 0, _stream()),
          "srgpt_u8_to_normalized_chw")
    return out


def resize_nearest_u8(img: torch.Tensor, out_h: int, out_w: int, ys: torch.Tensor, xs: torch.Tensor) -> torch.Tensor:
    _need(img, torch.uint8, "resize_nearest_u8.img"); _need(ys, torch.int32, "resize_nearest_u8.ys"); _need(xs, torch.int32, "resize_nearest_u8.xs")
    H, W = img.shape
    out = torch.empty((out_h, out_w), dtype=torch.float32, device=img.device)
    check(_lib.load().srgpt_resize_nearest_u8(_p(img), _p(out), H, W, out_h, out_w, _p(ys), _p(xs), _stream()), "srgpt_resize_nearest_u8")
    return out


# ---- batched decode ----------------------------------------------------------------------------------------------
def attention_decode_batched(q: torch.Tensor, out: torch.Tensor, kv_pages: torch.Tensor, page_tables: torch.Tensor, page_size: int, pos: torch.Tensor,
                             n_heads: int, n_kv_heads: int, head_dim: int, scale: float) -> torch.Tensor:
    """q [B, >= n_heads*hd] (row-strided view, e.g. the q columns of a fused qkv buffer), out [B, n_heads*hd], page_tables [>= B, cap],
    pos int32 [B] = position of every sequence's newest row."""
    _need(q, ELEM(), "attention_decode_batched.q"); _need(out, ELEM(), "attention_decode_batched.out")
    _need(page_tables, torch.int32, "attention_decode_batched.page_tables"); _need(pos, torch.int32, "attention_decode_batched.pos")
    B = q.shape[0]
    check(_lib.load().srgpt_attention_decode_batched_bf16(_p(q), _rowmajor2d(q, "q"), _p(out), _rowmajor2d(out, "out"), _p(kv_pages), _p(page_tables),
                                                          page_tables.stride(0), page_size, _p(pos), B, n_heads, n_kv_heads, head_dim, scale, _stream()),
          "srgpt_attention_decode_batched_bf16")
    return out


def decode_batch_advance(ids: torch.Tensor, embed_table: torch.Tensor, h: torch.Tensor, out_ids: torch.Tensor, step: torch.Tensor, pos: torch.Tensor,
                         ticket: torch.Tensor) -> None:
    _need(ids, torch.int64, "decode_batch_advance.ids"); _need(out_ids, torch.int64, "decode_batch_advance.out_ids")
    B, H = h.shape
    check(_lib.load().srgpt_decode_batch_advance(_p(ids), _p(embed_table), _p(h), H, _p(out_ids), _p(step), _p(pos), B, _p(ticket), _stream()),
          "srgpt_decode_batch_advance")


# ---- tensor-parallel decode (one rank's share) ---------------------------------------------------------------------
def gemv_tp_qkv(x, w_local, y_local, norm_weight, eps: float, n_heads_local: int, n_kv_local: int, head_dim: int, cos_tab, sin_tab, pos,
                kv_pages, page_table, page_size: int, kv_heads_total: int, kv_head_off: int) -> torch.Tensor:
    """RMSNorm + this rank's q/k/v rows + RoPE; K/V rows are appended to the full-layout cache at kv head `kv_head_off`."""
    N, K = w_local.shape
    check(_lib.load().srgpt_gemv_tp_bf16(_p(x), _p(w_local), w_local.stride(0), _p(y_local), N, K, _p(norm_weight), eps, GEMV_QKV_ROPE, n_heads_local,
                                         n_kv_local, head_dim, _p(cos_tab), _p(sin_tab), _p(pos), _p(kv_pages), _p(page_table), page_size,
                                         kv_heads_total, kv_head_off, None, _stream()), "srgpt_gemv_tp_bf16")
    return y_local


def gemv_tp_partial(x_local, w_local, partial_f32) -> torch.Tensor:
    """Row-parallel linear: fp32 partial sums over this rank's K slice (all-reduced by the caller)."""
    N, K = w_local.shape
    _need(partial_f32, torch.float32, "gemv_tp_partial.partial")
    check(_lib.load().srgpt_gemv_tp_bf16(_p(x_local), _p(w_local), w_local.stride(0), None, N, K, None, 0.0, GEMV_PLAIN, 0, 0, 0, None, None, None,
                                         None, None, 0, 0, 0, _p(partial_f32), _stream()), "srgpt_gemv_tp_bf16")
    return partial_f32


def attention_decode_tp(q_local, out_local, kv_pages, page_table, page_size: int, pos, n_heads_local: int, group: int, n_kv_total: int,
                        kv_head_off: int, head_dim: int, scale: float) -> torch.Tensor:
    check(_lib.load().srgpt_attention_decode_tp_bf16(_p(q_local), _p(out_local), _p(kv_pages), _p(page_table), page_size, _p(pos), n_heads_local, group,
                                                     n_kv_total, kv_head_off, head_dim, scale, _stream()), "srgpt_attention_decode_tp_bf16")
    return out_local


def tp_residual_add(h, partial_f32) -> None:
    check(_lib.load().srgpt_tp_residual_add_bf16(_p(h), _p(partial_f32), h.numel(), _stream()), "srgpt_tp_residual_add_bf16")


def lm_head_local_best(x, w_local, norm_weight, eps: float, workspace, index_base: int, best) -> None:
    V, K = w_local.shape
    _need(best, torch.int32, "lm_head_local_best.best")
    check(_lib.load().srgpt_lm_head_local_best_bf16(_p(x), _p(w_local), w_local.stride(0), V, K, _p(norm_weight), eps, _p(workspace), index_base, _p(best),
                                                    _stream()), "srgpt_lm_head_local_best_bf16")


def tp_pick_token(best_all, world: int, embed_table, next_x, out_ids, step, pos) -> None:
    _need(best_all, torch.int32, "tp_pick_token.best_all")
    K = 0 if embed_table is None else embed_table.shape[1]
    check(_lib.load().srgpt_tp_pick_token(_p(best_all), world, _p(embed_table), _p(next_x), K, _p(out_ids), _p(step), _p(pos), _stream()),
          "srgpt_tp_pick_token")


def tp_allreduce_residual(peer_bases, rank: int, world: int, slot_off: int, idx: int, epoch, step, h) -> None:
    """All-reduce of the ranks' fp32 partial sums (slot `slot_off` of every rank's symmetric buffer) over NVLink peer memory, fused
    with h = bf16(bf16(sum) + h).  ``peer_bases`` = ctypes array of the peer-mapped buffer addresses."""
    check(_lib.load().srgpt_tp_allreduce_residual_bf16(peer_bases, rank, world, slot_off, idx, _p(epoch), _p(step), _p(h), h.numel(), _stream()),
          "srgpt_tp_allreduce_residual_bf16")


def tp_allgather_pick(peer_bases, rank: int, world: int, slot_off: int, idx: int, epoch, embed_table, next_x, out_ids, step, pos) -> None:
    K = 0 if embed_table is None else embed_table.shape[1]
    check(_lib.load().srgpt_tp_allgather_pick_token(peer_bases, rank, world, slot_off, idx, _p(epoch), _p(embed_table), _p(next_x), K, _p(out_ids), _p(step),
                                                    _p(pos), _stream()), "srgpt_tp_allgather_pick_token")


def lm_head_workspace(V: int, device) -> torch.Tensor:
    return torch.empty(_lib.load().srgpt_lm_head_workspace(V), dtype=torch.uint8, device=device)


def lm_head_argmax(x: torch.Tensor, w: torch.Tensor, norm_weight: Optional[torch.Tensor], eps: float, workspace: torch.Tensor,
                   out_ids: torch.Tensor, step: torch.Tensor, pos: torch.Tensor, embed_table: Optional[torch.Tensor] = None,
                   next_x: Optional[torch.Tensor] = None, logits_out: Optional[torch.Tensor] = None) -> None:
    V, K = w.shape
    check(_lib.load().srgpt_lm_head_argmax_bf16(_p(x), _p(w), w.stride(0), V, K, _p(norm_weight), eps, _p(logits_out),
                                                _p(workspace), _p(embed_table), _p(next_x), _p(out_ids), _p(step), _p(pos),
                                                _stream()), "srgpt_lm_head_argmax_bf16")


def sample_top_p(logits: torch.Tensor, params: torch.Tensor, seed, step: torch.Tensor, step_offset: int, out_ids: torch.Tensor,
                 embed_table: Optional[torch.Tensor] = None, next_x: Optional[torch.Tensor] = None) -> None:
    """One token from softmax(logits / T) restricted to its top-p nucleus -> out_ids[step + step_offset] (and next_x = embed row).
    ``params`` = device float32 [temperature, top_p, top_k (0 = off)]; ``step`` = device int32 [1]; ``seed`` = device int64 [1]
    (read by the kernel at run time - graph-capturable), or a Python int for one-off eager calls."""
    if not isinstance(seed, torch.Tensor):
        seed = torch.tensor([int(seed) & 0x7FFFFFFFFFFFFFFF], dtype=torch.int64, device=logits.device)
    _need(seed, torch.int64, "sample_top_p.seed")
    _need(logits, torch.float32, "sample_top_p.logits"); _need(params, torch.float32, "sample_top_p.params")
    _need(step, torch.int32, "sample_top_p.step"); _need(out_ids, torch.int64, "sample_top_p.out_ids")
    if logits.dim() != 1 or not logits.is_contiguous() or params.numel() < 3:
        raise SrgptError("sample_top_p: logits must be a contiguous fp32 vector [V] and params [temperature, top_p, top_k]")
    K = 0 if embed_table is None else embed_table.shape[1]
    check(_lib.load().srgpt_sample_top_p_f32(_p(logits), logits.numel(), _p(params), _p(seed), _p(step), step_offset,
                                             _p(out_ids), _p(embed_table), _p(next_x), K, _stream()), "srgpt_sample_top_p_f32")


def beam_candidates(logits: torch.Tensor, beam_scores: torch.Tensor, cand_scores: torch.Tensor, cand_tokens: torch.Tensor) -> None:
    """Per beam row: the n_cand best (log_softmax(logits)[token] + beam_scores[row], token) -> cand_scores / cand_tokens [k, n_cand]."""
    _need(logits, ELEM(), "beam_candidates.logits"); _need(beam_scores, torch.float32, "beam_candidates.beam_scores")
    _need(cand_scores, torch.float32, "beam_candidates.cand_scores"); _need(cand_tokens, torch.int32, "beam_candidates.cand_tokens")
    k, V = logits.shape
    if cand_scores.shape != cand_tokens.shape or cand_scores.shape[0] != k or not cand_scores.is_contiguous() or not cand_tokens.is_contiguous():
        raise SrgptError("beam_candidates: cand_scores / cand_tokens must be contiguous [n_beams, n_cand]")
    check(_lib.load().srgpt_beam_candidates_bf16(_p(logits), _rowmajor2d(logits, "beam_candidates.logits"), k, V, _p(beam_scores), cand_scores.shape[1],
                                                 _p(cand_scores), _p(cand_tokens), _stream()), "srgpt_beam_candidates_bf16")


def argmax_f32(x: torch.Tensor) -> torch.Tensor:
    _need(x, torch.float32, "argmax_f32.x")
    rows, cols = x.shape
    out = torch.empty(rows, dtype=torch.int64, device=x.device)
    check(_lib.load().srgpt_argmax_f32(_p(x), rows, cols, _p(out), _stream()), "srgpt_argmax_f32")
    return out


def argmax_bf16(x: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    _need(x, ELEM(), "argmax_bf16.x")
    ldx = _rowmajor2d(x, "argmax_bf16.x")
    rows, cols = x.shape
    if out is None:
        out = torch.empty(rows, dtype=torch.int64, device=x.device)
    check(_lib.load().srgpt_argmax_bf16(_p(x), ldx, rows, cols, _p(out), _stream()), "srgpt_argmax_bf16")
    return out


# ------------------------------------------------------------------------------------------------ composite stacks
def _count(n: int) -> None:
    global LAUNCHES
    LAUNCHES += n - 1  # check() adds 1


def make_siglip_layer_array(layers):
    """ctypes array of srgpt_siglip_layer_weights over a list of VisionLayerW (keeps no tensor alive: the caller does)."""
    arr = (_lib.SiglipLayerWeights * len(layers))()
    for i, lw in enumerate(layers):
        for name in ("ln1_w", "ln1_b", "qkv_w", "qkv_b", "out_w", "out_b", "ln2_w", "ln2_b", "fc1_w", "fc1_b", "fc2_w", "fc2_b"):
            setattr(arr[i], name, getattr(lw, name).data_ptr())
    return arr


def make_llama_layer_array(layers, kv_pages_per_layer):
    arr = (_lib.LlamaLayerWeights * len(layers))()
    for i, lw in enumerate(layers):
        for name in ("in_norm", "qkv_w", "o_w", "post_norm", "gateup_w", "down_w"):
            setattr(arr[i], name, getattr(lw, name).data_ptr())
        arr[i].kv_pages = kv_pages_per_layer[i].data_ptr()
    return arr


def clip_embed(patch_embeds: torch.Tensor, class_embedding: torch.Tensor, position_embedding: torch.Tensor, n_img: int, T: int) -> torch.Tensor:
    """[n_img*T, D] patch embeddings -> [n_img*(T+1), D]: class token prepended, position embedding added (CLIPVisionEmbeddings)."""
    _need(patch_embeds, ELEM(), "clip_embed.patch_embeds")
    D = patch_embeds.shape[1]
    if patch_embeds.shape[0] != n_img * T or not patch_embeds.is_contiguous() or tuple(position_embedding.shape) != (T + 1, D):
        raise SrgptError(f"clip_embed: patch embeds {tuple(patch_embeds.shape)}, position embedding {tuple(position_embedding.shape)}, n_img {n_img}, T {T}")
    out = torch.empty((n_img * (T + 1), D), dtype=ELEM(), device=patch_embeds.device)
    check(_lib.load().srgpt_clip_embed_bf16(_p(patch_embeds), _p(class_embedding), _p(position_embedding), _p(out), n_img, T, D, _stream()),
          "srgpt_clip_embed_bf16")
    return out


def siglip_layers(x: torch.Tensor, layer_array, n_layers: int, n_img: int, T: int, D: int, heads: int, I: int, eps: float,
                  fc1_epilogue: int = EPI_BIAS_GELU_TANH) -> torch.Tensor:
    """n_layers pre-LN ViT encoder layers (SigLIP; CLIP with fc1_epilogue=EPI_BIAS_QUICK_GELU) in place on x [n_img*T, D]."""
    _need(x, ELEM(), "siglip_layers.x")
    _ensure_gemm_workspace(x.device)
    M = n_img * T
    dev = x.device
    ws_h = torch.empty((M, D), dtype=ELEM(), device=dev)
    ws_qkv = torch.empty((M, 3 * D), dtype=ELEM(), device=dev)
    ws_attn = torch.empty((M, D), dtype=ELEM(), device=dev)
    ws_mlp = torch.empty((M, I), dtype=ELEM(), device=dev)
    import ctypes
    check(_lib.load().srgpt_vit_layers_bf16(_p(x), ctypes.cast(layer_array, ctypes.c_void_p), n_layers, _p(ws_h), _p(ws_qkv),
                                            _p(ws_attn), _p(ws_mlp), n_img, T, D, heads, I, eps, fc1_epilogue, _stream()), "srgpt_vit_layers_bf16")
    _count(7 * n_layers)
    return x


def llama_prefill_layers(x: torch.Tensor, layer_array, n_layers: int, dims, cos, sin, start_pos, page_table, page_size: int,
                         cu_seqlens: Optional[torch.Tensor] = None, max_seqlen: int = 0) -> torch.Tensor:
    """All decoder layers over the prompt rows x [S, H] in place (K/V appended to the paged cache).  One prompt
    (page_table [cap], start_pos [1]) or, with cu_seqlens [n_seqs+1], n_seqs prompts packed back to back
    (page_table [n_seqs, cap], start_pos [n_seqs])."""
    _need(x, ELEM(), "llama_prefill_layers.x")
    _ensure_gemm_workspace(x.device)
    n_seqs, pt_stride = 1, 0
    if cu_seqlens is not None:
        _need(cu_seqlens, torch.int32, "llama_prefill_layers.cu_seqlens")
        n_seqs = cu_seqlens.numel() - 1
        if page_table.dim() != 2 or page_table.shape[0] < n_seqs or start_pos.numel() < n_seqs or page_table.stride(1) != 1:
            raise SrgptError("llama_prefill_layers: packed prompts need page_table [n_seqs, cap] and start_pos [n_seqs]")
        pt_stride = page_table.stride(0)
    S, H = x.shape
    nh, nkv, hd, I = dims.num_attention_heads, dims.num_key_value_heads, dims.head_dim, dims.intermediate_size
    dev = x.device
    ws_h = torch.empty((S, H), dtype=ELEM(), device=dev)
    ws_qkv = torch.empty((S, (nh + 2 * nkv) * hd), dtype=ELEM(), device=dev)
    ws_attn = torch.empty((S, nh * hd), dtype=ELEM(), device=dev)
    ws_act = torch.empty((S, I), dtype=ELEM(), device=dev)
    import ctypes
    check(_lib.load().srgpt_llama_prefill_layers_bf16(_p(x), ctypes.cast(layer_array, ctypes.c_void_p), n_layers, _p(ws_h), _p(ws_qkv),
                                                      _p(ws_attn), _p(ws_act), S, H, nh, nkv, hd, I, dims.rms_norm_eps, _p(cos), _p(sin),
                                                      _p(start_pos), _p(page_table), page_size, n_seqs, _p(cu_seqlens), max_seqlen, pt_stride,
                                                      _stream()), "srgpt_llama_prefill_layers_bf16")
    _count(8 * n_layers)
    return x


def llama_prefill_layers_paged(x: torch.Tensor, layer_array, n_layers: int, dims, cos, sin, start_pos, page_tables, page_size: int,
                               cu_seqlens: torch.Tensor, max_seqlen: int, max_ctx_len: int) -> torch.Tensor:
    """All decoder layers over new rows x [S, H] in place that CONTINUE cached sequences: chunk b (rows [cu_seqlens[b],
    cu_seqlens[b+1])) sits at positions start_pos[b].. and attends to everything its sequence has cached (page_tables [n_seqs, cap])."""
    _need(x, ELEM(), "llama_prefill_layers_paged.x")
    for t, nm in ((start_pos, "start_pos"), (page_tables, "page_tables"), (cu_seqlens, "cu_seqlens")):
        _need(t, torch.int32, f"llama_prefill_layers_paged.{nm}")
    n_seqs = cu_seqlens.numel() - 1
    if page_tables.dim() != 2 or page_tables.shape[0] < n_seqs or start_pos.numel() < n_seqs or page_tables.stride(1) != 1:
        raise SrgptError("llama_prefill_layers_paged: page_tables [n_seqs, cap] and start_pos [n_seqs] expected")
    _ensure_gemm_workspace(x.device)
    S, H = x.shape
    nh, nkv, hd, I = dims.num_attention_heads, dims.num_key_value_heads, dims.head_dim, dims.intermediate_size
    dev = x.device
    ws_h = torch.empty((S, H), dtype=ELEM(), device=dev)
    ws_qkv = torch.empty((S, (nh + 2 * nkv) * hd), dtype=ELEM(), device=dev)
    ws_attn = torch.empty((S, nh * hd), dtype=ELEM(), device=dev)
    ws_act = torch.empty((S, I), dtype=ELEM(), device=dev)
    ws_split = attention_prefill_paged_workspace(n_seqs, max_seqlen, max_ctx_len, nh, nkv, dev)
    import ctypes
    check(_lib.load().srgpt_llama_prefill_layers_paged_bf16(_p(x), ctypes.cast(layer_array, ctypes.c_void_p), n_layers, _p(ws_h), _p(ws_qkv),
                                                            _p(ws_attn), _p(ws_act), _p(ws_split), 0 if ws_split is None else ws_split.numel() * 4,
                                                            S, H, nh, nkv, hd, I, dims.rms_norm_eps, _p(cos), _p(sin), _p(start_pos), _p(page_tables),
                                                            page_tables.stride(0), page_size, n_seqs, _p(cu_seqlens), max_seqlen, max_ctx_len, _stream()),
          "srgpt_llama_prefill_layers_paged_bf16")
    _count((8 + (ws_split is not None)) * n_layers)
    return x


def llama_decode_step(h, layer_array, n_layers: int, q_buf, attn_buf, act_buf, dims, cos, sin, pos, page_table, page_size: int,
                      final_norm, lm_head, embed, lm_ws, out_ids, step, logits_out=None) -> None:
    import ctypes
    nh, nkv, hd, I = dims.num_attention_heads, dims.num_key_value_heads, dims.head_dim, dims.intermediate_size
    check(_lib.load().srgpt_llama_decode_step_bf16(_p(h), ctypes.cast(layer_array, ctypes.c_void_p), n_layers, _p(q_buf), _p(attn_buf),
                                                   _p(act_buf), dims.hidden_size, nh, nkv, hd, I, dims.rms_norm_eps, _p(cos), _p(sin),
                                                   _p(pos), _p(page_table), page_size, _p(final_norm), _p(lm_head), dims.vocab_size,
                                                   _p(embed), _p(lm_ws), _p(logits_out), _p(out_ids), _p(step), _stream()),
          "srgpt_llama_decode_step_bf16")
    _count(5 * n_layers + 2)
