"""Llama decoder on the sm_100a kernels: prefill (tcgen05 GEMMs + flash attention), paged KV cache,
and a CUDA-graph-captured decode step made of weight-streaming GEMV kernels.

Reference: llava/train/transformers_replace/models/llama/modeling_llama.py — LlamaModel.forward
(824-936), LlamaDecoderLayer (611-684), LlamaFlashAttention2 (405-566), LlamaMLP (194-223),
LlamaRMSNorm (61-75), rotary embedding (81-130, 160-191), lm_head + float() (1044-1045),
prepare_inputs_for_generation (1112-1149); greedy loop = HF GenerationMixin (llava_llama.py:212).
The reference re-allocates the KV cache with torch.cat every step (451-456) and launches ~25
torch kernels per layer per token; here one token is 5 kernels per layer replayed from a CUDA graph
with the position / step counters living in device memory.
"""
from __future__ import annotations

from typing import List, Optional

import torch

from . import ops
from .config import LlamaDims
from .weights import LlamaW

PAGE_SIZE = 16


def build_rope_tables(dims: LlamaDims, max_pos: int, device, dtype: torch.dtype = torch.bfloat16) -> (torch.Tensor, torch.Tensor):
    """cos/sin exactly as LlamaRotaryEmbedding.forward computes them (modeling_llama.py:86,117-130):
    fp32 inv_freq, fp32 outer product, cos/sin in fp32, cast to the model dtype.  Host-side table build (once)."""
    hd = dims.head_dim
    inv_freq = 1.0 / (dims.rope_theta ** (torch.arange(0, hd, 2, dtype=torch.int64).float() / hd))
    t = torch.arange(max_pos, dtype=torch.int64).float()
    if getattr(dims, "rope_scaling_factor", 1.0) != 1.0:  # LlamaLinearScalingRotaryEmbedding.forward (modeling_llama.py:136-140)
        t = t / float(dims.rope_scaling_factor)
    freqs = t[:, None] * inv_freq[None, :]
    return freqs.cos().to(dtype).to(device).contiguous(), freqs.sin().to(dtype).to(device).contiguous()


class PagedKVCache:
    """KV pages for all layers: [layers, n_pages, 2 (k,v), PAGE_SIZE, n_kv_heads, head_dim] bf16, a free list
    and per-sequence page tables (int32, device) of fixed capacity so decode graphs stay valid."""

    def __init__(self, dims: LlamaDims, n_pages: int, max_seqs: int, max_pages_per_seq: int, device, dtype: torch.dtype = torch.bfloat16):
        self.dims = dims
        self.n_pages = n_pages
        self.max_pages_per_seq = max_pages_per_seq
        self.pages = torch.zeros((dims.num_hidden_layers, n_pages, 2, PAGE_SIZE, dims.num_key_value_heads, dims.head_dim),
                                 dtype=dtype, device=device)
        # +1 spare column (a measured-and-dropped decode-attention variant read the page id of row pos+1; kept so tables stay 16-byte padded)
        self.page_tables = torch.zeros((max_seqs, max_pages_per_seq + 1), dtype=torch.int32, device=device)
        self.free: List[int] = list(range(n_pages - 1, -1, -1))
        self.owned: List[List[int]] = [[] for _ in range(max_seqs)]

    def reserve(self, seq: int, n_tokens: int) -> None:
        """Make sure sequence `seq` owns pages for positions [0, n_tokens)."""
        need = (n_tokens + PAGE_SIZE - 1) // PAGE_SIZE
        if need > self.max_pages_per_seq:
            raise RuntimeError(f"sequence needs {need} KV pages > capacity {self.max_pages_per_seq}")
        own = self.owned[seq]
        if need > len(own):
            add = need - len(own)
            if add > len(self.free):
                raise RuntimeError("KV cache exhausted")
            new = [self.free.pop() for _ in range(add)]
            start = len(own)
            own.extend(new)
            self.page_tables[seq, start:start + add] = torch.tensor(new, dtype=torch.int32)

    def reserve_many(self, n_tokens: List[int]) -> None:
        """reserve() for sequences 0..len-1 with ONE host->device copy of the page tables (a 32-request batch otherwise issues
        32 tiny copies between the encoders and the prefill)."""
        host = torch.zeros((len(n_tokens), self.page_tables.shape[1]), dtype=torch.int32)
        for seq, n in enumerate(n_tokens):
            need = (n + PAGE_SIZE - 1) // PAGE_SIZE
            if need > self.max_pages_per_seq:
                raise RuntimeError(f"sequence needs {need} KV pages > capacity {self.max_pages_per_seq}")
            own = self.owned[seq]
            if need > len(own):
                if need - len(own) > len(self.free):
                    raise RuntimeError("KV cache exhausted")
                own.extend(self.free.pop() for _ in range(need - len(own)))
            host[seq, :len(own)] = torch.tensor(own, dtype=torch.int32)
        self.page_tables[:len(n_tokens)].copy_(host, non_blocking=True)

    def release(self, seq: int) -> None:
        self.free.extend(reversed(self.owned[seq]))
        self.owned[seq] = []

    def layer(self, l: int) -> torch.Tensor:
        return self.pages[l]


class LlamaDecoder:
    def __init__(self, dims: LlamaDims, w: LlamaW, max_seq_len: int = 4096, max_new_tokens_cap: int = 4096, max_seqs: int = 1,
                 kv_pages: Optional[int] = None):
        self.dims = dims
        self.w = w
        dev = w.embed.device
        self.device = dev
        self.max_seq_len = max_seq_len
        self.dtype = w.embed.dtype  # torch.bfloat16 or torch.float16: selects the build of the kernels (ops.elem_dtype)
        self.cos, self.sin = build_rope_tables(dims, max_seq_len, dev, self.dtype)
        ppseq = (max_seq_len + PAGE_SIZE - 1) // PAGE_SIZE
        self.cache = PagedKVCache(dims, kv_pages if kv_pages is not None else ppseq * max_seqs, max_seqs, ppseq, dev, self.dtype)
        # the decode graph reads the page table of the sequence being decoded from this fixed buffer
        self.active_pt = torch.zeros(ppseq + 1, dtype=torch.int32, device=dev)
        H, nh, hd, I = dims.hidden_size, dims.num_attention_heads, dims.head_dim, dims.intermediate_size
        # decode-step state (static addresses -> graph-capturable)
        self.pos = torch.zeros(1, dtype=torch.int32, device=dev)       # position of the token being processed
        self.step = torch.zeros(1, dtype=torch.int32, device=dev)      # number of generated tokens so far
        self.out_ids = torch.zeros(max_new_tokens_cap, dtype=torch.int64, device=dev)
        self.h = torch.zeros(H, dtype=self.dtype, device=dev)      # residual stream of the current token
        self.q_buf = torch.zeros(nh * hd, dtype=self.dtype, device=dev)
        self.attn_buf = torch.zeros(nh * hd, dtype=self.dtype, device=dev)
        self.act_buf = torch.zeros(I, dtype=self.dtype, device=dev)
        self.lm_ws = ops.lm_head_workspace(dims.vocab_size, dev)
        self.scale = hd ** -0.5
        self._layer_array = ops.make_llama_layer_array(w.layers, [self.cache.layer(l) for l in range(dims.num_hidden_layers)])
        self._graph: Optional[torch.cuda.CUDAGraph] = None
        self._graph_sample: Optional[torch.cuda.CUDAGraph] = None
        self.kernels_per_decode_step = 5 * dims.num_hidden_layers + 2
        # sampling mode (do_sample=True): temperature / top_p live in device memory so one captured graph serves any setting
        self.sample_params = torch.tensor([1.0, 1.0, 0.0], dtype=torch.float32, device=dev)
        self.sample_logits: Optional[torch.Tensor] = None
        self.sample_seed = 0
        self.sample_seed_dev = torch.zeros(1, dtype=torch.int64, device=dev)  # device copy: the captured graph reads the seed at run time
        # bumped by every call that releases or re-lays out the cached pages: a KV handle filled in an older epoch is stale
        self.kv_epoch = 0

    def release_all(self) -> None:
        """Drop every cached sequence (the start of an unrelated request)."""
        for b in range(len(self.cache.owned)):
            self.cache.release(b)
        self.kv_epoch += 1

    # ---------------------------------------------------------------------------------------------
    @ops.in_own_dtype
    def ensure_capacity(self, n_seqs: int, tokens_per_seq: int) -> None:
        """Grow the paged cache so `n_seqs` sequences of `tokens_per_seq` tokens fit at once (batched prefill).
        Re-allocation drops all cached sequences and the captured decode graph (page addresses change)."""
        c = self.cache
        need_pages = n_seqs * ((tokens_per_seq + PAGE_SIZE - 1) // PAGE_SIZE)
        if n_seqs <= len(c.owned) and need_pages <= c.n_pages:
            return
        d = self.dims
        per_page = 2 * PAGE_SIZE * d.num_key_value_heads * d.head_dim * 2 * d.num_hidden_layers
        free_b, _ = torch.cuda.mem_get_info(self.device)
        cur_b = c.pages.numel() * 2
        if need_pages * per_page > free_b + cur_b - (2 << 30):
            raise RuntimeError(f"KV cache for {n_seqs} x {tokens_per_seq} tokens needs {need_pages * per_page >> 20} MiB, not available")
        self._graph = None
        self._graph_sample = None
        self.kv_epoch += 1
        n_pages_old, n_seqs_old = c.n_pages, len(c.owned)
        self.cache = None
        del c
        self.cache = PagedKVCache(d, max(need_pages, n_pages_old), max(n_seqs, n_seqs_old), (self.max_seq_len + PAGE_SIZE - 1) // PAGE_SIZE, self.device, self.dtype)
        self._layer_array = ops.make_llama_layer_array(self.w.layers, [self.cache.layer(l) for l in range(d.num_hidden_layers)])

    @ops.in_own_dtype
    def embed_tokens(self, ids: torch.Tensor) -> torch.Tensor:
        """Embedding gather through the splice kernel (source 0 only)."""
        flat = ids.reshape(-1).to(device=self.device, dtype=torch.int32)
        if flat.numel():  # nn.Embedding raises on an out-of-range id; the gather kernel itself has no bounds check
            lo, hi = int(flat.min()), int(flat.max())
            if lo < 0 or hi >= self.w.embed.shape[0]:
                raise IndexError(f"token id {lo if lo < 0 else hi} is outside the token table [0, {self.w.embed.shape[0]})")
        return ops.splice_rows(self.w.embed, None, None, None, torch.zeros_like(flat), flat)

    @ops.in_own_dtype
    def prefill_hidden(self, inputs_embeds: torch.Tensor, seq: int = 0, start_pos: int = 0) -> torch.Tensor:
        """Run all layers over one sequence's prompt rows [S, H] at positions [start_pos, start_pos + S); fills the KV cache;
        returns the final-layer residual stream [S, H] (before the final norm).  With start_pos > 0 the rows attend to the
        positions [0, start_pos) this sequence already holds in the cache (srgpt_llama_prefill_layers_paged_bf16), so calling it
        chunk by chunk is chunked prefill; start_pos == 0 is the one-shot prompt path."""
        d, w = self.dims, self.w
        S = inputs_embeds.shape[0]
        if start_pos + S > self.max_seq_len:
            raise RuntimeError(f"prompt of {S} tokens at {start_pos} exceeds max_seq_len {self.max_seq_len}")
        self.cache.reserve(seq, start_pos + S)
        sp = torch.tensor([start_pos], dtype=torch.int32, device=self.device)
        pt = self.cache.page_tables[seq]
        x = inputs_embeds.to(self.dtype).contiguous().clone()
        if start_pos == 0:
            return ops.llama_prefill_layers(x, self._layer_array, d.num_hidden_layers, d, self.cos, self.sin, sp, pt, PAGE_SIZE)
        cu = torch.tensor([0, S], dtype=torch.int32, device=self.device)
        return ops.llama_prefill_layers_paged(x, self._layer_array, d.num_hidden_layers, d, self.cos, self.sin, sp, self.cache.page_tables[seq:seq + 1],
                                              PAGE_SIZE, cu, S, start_pos + S)

    @ops.in_own_dtype
    def prefill_packed(self, packed_embeds: torch.Tensor, seq_lens: List[int]) -> torch.Tensor:
        """Prefill `len(seq_lens)` prompts packed back to back ([sum S_b, H]) into sequence slots 0..B-1 in ONE pass:
        every GEMM runs over all rows, attention / RoPE / KV append per sequence (the unpadded varlen path of
        modeling_llama.py:540-562).  The caller has reserved the pages.  Returns the final residual stream, packed."""
        d = self.dims
        B = len(seq_lens)
        if packed_embeds.shape[0] != sum(seq_lens) or B < 1 or min(seq_lens) < 1:
            raise RuntimeError("prefill_packed: rows do not match seq_lens")
        if max(seq_lens) > self.max_seq_len:
            raise RuntimeError(f"prompt of {max(seq_lens)} tokens exceeds max_seq_len {self.max_seq_len}")
        cu = torch.tensor([0] + list(torch.tensor(seq_lens).cumsum(0).tolist()), dtype=torch.int32).to(self.device)
        sp = torch.zeros(B, dtype=torch.int32, device=self.device)
        x = packed_embeds.to(self.dtype).contiguous().clone()
        return ops.llama_prefill_layers(x, self._layer_array, d.num_hidden_layers, d, self.cos, self.sin, sp, self.cache.page_tables[:B],
                                        PAGE_SIZE, cu_seqlens=cu, max_seqlen=max(seq_lens))

    @ops.in_own_dtype
    def first_tokens(self, hidden_packed: torch.Tensor, seq_lens: List[int], return_logits: bool = False):
        """Greedy first token of every packed sequence: final norm + lm_head over the B last rows as one GEMM
        (bf16 logits, modeling_llama.py:1044-1045), argmax with the lowest index on ties."""
        last = (torch.tensor(seq_lens).cumsum(0) - 1).to(torch.int32).to(self.device)
        rows = ops.splice_rows(hidden_packed, None, None, None, torch.zeros_like(last), last)
        hn = ops.rmsnorm(rows, self.w.norm, self.dims.rms_norm_eps)
        lg = ops.gemm(hn, self.w.lm_head, out=self._logits_buffer(hn.shape[0]))
        ids = ops.argmax_bf16(lg)
        return (ids, lg) if return_logits else ids

    def _logits_buffer(self, rows: int) -> torch.Tensor:
        """bf16 [rows, V] view with a 16-byte-aligned row stride (V = 128259 is odd; the GEMM stores 16-byte vectors)."""
        V = self.dims.vocab_size
        return torch.empty((rows, (V + 7) // 8 * 8), dtype=self.dtype, device=self.device)[:, :V]

    @ops.in_own_dtype
    def logits_all(self, hidden: torch.Tensor) -> torch.Tensor:
        """lm_head over every row -> fp32 logits [S, V] (LlamaForCausalLM.forward semantics, 1044-1045)."""
        hn = ops.rmsnorm(hidden, self.w.norm, self.dims.rms_norm_eps)
        lg = ops.gemm(hn, self.w.lm_head, out=self._logits_buffer(hn.shape[0]))  # bf16 rounding first, then .float()
        return lg.float()

    # ---------------------------------------------------------------------------------------------
    def _decode_step_launch(self, seq: int, logits_out: Optional[torch.Tensor] = None, sample: bool = False) -> None:
        d, w = self.dims, self.w
        if sample and logits_out is None:
            logits_out = self._sample_buffer()
        ops.llama_decode_step(self.h, self._layer_array, d.num_hidden_layers, self.q_buf, self.attn_buf, self.act_buf, d, self.cos,
                              self.sin, self.pos, self.active_pt, PAGE_SIZE, w.norm, w.lm_head, w.embed, self.lm_ws,
                              self.out_ids, self.step, logits_out)
        if sample:  # replaces the greedy id / next embedding row the finalize kernel just wrote (step already advanced)
            ops.sample_top_p(logits_out, self.sample_params, self.sample_seed_dev, self.step, -1, self.out_ids, w.embed, self.h)

    def _sample_buffer(self) -> torch.Tensor:
        if self.sample_logits is None:
            self.sample_logits = torch.empty(self.dims.vocab_size, dtype=torch.float32, device=self.device)
        return self.sample_logits

    def _ensure_graph(self, seq: int, sample: bool = False) -> None:
        if (self._graph_sample if sample else self._graph) is not None:
            return
        # warm up once outside capture (lazy cudaFuncSetAttribute calls etc.), on a side stream
        saved = (self.pos.clone(), self.step.clone(), self.h.clone(), self.out_ids.clone())
        s = torch.cuda.Stream(device=self.device)
        s.wait_stream(torch.cuda.current_stream())  # after the clones are enqueued
        with torch.cuda.stream(s):
            self._decode_step_launch(seq, sample=sample)
        torch.cuda.current_stream().wait_stream(s)
        torch.cuda.synchronize()
        self.pos.copy_(saved[0]); self.step.copy_(saved[1]); self.h.copy_(saved[2]); self.out_ids.copy_(saved[3])
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            self._decode_step_launch(seq, sample=sample)
        if sample:
            self._graph_sample = g
        else:
            self._graph = g

    def _set_sampling(self, sampling) -> bool:
        """sampling = None (greedy) or dict(temperature=, top_p=, top_k=, seed=).  Returns True when tokens are sampled."""
        if not sampling:
            return False
        t = float(sampling.get("temperature") or 1.0)
        p = sampling.get("top_p")
        p = 1.0 if p is None else float(p)
        k = sampling.get("top_k")
        k = 50 if k is None else int(k)  # GenerationConfig's default top_k, applied by HF whenever do_sample=True
        if t <= 0.0 or not (0.0 < p <= 1.0) or k < 0:
            raise ValueError(f"sampling needs temperature > 0, 0 < top_p <= 1 and top_k >= 0, got temperature={t}, top_p={p}, top_k={k}")
        self.sample_params.copy_(torch.tensor([t, p, float(k)], dtype=torch.float32))
        seed = sampling.get("seed")
        self._set_seed(int(torch.initial_seed() if seed is None else seed))
        return True

    def _set_seed(self, seed: int) -> None:
        self.sample_seed = seed & 0x7FFFFFFFFFFFFFFF
        self.sample_seed_dev.copy_(torch.tensor([self.sample_seed], dtype=torch.int64))

    @torch.no_grad()
    @ops.in_own_dtype
    def generate_from_embeds(self, inputs_embeds: torch.Tensor, max_new_tokens: int, eos_token_ids=None, stopping_fn=None,
                             use_graph: bool = True, return_logits: bool = False, seq: int = 0, sampling=None, prefix_len: int = 0):
        """Greedy (or, with ``sampling=dict(temperature, top_p, seed)``, nucleus-sampled) decoding started from prompt
        embeddings [S, H].  Returns LongTensor [n_new] (and fp32 logits [n_new, V] when return_logits).
        ``stopping_fn(ids_so_far: LongTensor) -> bool``.

        ``prefix_len`` = L > 0 continues what sequence `seq` already caches: its pages for positions [0, L) are kept (the caller
        has checked that they hold exactly inputs_embeds[:L]) and only rows [L, S) are prefilled, at position L.  L = 0 releases
        every cached sequence first.  After S prompt rows and n returned tokens the cache holds the final KV of positions
        [0, S + n - 1): see cached_length()."""
        d, w = self.dims, self.w
        S = inputs_embeds.shape[0]
        if max_new_tokens < 1:
            return torch.empty(0, dtype=torch.int64, device=self.device)
        if max_new_tokens > self.out_ids.numel():
            raise RuntimeError(f"max_new_tokens {max_new_tokens} exceeds the decoder's cap {self.out_ids.numel()}")
        if S + max_new_tokens > self.max_seq_len:
            raise RuntimeError(f"{S} prompt + {max_new_tokens} new tokens exceed max_seq_len {self.max_seq_len}")
        eos = set()
        if eos_token_ids is not None:
            eos = set(int(e) for e in (eos_token_ids if isinstance(eos_token_ids, (list, tuple, set)) else [eos_token_ids]))
        if not 0 <= prefix_len < S:
            raise ValueError(f"prefix_len {prefix_len} must lie in [0, {S}): at least one prompt row is prefilled")
        if prefix_len == 0:
            self.release_all()  # a previous batched generate leaves pages owned by sequences 1..B-1
        else:
            for b in range(len(self.cache.owned)):
                if b != seq:
                    self.cache.release(b)
        self.cache.reserve(seq, S + max_new_tokens)
        hidden = self.prefill_hidden(inputs_embeds[prefix_len:], seq, prefix_len)
        logits = torch.empty((max_new_tokens, d.vocab_size), dtype=torch.float32, device=self.device) if return_logits else None
        # first token: final norm + lm_head + argmax on the last prompt row; afterwards pos == S
        self.pos.fill_(S - 1)
        self.step.zero_()
        sample = self._set_sampling(sampling)
        first_logits = logits[0] if logits is not None else (self._sample_buffer() if sample else None)
        ops.lm_head_argmax(hidden[S - 1 - prefix_len], w.lm_head, w.norm, d.rms_norm_eps, self.lm_ws, self.out_ids, self.step, self.pos,
                           embed_table=w.embed, next_x=self.h, logits_out=first_logits)
        if sample:
            ops.sample_top_p(first_logits, self.sample_params, self.sample_seed_dev, self.step, -1, self.out_ids, w.embed, self.h)
        return self._decode_loop(seq, 1, max_new_tokens, eos, stopping_fn, use_graph, logits, sample)

    @staticmethod
    def cached_length(prompt_len: int, n_new: int) -> int:
        """Positions whose KV is final after generate_from_embeds returned n_new >= 1 tokens for a prompt of prompt_len rows.
        Decode step k (k = 1..n_new-1, _decode_loop) feeds token k-1 at position prompt_len + k - 1, so positions
        [0, prompt_len + n_new - 1) are written by the prompt and the kept steps; the last returned token was never fed.  On an
        EOS / stopping-criteria stop the loop may have run ONE speculative step past the stop, which wrote slot
        prompt_len + n_new - 1 only; that slot is outside the cached length, and the next prefill overwrites it."""
        return prompt_len + n_new - 1 if n_new > 0 else prompt_len

    def _decode_loop(self, seq: int, n: int, max_new_tokens: int, eos, stopping_fn, use_graph: bool, logits, sample: bool = False):
        """Steps n..max_new_tokens-1 of sequence `seq` (greedy, or sampled); pos / step / h / out_ids[:n] are already set."""
        self.active_pt.copy_(self.cache.page_tables[seq])
        need_host_check = bool(eos) or stopping_fn is not None
        return_logits = logits is not None
        graph = None
        if use_graph and not return_logits:
            self._ensure_graph(seq, sample)
            graph = self._graph_sample if sample else self._graph

        def launch_step(k: int) -> None:
            if graph is not None:
                graph.replay()
                ops.LAUNCHES += self.kernels_per_decode_step + (1 if sample else 0)
            else:
                self._decode_step_launch(seq, None if logits is None else logits[k], sample)

        if not need_host_check:
            while n < max_new_tokens:
                launch_step(n)
                n += 1
        else:
            # EOS / stopping criteria (the mode eval_spatial.py:223-237 runs) WITHOUT a host round trip per token: the step that
            # produces token n is enqueued BEFORE token n-1 is inspected, token ids reach the host through a side stream into
            # pinned memory, and the host inspects token n-1 while the GPU computes token n.  On a stop the one speculative
            # step is discarded (it only touched this sequence's own KV slot and the step counters, which the next request
            # resets).  HF inspects after every token too (a blocking .item()); the result is identical.
            if getattr(self, "_host_ids", None) is None:
                self._host_ids = torch.empty(self.out_ids.numel(), dtype=torch.int64, pin_memory=True)
                self._copy_stream = torch.cuda.Stream(device=self.device)
            host, side = self._host_ids, self._copy_stream
            done = {}

            def fetch(lo: int, hi: int) -> None:  # tokens [lo, hi) -> host, ordered after the work enqueued so far
                e = torch.cuda.Event()
                e.record()
                side.wait_event(e)
                with torch.cuda.stream(side):
                    host[lo:hi].copy_(self.out_ids[lo:hi], non_blocking=True)
                    d = torch.cuda.Event()
                    d.record(side)
                for k in range(lo, hi):
                    done[k] = d

            fetch(0, n)
            checked = 0
            while True:
                launched = n < max_new_tokens
                if launched:
                    launch_step(n)
                    fetch(n, n + 1)
                else:
                    break  # the token budget is spent: the last token is returned whatever it is (HF semantics)
                stop_len = None
                for k in range(checked, n):
                    done.pop(k).synchronize()
                    if int(host[k]) in eos or (stopping_fn is not None and stopping_fn(host[:k + 1])):
                        stop_len = k + 1
                        break
                checked = n
                if stop_len is not None:
                    n = stop_len
                    break
                n += 1
        out = self.out_ids[:n].clone()
        if return_logits:
            return out, logits[:n]
        return out

    # ---- batched decode: B sequences advance one token per step, every weight streamed ONCE for the whole batch ----------------
    def _batch_state(self, B: int):
        st = getattr(self, "_bstate", None)
        if st is not None and st["B"] == B and st["cache"] is self.cache:
            return st
        d, dev = self.dims, self.device
        H, nh, nkv, hd, I, V = d.hidden_size, d.num_attention_heads, d.num_key_value_heads, d.head_dim, d.intermediate_size, d.vocab_size
        z = lambda *shape, dtype=self.dtype: torch.zeros(shape, dtype=dtype, device=dev)  # noqa: E731
        st = dict(B=B, cache=self.cache, graph=None, h=z(B, H), xn=z(B, H), qkv=z(B, (nh + 2 * nkv) * hd), attn=z(B, nh * hd), act=z(B, I),
                  logits=z(B, (V + 7) // 8 * 8), pos=z(B, dtype=torch.int32), step=z(1, dtype=torch.int32), ids=z(B, dtype=torch.int64),
                  out=z(self.out_ids.numel() * B, dtype=torch.int64), ticket=z(1, dtype=torch.int32),
                  cu=torch.arange(B + 1, dtype=torch.int32, device=dev))
        self._bstate = st
        return st

    def _batch_step_launch(self, st, logits_only: bool = False) -> None:
        """One decode step of all B sequences (llava_arch.py:549-611 + modeling_llama.py:540-562 semantics without padding): the
        projections are tcgen05 GEMMs over the B rows (tall stream-K configuration), RoPE / KV append and attention per sequence."""
        d, w, B = self.dims, self.w, st["B"]
        nh, nkv, hd, V = d.num_attention_heads, d.num_key_value_heads, d.head_dim, d.vocab_size
        qd = nh * hd
        h, xn, qkv, attn, act = st["h"], st["xn"], st["qkv"], st["attn"], st["act"]
        pts = self.cache.page_tables
        for l, lw in enumerate(w.layers):
            pages = self.cache.layer(l)
            ops.rmsnorm(h, lw.in_norm, d.rms_norm_eps, out=xn)
            ops.gemm(xn, lw.qkv_w, out=qkv)
            ops.rope_kv_append_varlen(qkv, nh, nkv, hd, self.cos, self.sin, st["pos"], pages, pts, PAGE_SIZE, st["cu"])
            ops.attention_decode_batched(qkv[:, :qd], attn, pages, pts, PAGE_SIZE, st["pos"], nh, nkv, hd, self.scale)
            ops.gemm(attn, lw.o_w, residual=h, epilogue=ops.EPI_BIAS_RESIDUAL, out=h)
            ops.rmsnorm(h, lw.post_norm, d.rms_norm_eps, out=xn)
            ops.gemm(xn, lw.gateup_w, epilogue=ops.EPI_SWIGLU, out=act)
            ops.gemm(act, lw.down_w, residual=h, epilogue=ops.EPI_BIAS_RESIDUAL, out=h)
        ops.rmsnorm(h, w.norm, d.rms_norm_eps, out=xn)
        lg = st["logits"][:, :V]
        ops.gemm(xn, w.lm_head, out=lg)  # bf16 logits (modeling_llama.py:1044), arg max with the lowest index on ties
        if logits_only:  # beam search: the host picks the next tokens from the candidates of these logits
            return
        ops.argmax_bf16(lg, out=st["ids"])
        ops.decode_batch_advance(st["ids"], w.embed, h, st["out"], st["step"], st["pos"], st["ticket"])

    def _decode_batched(self, first: torch.Tensor, seq_lens: List[int], max_new_tokens: int, eos, stopping_fn, use_graph: bool):
        """Greedy decode of B prefilled sequences together.  Returns a list of LongTensor [n_b] (each cut at its own stop)."""
        B = len(seq_lens)
        st = self._batch_state(B)
        zero = torch.zeros(B, dtype=torch.int32, device=self.device)
        st["out"][:B].copy_(first)
        st["h"].copy_(ops.splice_rows(self.w.embed, None, None, None, zero, first.to(torch.int32)))
        st["pos"].copy_(torch.tensor(seq_lens, dtype=torch.int32))
        st["step"].fill_(1)
        if use_graph and st["graph"] is None:
            saved = {k: st[k].clone() for k in ("h", "pos", "step", "out")}
            s = torch.cuda.Stream(device=self.device)
            s.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(s):
                self._batch_step_launch(st)  # warm-up outside capture (lazy kernel attribute setup)
            torch.cuda.current_stream().wait_stream(s)
            torch.cuda.synchronize()
            for k, v in saved.items():
                st[k].copy_(v)
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                self._batch_step_launch(st)
            st["graph"] = g
        kernels = 8 * self.dims.num_hidden_layers + 4
        need_check = bool(eos) or stopping_fn is not None
        host = torch.empty((max_new_tokens, B), dtype=torch.int64, pin_memory=True) if need_check else None
        side = getattr(self, "_copy_stream", None) or torch.cuda.Stream(device=self.device)
        self._copy_stream = side
        out2d = st["out"][: max_new_tokens * B].view(max_new_tokens, B)
        stopped = [None] * B  # length at which sequence b stopped
        done = {}

        def fetch(k: int) -> None:
            e = torch.cuda.Event()
            e.record()
            side.wait_event(e)
            with torch.cuda.stream(side):
                host[k].copy_(out2d[k], non_blocking=True)
                dn = torch.cuda.Event()
                dn.record(side)
            done[k] = dn

        n = 1
        if need_check:
            fetch(0)
        checked = 0
        while n < max_new_tokens:
            if use_graph:
                st["graph"].replay()
                ops.LAUNCHES += kernels
            else:
                self._batch_step_launch(st)
            if need_check:  # same pipelining as the single-sequence loop: inspect row n-1 while row n is being computed
                fetch(n)
                for k in range(checked, n):
                    done.pop(k).synchronize()
                    for b in range(B):
                        if stopped[b] is None and (int(host[k, b]) in eos or (stopping_fn is not None and stopping_fn(host[:k + 1, b]))):
                            stopped[b] = k + 1
                checked = n
                if all(s is not None for s in stopped):
                    break
            n += 1
        n = min(n, max_new_tokens)
        res = out2d[:n].t().contiguous()
        return [res[b, : (stopped[b] if stopped[b] is not None else n)].clone() for b in range(B)]

    @torch.no_grad()
    @ops.in_own_dtype
    def generate_beam(self, inputs_embeds: torch.Tensor, num_beams: int, max_new_tokens: int, eos_token_ids=None, stopping_fn=None,
                      length_penalty: float = 1.0, early_stopping: bool = False, use_graph: bool = True) -> torch.Tensor:
        """Beam search from prompt embeddings [S, H] (HF GenerationMixin.beam_search + BeamSearchScorer behind llava_llama.py:212 when
        the eval scripts pass --num_beams > 1; restated by the CPU checker of the test suite (beam_search_generate), which is pinned to HF's own
        generate()).  Device side: the prompt is prefilled once per beam as one packed batch (HF expands the inputs the same way), every
        step runs the batched decode layers over the num_beams rows, a kernel reduces each row's logits to its 2 x num_beams best
        (log-prob + beam score, token) pairs, and the surviving beams' KV rows are re-ordered page-wise.  Host side: the hypothesis
        bookkeeping on the num_beams x 2 num_beams candidates - the same control logic HF runs in Python.  Returns the NEW ids."""
        d, w, k = self.dims, self.w, int(num_beams)
        S, V = inputs_embeds.shape[0], d.vocab_size
        if k < 2:
            raise ValueError("generate_beam needs num_beams >= 2")
        if max_new_tokens < 1:
            return torch.empty(0, dtype=torch.int64, device=self.device)
        if S + max_new_tokens > self.max_seq_len:
            raise RuntimeError(f"{S} prompt + {max_new_tokens} new tokens exceed max_seq_len {self.max_seq_len}")
        eos = []
        if eos_token_ids is not None:
            eos = [int(e) for e in (eos_token_ids if isinstance(eos_token_ids, (list, tuple, set)) else [eos_token_ids])]
        n_cand = max(2, 1 + len(eos)) * k
        self.release_all()
        self.ensure_capacity(k, S + max_new_tokens)
        self.cache.reserve_many([S + max_new_tokens] * k)
        hidden = self.prefill_packed(inputs_embeds.to(self.dtype).repeat(k, 1), [S] * k)
        _, lg = self.first_tokens(hidden, [S] * k, return_logits=True)
        st = self._batch_state(k)
        st["logits"][:, :V].copy_(lg)
        dev = self.device
        beam_scores = torch.full((k,), -1e9, dtype=torch.float32)
        beam_scores[0] = 0.0
        d_scores = beam_scores.to(dev)
        cand_s = torch.empty((k, n_cand), dtype=torch.float32, device=dev)
        cand_t = torch.empty((k, n_cand), dtype=torch.int32, device=dev)
        h_s = torch.empty((k, n_cand), dtype=torch.float32, pin_memory=True)
        h_t = torch.empty((k, n_cand), dtype=torch.int32, pin_memory=True)
        seqs: List[List[int]] = [[] for _ in range(k)]
        hyps: List = []  # (score, tokens) of finished hypotheses, at most k kept
        worst, done = 1e9, False
        zero = torch.zeros(k, dtype=torch.int32, device=dev)
        tables = [list(self.cache.owned[b]) for b in range(k)]  # page ids by position // PAGE_SIZE
        pages_all = self.cache.pages
        graph = st.get("beam_graph") if use_graph else None

        def keep(score: float, toks: List[int]) -> None:
            nonlocal worst
            if len(hyps) < k or score > worst:
                hyps.append((score, toks))
                if len(hyps) > k:
                    hyps.remove(min(hyps, key=lambda x: x[0]))
                worst = min(x[0] for x in hyps)

        for step in range(max_new_tokens):
            ops.beam_candidates(st["logits"][:, :V], d_scores, cand_s, cand_t)
            h_s.copy_(cand_s, non_blocking=True)
            h_t.copy_(cand_t, non_blocking=True)
            torch.cuda.current_stream().synchronize()
            # merge the per-beam candidates: (score desc, beam asc, token asc) = the flat-index order of HF's topk on ties
            flat = sorted(((-float(h_s[b, j]), b, int(h_t[b, j])) for b in range(k) for j in range(n_cand) if int(h_t[b, j]) >= 0))[:n_cand]
            cur_len = step + 1
            nxt = []
            for rank, (neg, b, t) in enumerate(flat):
                sc = -neg
                if t in eos:
                    if rank >= k:
                        continue
                    keep(sc / (cur_len ** length_penalty), list(seqs[b]))
                else:
                    nxt.append((sc, b, t))
                if len(nxt) == k:
                    break
            if len(nxt) < k:
                raise RuntimeError("beam search ran out of non-EOS candidates")  # HF asserts the same
            if len(hyps) >= k and (early_stopping or worst >= (-flat[0][0]) / (cur_len ** length_penalty)):
                done = True
            seqs = [seqs[b] + [t] for _, b, t in nxt]
            beam_scores = torch.tensor([sc for sc, _, _ in nxt], dtype=torch.float32)
            if done or step == max_new_tokens - 1:
                break
            if stopping_fn is not None and all(stopping_fn(torch.tensor(q, dtype=torch.int64)) for q in seqs):
                break  # KeywordsStoppingCriteria.__call__ requires every row (beam) to have hit (mm_utils.py:616-617)
            # ---- device state of the next step: KV rows of the generated region follow their parents (HF _reorder_cache,
            #      modeling_llama.py:1151-1158, copies the WHOLE cache; here only the pages that hold generated tokens)
            parents = [b for _, b, _ in nxt]
            if step > 0 and any(p != i for i, p in enumerate(parents)):
                j0, j1 = S // PAGE_SIZE, (S + step - 1) // PAGE_SIZE
                src = [tables[p][j] for i, p in enumerate(parents) if p != i for j in range(j0, j1 + 1)]
                dst = [tables[i][j] for i, p in enumerate(parents) if p != i for j in range(j0, j1 + 1)]
                src_t = torch.tensor(src, dtype=torch.int64).to(dev)
                dst_t = torch.tensor(dst, dtype=torch.int64).to(dev)
                pages_all[:, dst_t] = pages_all[:, src_t]  # gather into a temporary, then scatter: permutations are safe
            ids = torch.tensor([t for _, _, t in nxt], dtype=torch.int32).to(dev)
            st["h"].copy_(ops.splice_rows(w.embed, None, None, None, zero, ids))
            st["pos"].fill_(S + step)
            d_scores.copy_(beam_scores, non_blocking=True)
            if use_graph and graph is None:
                saved = st["h"].clone()
                self._batch_step_launch(st, logits_only=True)  # warm-up outside capture; rewrites only this step's own KV rows
                torch.cuda.synchronize()
                st["h"].copy_(saved)
                graph = torch.cuda.CUDAGraph()
                with torch.cuda.graph(graph):
                    self._batch_step_launch(st, logits_only=True)
                st["beam_graph"] = graph
            if graph is not None:
                graph.replay()
                ops.LAUNCHES += 8 * d.num_hidden_layers + 2
            else:
                self._batch_step_launch(st, logits_only=True)
        if not done:  # finalize (beam_search.py): the running beams become hypotheses over their generated length
            for i in range(k):
                keep(float(beam_scores[i]) / (len(seqs[i]) ** length_penalty), list(seqs[i]))
        best = list(max(hyps, key=lambda x: x[0])[1])
        if len(best) < max_new_tokens and eos:
            best.append(eos[0])
        return torch.tensor(best, dtype=torch.int64, device=dev)

    @torch.no_grad()
    @ops.in_own_dtype
    def generate_batch(self, packed_embeds: torch.Tensor, seq_lens: List[int], max_new_tokens: int, eos_token_ids=None,
                       stopping_fn=None, use_graph: bool = True, return_logits: bool = False, sampling=None):
        """Decoding of B prompts: ONE packed prefill pass (tensor-core bound, all prompts share every GEMM), one lm_head GEMM for the
        B first tokens, then BATCHED decode: every step advances all B sequences, each weight streamed once per step for the
        whole batch (_decode_batched).  With ``return_logits`` or sampling the sequences are decoded one after the other with the
        single-sequence weight-streaming step.  Returns a list of LongTensor [n_b] (and a list of fp32 logits)."""
        d, w = self.dims, self.w
        B = len(seq_lens)
        if max_new_tokens < 1:
            return [torch.empty(0, dtype=torch.int64, device=self.device) for _ in range(B)]
        if max_new_tokens > self.out_ids.numel():
            raise RuntimeError(f"max_new_tokens {max_new_tokens} exceeds the decoder's cap {self.out_ids.numel()}")
        if max(seq_lens) + max_new_tokens > self.max_seq_len:
            raise RuntimeError(f"{max(seq_lens)} prompt + {max_new_tokens} new tokens exceed max_seq_len {self.max_seq_len}")
        eos = set()
        if eos_token_ids is not None:
            eos = set(int(e) for e in (eos_token_ids if isinstance(eos_token_ids, (list, tuple, set)) else [eos_token_ids]))
        self.release_all()
        self.ensure_capacity(B, max(seq_lens) + max_new_tokens)
        self.cache.reserve_many([n + max_new_tokens for n in seq_lens])
        hidden = self.prefill_packed(packed_embeds, seq_lens)
        first, lg = self.first_tokens(hidden, seq_lens, return_logits=True)
        outs, all_logits = [], []
        sample = self._set_sampling(sampling)
        if max_new_tokens == 1 and not return_logits and not sample:
            return [first[b:b + 1] for b in range(B)]
        if not return_logits and not sample and B > 1:
            return self._decode_batched(first, seq_lens, max_new_tokens, eos, stopping_fn, use_graph)
        zero = torch.zeros(1, dtype=torch.int32, device=self.device)
        for b in range(B):
            logits = None
            if return_logits:
                logits = torch.empty((max_new_tokens, d.vocab_size), dtype=torch.float32, device=self.device)
                logits[0].copy_(lg[b])
            # decode state of sequence b: token 0 is known, the next step processes it at position S_b
            self.out_ids[0:1].copy_(first[b:b + 1])
            self.h.copy_(ops.splice_rows(w.embed, None, None, None, zero, first[b:b + 1].to(torch.int32))[0])
            self.pos.fill_(seq_lens[b])
            self.step.fill_(1)
            if sample:  # re-draw the first token of this sequence from its logits row (a different draw per sequence: the seed moves)
                self._set_seed(self.sample_seed + 0x9E3779B97F4A7C15 * (b + 1))
                ops.sample_top_p(lg[b].float().contiguous(), self.sample_params, self.sample_seed_dev, self.step, -1, self.out_ids, w.embed, self.h)
            r = self._decode_loop(b, 1, max_new_tokens, eos, stopping_fn, use_graph, logits, sample)
            if return_logits:
                outs.append(r[0]); all_logits.append(r[1])
            else:
                outs.append(r)
        return (outs, all_logits) if return_logits else outs
