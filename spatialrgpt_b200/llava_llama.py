"""``LlavaLlamaModel`` — the reference's VLM class (llava/model/language_model/llava_llama.py:48-213
+ llava/model/llava_arch.py:252-650) re-built over the sm_100a kernels, keeping its public surface:
``generate(input_ids, images=, depths=, masks=, attention_mask=, **generation_kwargs)``, ``forward``,
``prepare_inputs_labels_for_multimodal``, ``encode_images``, the ``get_*`` accessors, ``config``,
``tokenizer``, ``device`` / ``dtype``.  ``past_key_values=`` takes a ``PagedKVCacheHandle`` (kv_handle.py): the KV of a
previous call stays in the paged cache and only the new rows are prefilled.  ``LlavaLlamaForCausalLM`` is an alias (the name the north
star and llava/model/builder.py:138 use; the reference never defines it)."""
from __future__ import annotations

from dataclasses import dataclass
from typing import Any, List, Optional, Sequence, Tuple, Union

import torch

from . import ops
from .config import LlavaConfig
from .constants import IGNORE_INDEX, IMAGE_TOKEN_INDEX
from .kv_handle import PagedKVCacheHandle, reusable_prefix
from .llama_decoder import LlamaDecoder
from .multimodal_encoder import VisionTower
from .multimodal_projector import MultimodalProjector
from .region_extractor import RegionExtractor
from .splice_plan import build_splice_plan
from .weights import ModelWeights


@dataclass
class CausalLMOutputWithPast:
    logits: torch.Tensor
    loss: Optional[torch.Tensor] = None
    past_key_values: Any = None
    hidden_states: Any = None
    attentions: Any = None


class LlavaLlamaModel:
    config_class = LlavaConfig
    main_input_name = "input_embeds"

    def __init__(self, config: LlavaConfig, weights: ModelWeights, tokenizer=None, image_processor=None,
                 max_seq_len: int = 4096, tensor_parallel=None):
        """``tensor_parallel`` = None, or (rank, world[, process_group]): the Llama DECODE step is sharded over `world` ranks
        (tensor_parallel.py, BASELINE config c5); encoders and the prompt prefill stay replicated."""
        # fail loudly when the CUDA extension or a B200 is missing: there is no CPU path
        from . import _lib
        self.config = config
        self.weights = weights
        if self.dtype not in (torch.bfloat16, torch.float16):
            raise _lib.SrgptError(f"weights are {self.dtype}: the kernels compute in torch.bfloat16 or torch.float16")
        with ops.elem_dtype(self.dtype):
            _lib.load()
            if not torch.cuda.is_available():
                raise _lib.SrgptError("spatialrgpt_b200 needs a CUDA device (sm_100a); no CPU fallback exists")
            _lib.device_info()
        self.tokenizer = tokenizer
        self._image_processor = image_processor
        self._max_seq_len = max_seq_len
        self._tensor_parallel = tensor_parallel
        self.training = False
        config.model_dtype = str(self.dtype)
        self._build_modules()

    @ops.in_own_dtype
    def _build_modules(self) -> None:
        config, weights, image_processor, max_seq_len, tensor_parallel = (self.config, self.weights, self._image_processor, self._max_seq_len,
                                                                          self._tensor_parallel)
        self.vision_tower = VisionTower(config, weights.vision, image_processor)
        self.mm_projector = MultimodalProjector(config, weights.projector)
        self.region_extractor = RegionExtractor(config, weights.region) if (config.enable_region and weights.region is not None) else None
        if tensor_parallel is not None and int(tensor_parallel[1]) > 1:
            from .tensor_parallel import TPLlamaDecoder
            self.llm = TPLlamaDecoder(config.llama, weights.llama, int(tensor_parallel[0]), int(tensor_parallel[1]),
                                      group=tensor_parallel[2] if len(tensor_parallel) > 2 else None, max_seq_len=max_seq_len)
        else:
            self.llm = LlamaDecoder(config.llama, weights.llama, max_seq_len=max_seq_len)

    # ---- accessors (llava_arch.py:252-278) -----------------------------------------------------------
    def get_llm(self):
        return self.llm

    def get_lm_head(self):
        return self.weights.llama.lm_head

    def get_vision_tower(self):
        return self.vision_tower

    def get_mm_projector(self):
        return self.mm_projector

    def get_region_extractor(self):
        return self.region_extractor

    def get_input_embeddings(self):
        return self.llm.embed_tokens

    @property
    def device(self):
        return self.weights.llama.embed.device

    @property
    def dtype(self):
        """torch.bfloat16 or torch.float16 - the dtype of the weights, which is also the compute dtype (the matching build of the
        kernels is selected around every public call, ops.elem_dtype)."""
        return self.weights.dtype

    def eval(self):
        return self

    def cuda(self, *a, **k):
        return self

    def to(self, *a, **k):
        dt = k.get("dtype", None)
        for x in a:
            if isinstance(x, torch.dtype):
                dt = x
        if dt is not None and dt != self.dtype:
            # nn.Module.to(dtype): cast the weights and rebuild what is derived from them (rope tables, KV cache, decode graphs).
            # The reference's eval does exactly this after an fp16 load: model.to(dtype=torch.bfloat16) (eval_spatial.py:221).
            if dt not in (torch.bfloat16, torch.float16):
                raise NotImplementedError(f"the sm_100a path computes in torch.bfloat16 or torch.float16, not {dt}")
            self.weights.to(dt)
            self.config.model_dtype = str(dt)
            self._build_modules()
        return self

    # ---- encoders ---------------------------------------------------------------------------------
    @ops.in_own_dtype
    def encode_images(self, images: torch.Tensor) -> torch.Tensor:
        """llava_arch.py:307-310 (tower -> projector, no regions)."""
        return self.mm_projector(self.vision_tower(images))

    def _start_host_copies(self, tensors):
        """Device tensors -> pinned host copies on a side stream (None entries pass through).  Returns (host tensors, event):
        the caller synchronises the event, not the compute stream."""
        out, any_dev = [], False
        side = getattr(self, "_side_stream", None)
        for t in tensors:
            if t is None or not t.is_cuda:
                out.append(None if t is None else t.detach())
                continue
            if side is None:
                side = self._side_stream = torch.cuda.Stream(device=self.device)
            if not any_dev:
                side.wait_stream(torch.cuda.current_stream())
                any_dev = True
            with torch.cuda.stream(side):
                h = torch.empty(t.shape, dtype=t.dtype, pin_memory=True)
                h.copy_(t.detach(), non_blocking=True)
            out.append(h)
        if not any_dev:
            return out, None
        ev = torch.cuda.Event()
        ev.record(side)
        return out, ev

    def _tokens_per_image(self) -> int:
        """Rows one <image> slot expands to: the projector's 2x2 down-sampling of the 27x27 refined map (regions on) or of the
        tower grid (base_projector.py:32-52)."""
        from .region_extractor import ADA_POOL
        side = ADA_POOL if (self.config.enable_region and self.region_extractor is not None) else self.config.vision.grid
        return self.mm_projector.tokens_out(side)

    def _encode_multimodal(self, images, masks, depths):
        """llava_arch.py:387-411.  Returns (image_features [N,196,H], mask_embeds, depth_embeds)."""
        cfg = self.config
        if isinstance(images, (list, tuple)):
            images = torch.cat([im if im.dim() == 4 else im[None] for im in images], dim=0)
        elif images.dim() == 5:
            images = images.flatten(0, 1)
        if depths is not None:
            if isinstance(depths, (list, tuple)):
                depths = torch.cat([d if d.dim() == 4 else d[None] for d in depths], dim=0)
            elif depths.dim() == 5:
                depths = depths.flatten(0, 1)
        N = images.shape[0]
        mask_embeds = depth_embeds = None
        use_depth = cfg.enable_region and cfg.enable_depth and depths is not None
        if cfg.enable_region and self.region_extractor is not None and masks is not None:
            # the mask -> pooling-weight kernels need only the masks: side stream, under the tower passes launched next
            g = cfg.vision.grid
            self.region_extractor.mask_pooling.precompute(masks, N, [(4 * g, ops.ORDER_NESTED)] + ([(g, ops.ORDER_ROWMAJOR)] if use_depth else []),
                                                          self.device)
        if use_depth and depths.shape == images.shape:
            # one tower pass over [images; depths] (same weights, llava_arch.py:398,404): twice the GEMM M
            both = self.vision_tower(torch.cat([images.to(self.device), depths.to(self.device).to(images.dtype)], dim=0))
            tower_features, depth_features = both[:N], both[N:]
        else:
            tower_features = self.vision_tower(images)
            depth_features = self.vision_tower(depths) if use_depth else None
        if cfg.enable_region and self.region_extractor is not None:
            hres, lres = self.region_extractor.feature_refinement_nested(tower_features.contiguous())
            mask_embeds, depth_embeds = self.region_extractor(hres, None if depth_features is None else depth_features.contiguous(),
                                                              masks, hres_order=ops.ORDER_NESTED)
        else:
            lres = tower_features
        image_features = self.mm_projector(lres)
        return image_features, mask_embeds, depth_embeds

    # ---- embedding splice (llava_arch.py:333-650) -----------------------------------------------------
    @ops.in_own_dtype
    def prepare_inputs_labels_for_multimodal(self, input_ids, position_ids, attention_mask, past_key_values, labels, images,
                                             masks=None, depths=None, _packed_only: bool = False):
        if images is None or (input_ids is not None and input_ids.shape[1] == 1):
            return input_ids, position_ids, attention_mask, past_key_values, None, labels  # llava_arch.py:355-385
        cfg = self.config
        dev = self.device
        # The splice plan needs only host-side facts (token ids, images / regions per request).  Order of events: (1) the ids
        # (and masks / labels) start their device->host copy on a side stream, (2) the encoders are launched, (3) the host
        # builds the plan while the GPU runs the tower, (4) plan upload + one gather kernel.  The host never waits on the tower
        # and the GPU never waits on the Python loop below (it cost ~15 % of a 32-request batch when it came in between).
        host_copies, copy_done = self._start_host_copies([input_ids, attention_mask, labels])
        encoded = self._encode_multimodal(images, masks, depths)
        if copy_done is not None:
            copy_done.synchronize()
        ids_cpu = host_copies[0].to(torch.int64)
        B, T = ids_cpu.shape
        am_cpu = torch.ones((B, T), dtype=torch.bool) if attention_mask is None else host_copies[1].bool()
        lab_cpu = torch.full((B, T), IGNORE_INDEX, dtype=torch.int64) if labels is None else host_copies[2].to(torch.int64)
        if isinstance(images, (list, tuple)):
            n_img = sum(im.shape[0] if im.dim() == 4 else 1 for im in images)
        else:
            n_img = images.shape[0] * images.shape[1] if images.dim() == 5 else images.shape[0]
        n_tok = self._tokens_per_image()
        region_on = cfg.enable_region and self.region_extractor is not None
        depth_on = region_on and cfg.enable_depth and depths is not None
        mask_list = (list(masks) if masks is not None else []) + [None] * n_img
        plan = build_splice_plan(ids_cpu, None if attention_mask is None else am_cpu, None if labels is None else lab_cpu, n_tok,
                                 [0 if m is None else int(m.shape[0]) for m in mask_list[:n_img]], [m is not None for m in mask_list[:n_img]],
                                 cfg.llm_mask_token_id, cfg.llm_depth_token_id, region_on, depth_on,
                                 getattr(cfg.llama, "tokenizer_model_max_length", None), vocab_size=self.weights.llama.embed.shape[0])
        for w in plan.warnings:
            print(w)
        lens, new_labels = plan.lens, plan.labels
        sid_dev, srow_dev = plan.src_id.to(dev, non_blocking=True), plan.src_row.to(dev, non_blocking=True)

        # ---- ONE gather kernel builds the embeddings of the whole batch from the encoder outputs
        image_features, mask_embeds, depth_embeds = encoded
        if tuple(image_features.shape[:2]) != (n_img, n_tok):
            raise RuntimeError(f"splice plan expected {(n_img, n_tok)} image tokens, encoders produced {tuple(image_features.shape[:2])}")
        H = image_features.shape[2]

        def cat_rows(embeds):
            parts = [] if embeds is None else [e for e in embeds if e is not None]
            return torch.cat(parts, 0).contiguous() if parts else None

        mflat, dflat = cat_rows(mask_embeds), cat_rows(depth_embeds)
        img_flat = image_features.reshape(n_img * n_tok, H)
        packed = ops.splice_rows(self.weights.llama.embed, img_flat, mflat if mflat is not None else img_flat,
                                 dflat if dflat is not None else img_flat, sid_dev, srow_dev)
        self._last_packed = (packed, lens)
        self._last_seq_lens = lens
        if _packed_only:  # generate(): the unpadded rows are what the decoder consumes (no [B, max_len, H] copy)
            return None, None, attention_mask, past_key_values, None, None
        new_embeds = list(torch.split(packed, lens, 0))

        max_len = max(x.shape[0] for x in new_embeds)
        left = getattr(cfg.llama, "tokenizer_padding_side", "right") == "left"
        out = torch.zeros((B, max_len, H), dtype=self.dtype, device=dev)
        lab_out = torch.full((B, max_len), IGNORE_INDEX, dtype=torch.int64)
        am_out = torch.zeros((B, max_len), dtype=torch.bool)
        pos_out = torch.zeros((B, max_len), dtype=torch.int64)
        for b, (e, l) in enumerate(zip(new_embeds, new_labels)):
            n = e.shape[0]
            sl = slice(max_len - n, max_len) if left else slice(0, n)
            out[b, sl] = e
            lab_out[b, sl] = l
            am_out[b, sl] = True
            pos_out[b, sl] = torch.arange(n)
        ret_labels = None if labels is None else lab_out.to(dev)
        ret_am = None if attention_mask is None else am_out.to(device=dev, dtype=attention_mask.dtype)
        ret_pos = None if position_ids is None else pos_out.to(dev)
        self._last_seq_lens = [x.shape[0] for x in new_embeds]
        return None, ret_pos, ret_am, past_key_values, out, ret_labels

    # ---- KV handles (past_key_values) ------------------------------------------------------------------
    def _check_handle(self, handle, batch: int, num_beams: int = 1) -> None:
        if not isinstance(handle, PagedKVCacheHandle):
            raise NotImplementedError("past_key_values must be a PagedKVCacheHandle; HF tensor caches (DynamicCache / legacy tuples) are "
                                      "not imported, the KV cache is paged and internal")
        if batch != 1:
            raise NotImplementedError("past_key_values is supported for batch 1 only")
        if num_beams != 1:
            raise NotImplementedError("past_key_values is not supported with beam search (num_beams > 1)")
        if type(self.llm).__name__ == "TPLlamaDecoder":
            raise NotImplementedError("past_key_values is not supported on the tensor-parallel decoder")

    def _forward_continue(self, input_ids, inputs_embeds, attention_mask, handle: PagedKVCacheHandle) -> CausalLMOutputWithPast:
        """Incremental forward (modeling_llama.py:451-456 + 564-566): the new rows are appended at handle.length and attend to
        everything the handle's sequence caches; fp32 logits of the new rows only."""
        llm = self.llm
        if not handle.is_live_for(llm):
            raise ValueError("stale past_key_values: the decoder's KV cache has served another request since this handle was filled")
        if inputs_embeds is None:
            inputs_embeds = llm.embed_tokens(input_ids).view(*input_ids.shape, -1)
        if attention_mask is not None and not bool(attention_mask.bool().all()):
            raise NotImplementedError("padding with past_key_values is not supported")
        rows = inputs_embeds[0].to(self.dtype)
        L = handle.length
        hid = llm.prefill_hidden(rows, 0, L)
        logits = llm.logits_all(hid)[None]
        handle.update(llm, torch.cat([handle.rows[:L], rows], 0), L + rows.shape[0])
        handle.last_reused = L
        return CausalLMOutputWithPast(logits=logits, past_key_values=handle)

    # ---- forward: logits for every position (llava_llama.py:100-192) ----------------------------------
    @torch.no_grad()
    @ops.in_own_dtype
    def forward(self, input_ids=None, images=None, masks=None, depths=None, attention_mask=None, position_ids=None,
                past_key_values=None, seqlens_in_batch=None, inputs_embeds=None, labels=None, use_cache=None, **kwargs):
        """``past_key_values=h`` (a PagedKVCacheHandle, batch 1, text rows only): ``input_ids`` are the rows AFTER the cached
        ones (as prepare_inputs_for_generation feeds them, modeling_llama.py:1112-1149); they are prefilled at h.length over the
        cached positions, the logits cover the new rows, and h is advanced in place.  An empty handle, or ``use_cache=True``
        without one (batch 1), runs the full forward and returns the filled handle in ``past_key_values``."""
        if past_key_values is not None:
            n_batch = (input_ids if inputs_embeds is None else inputs_embeds).shape[0]
            self._check_handle(past_key_values, n_batch)
            if past_key_values.length > 0:
                if images is not None:
                    raise NotImplementedError("images together with a non-empty past_key_values: the reference re-splices the image into "
                                              "the new chunk there; pass the whole conversation to generate(..., past_key_values=) instead")
                return self._forward_continue(input_ids, inputs_embeds, attention_mask, past_key_values)
        if inputs_embeds is None:
            if images is None:
                inputs_embeds = self.llm.embed_tokens(input_ids).view(*input_ids.shape, -1)
            else:
                (_, position_ids, attention_mask, _, inputs_embeds, labels) = self.prepare_inputs_labels_for_multimodal(
                    input_ids, position_ids, attention_mask, None, labels, images, masks, depths)
        B, S, H = inputs_embeds.shape
        lens = [S] * B if attention_mask is None else attention_mask.bool().sum(-1).tolist()
        lens = [int(n) for n in lens]
        logits = torch.zeros((B, S, self.config.llama.vocab_size), dtype=torch.float32, device=self.device)
        valid = [slice(0, n) for n in lens]
        if attention_mask is not None:  # either padding side: the valid rows of a sequence are contiguous
            am = attention_mask.bool()
            for b in range(B):
                idx = torch.nonzero(am[b]).flatten()
                if idx.numel() != lens[b] or (lens[b] and int(idx[-1]) - int(idx[0]) + 1 != lens[b]):
                    raise NotImplementedError("attention masks with holes are not supported")
                valid[b] = slice(int(idx[0]), int(idx[0]) + lens[b]) if lens[b] else slice(0, 0)
        llm = self.llm
        llm.release_all()
        if B == 1:
            hid = llm.prefill_hidden(inputs_embeds[0, valid[0]], 0, 0)
        else:  # one packed pass over all rows of the batch
            llm.ensure_capacity(B, max(lens))
            llm.cache.reserve_many(lens)
            hid = llm.prefill_packed(torch.cat([inputs_embeds[b, valid[b]] for b in range(B)], 0), lens)
        lg = llm.logits_all(hid)
        o = 0
        for b in range(B):
            logits[b, valid[b]] = lg[o:o + lens[b]]
            o += lens[b]
        handle = past_key_values
        if handle is None and use_cache and B == 1 and type(llm).__name__ != "TPLlamaDecoder":
            handle = PagedKVCacheHandle()
        if handle is not None:
            handle.update(llm, inputs_embeds[0, valid[0]].to(self.dtype), lens[0])
            handle.last_reused = 0
        return CausalLMOutputWithPast(logits=logits, past_key_values=handle)

    __call__ = forward

    # ---- generate (llava_llama.py:194-213) --------------------------------------------------------------
    @torch.no_grad()
    @ops.in_own_dtype
    def generate(self, input_ids: Optional[torch.Tensor] = None, images: Optional[torch.Tensor] = None,
                 depths: Optional[torch.Tensor] = None, masks: Optional[List[torch.Tensor]] = None,
                 attention_mask: Optional[torch.Tensor] = None, **generation_kwargs):
        do_sample = bool(generation_kwargs.pop("do_sample", False))
        temperature = generation_kwargs.pop("temperature", None)
        top_p = generation_kwargs.pop("top_p", None)
        top_k = generation_kwargs.pop("top_k", None)
        seed = generation_kwargs.pop("seed", None)
        num_beams = int(generation_kwargs.pop("num_beams", 1) or 1)
        max_new_tokens = generation_kwargs.pop("max_new_tokens", None)
        max_length = generation_kwargs.pop("max_length", None)
        generation_kwargs.pop("use_cache", None)
        stopping_criteria = generation_kwargs.pop("stopping_criteria", None)
        pad_token_id = generation_kwargs.pop("pad_token_id", None)
        eos_token_id = generation_kwargs.pop("eos_token_id", self.config.llama.eos_token_id)
        return_logits = bool(generation_kwargs.pop("output_logits", False))
        use_graph = bool(generation_kwargs.pop("use_cuda_graph", True))
        handle = generation_kwargs.pop("past_key_values", None)
        # do_sample=True -> HF's TemperatureLogitsWarper + TopPLogitsWarper + multinomial, here one kernel per token
        # (eval_spatial.py:231-236 passes do_sample = temperature > 0, so temperature 0 stays greedy)
        sampling = None
        if do_sample and temperature not in (0, 0.0):
            sampling = dict(temperature=1.0 if temperature is None else float(temperature), top_p=top_p, top_k=top_k, seed=seed)
        length_penalty = float(generation_kwargs.pop("length_penalty", 1.0))
        early_stopping = bool(generation_kwargs.pop("early_stopping", False))
        if num_beams != 1 and (sampling is not None or return_logits):
            raise NotImplementedError("beam search is implemented for do_sample=False without output_logits (the eval scripts' mode)")
        if generation_kwargs:
            raise TypeError(f"unsupported generation kwargs: {sorted(generation_kwargs)}")
        if handle is not None:  # HF semantics: input_ids is the WHOLE sequence; the cached prefix is found by comparing input rows
            self._check_handle(handle, input_ids.shape[0], num_beams)

        packed = None
        if images is not None:
            self.prepare_inputs_labels_for_multimodal(input_ids, None, attention_mask, None, None, images, masks, depths, _packed_only=True)
            packed, lens = self._last_packed
            B = len(lens)
        else:
            inputs_embeds = self.llm.embed_tokens(input_ids).view(*input_ids.shape, -1)
            lens = [input_ids.shape[1]] * input_ids.shape[0] if attention_mask is None else attention_mask.sum(-1).tolist()
            B = inputs_embeds.shape[0]
        if max_new_tokens is None:
            max_new_tokens = 20 if max_length is None else max(int(max_length) - max(lens), 1)  # HF default max_length=20
        pad = pad_token_id if pad_token_id is not None else (self.config.llama.pad_token_id or 0)

        outs, all_logits = [], []
        stop_fn = None
        if stopping_criteria:
            def stop_fn(ids, _sc=stopping_criteria):
                return any(bool(c(ids[None], None)) for c in _sc)
        lens = [int(n) for n in lens]
        left = getattr(self.config.llama, "tokenizer_padding_side", "right") == "left"
        if num_beams != 1 and B != 1:
            raise NotImplementedError("beam search over a batch of prompts (the reference's eval scripts run batch 1)")
        if B == 1 and num_beams != 1:
            n = lens[0]
            emb = packed if packed is not None else (inputs_embeds[0, inputs_embeds.shape[1] - n:] if left else inputs_embeds[0, :n])
            if not hasattr(self.llm, "generate_beam") or type(self.llm).__name__ == "TPLlamaDecoder":
                raise NotImplementedError("beam search on the tensor-parallel decoder")
            outs.append(self.llm.generate_beam(emb, num_beams, int(max_new_tokens), eos_token_ids=eos_token_id, stopping_fn=stop_fn,
                                               length_penalty=length_penalty, early_stopping=early_stopping, use_graph=use_graph))
        elif B == 1:
            n = lens[0]
            emb = packed if packed is not None else (inputs_embeds[0, inputs_embeds.shape[1] - n:] if left else inputs_embeds[0, :n])
            reuse = 0
            if handle is not None:
                reuse = reusable_prefix(emb, handle.rows, handle.length, handle.is_live_for(self.llm))
            r = self.llm.generate_from_embeds(emb, int(max_new_tokens), eos_token_ids=eos_token_id, stopping_fn=stop_fn,
                                              use_graph=use_graph, return_logits=return_logits, sampling=sampling, prefix_len=reuse)
            if return_logits:
                r, lg = r
                all_logits.append(lg)
            outs.append(r)
            if handle is not None and r.numel():
                # the handle now describes prompt + answer; the KV of the last answer token is not final (cached_length)
                rows = torch.cat([emb.to(self.dtype), self.llm.embed_tokens(r)], 0)
                handle.update(self.llm, rows, LlamaDecoder.cached_length(n, r.numel()))
                handle.last_reused = reuse
        else:
            # batch > 1: one packed prefill over all prompts (llava_arch.py:549-611 pads, modeling_llama.py:540-562 unpads
            # again; here the rows were never padded), then per-sequence decode
            if packed is None:
                T = inputs_embeds.shape[1]
                packed = torch.cat([inputs_embeds[b, T - lens[b]:] if left else inputs_embeds[b, :lens[b]] for b in range(B)], 0)
            r = self.llm.generate_batch(packed, lens, int(max_new_tokens), eos_token_ids=eos_token_id, stopping_fn=stop_fn,
                                        use_graph=use_graph, return_logits=return_logits, sampling=sampling)
            if return_logits:
                outs, all_logits = r
            else:
                outs = r
        n_max = max(o.numel() for o in outs)
        seqs = torch.full((B, n_max), int(pad), dtype=torch.int64, device=self.device)
        for b, o in enumerate(outs):
            seqs[b, : o.numel()] = o
        if return_logits:
            return seqs, all_logits
        return seqs


LlavaLlamaForCausalLM = LlavaLlamaModel
