"""Multi-turn region chat: the follow-up flow of the reference's demo (``demo/gradio_web_server_multi.py:137-236``,
``inference_vlm``) without the Gradio / SAM / DepthAnything front end (those are outside the hot path, SURVEY.md §8f.3).

A session keeps the conversation template and the user turns; in every turn
  * ``<regionN>`` in the user text becomes ``<mask> <depth>`` (or ``<mask>`` without the depth branch)            (:143-146)
  * the first turn gets the ``<image>`` token, a follow-up continues the running conversation                    (:148-154)
  * the region masks handed to ``generate()`` are the masks of ALL region references so far, in order of appearance,
    because the whole conversation is prefilled again and every ``<mask>`` token consumes one mask row          (:163-186)
  * ``KeywordsStoppingCriteria`` on the template's stop string, decoding, stop-string strip                      (:193-222)
  * ``[k]`` in the answer (the k-th region of THIS turn) is mapped back to the user's region number              (:225-228)
  * the answer replaces the open assistant slot of the conversation                                              (:234-236)

``reuse_kv=True`` keeps the KV of the conversation in the decoder's paged cache between turns (a ``PagedKVCacheHandle`` passed
as ``past_key_values``): a follow-up prefills only the rows that differ from the previous turn's prompt and answer, instead of
the whole conversation.  The answers then differ from a full re-prefill (what the reference does) at bf16-noise level only,
which is why it is opt-in.
"""
from __future__ import annotations

import re
from typing import List, Optional, Sequence

import numpy as np
import torch

from .constants import DEFAULT_IMAGE_TOKEN, IMAGE_TOKEN_INDEX
from .conversation import conv_templates
from .eval_spatial import clean_output, stop_string
from .kv_handle import PagedKVCacheHandle
from .mm_utils import KeywordsStoppingCriteria, process_images, process_regions, tokenizer_image_token


class RegionChat:
    def __init__(self, model, tokenizer, image_processor, conv_mode: str = "llama_3", temperature: float = 0.0, max_new_tokens: int = 512,
                 reuse_kv: bool = False):
        self.model, self.tokenizer, self.image_processor = model, tokenizer, image_processor
        self.conv_mode, self.temperature, self.max_new_tokens = conv_mode, temperature, max_new_tokens
        self.reuse_kv = reuse_kv
        self.kv: Optional[PagedKVCacheHandle] = None
        self.conv = conv_templates[conv_mode].copy()
        self.user_turns: List[str] = []
        self.model_turns: List[str] = []

    def reset(self) -> None:
        self.conv = conv_templates[self.conv_mode].copy()
        self.user_turns, self.model_turns = [], []
        self.kv = PagedKVCacheHandle() if self.reuse_kv else None

    def ask(self, text: str, image, seg_masks: Sequence[np.ndarray], depth_image=None, follow_up: bool = False) -> str:
        """``image`` / ``depth_image``: PIL images (the depth one as ``get_depth_map`` colours it, or None without the depth branch);
        ``seg_masks``: uint8 masks [H, W], ``<regionN>`` refers to ``seg_masks[N]``."""
        use_depth = depth_image is not None
        query = re.sub(r"<region\d+>", "<mask> <depth>" if use_depth else "<mask>", text)
        if not follow_up:
            query = DEFAULT_IMAGE_TOKEN + "\n" + query
            self.reset()
        self.user_turns.append(text)
        self.conv.append_message(self.conv.roles[0], query)
        self.conv.append_message(self.conv.roles[1], None)
        prompt = self.conv.get_prompt()
        region_indices = [int(i) for turn in self.user_turns for i in re.findall(r"<region(\d+)>", turn)]
        model, dev = self.model, self.model.device
        images = process_images([image], self.image_processor, model.config).to(dev, dtype=model.dtype)
        depths = process_images([depth_image], self.image_processor, model.config).to(dev, dtype=model.dtype) if use_depth else None
        masks: Optional[torch.Tensor] = None
        if len(seg_masks) > 0:
            masks = process_regions(list(seg_masks), self.image_processor, model.config)[region_indices].to(dev, dtype=model.dtype)
        input_ids = tokenizer_image_token(prompt, self.tokenizer, IMAGE_TOKEN_INDEX, return_tensors="pt").unsqueeze(0).to(dev)
        stop = stop_string(self.conv_mode)
        extra = {}
        if self.reuse_kv:
            if self.kv is None:
                self.kv = PagedKVCacheHandle()
            extra["past_key_values"] = self.kv
        out = model.generate(input_ids, images=[images], depths=None if depths is None else [depths], masks=[masks],
                             do_sample=self.temperature > 0, temperature=self.temperature, max_new_tokens=self.max_new_tokens, use_cache=True,
                             stopping_criteria=[KeywordsStoppingCriteria([stop], self.tokenizer, input_ids)], **extra)
        answer = clean_output(self.tokenizer.batch_decode(out, skip_special_tokens=True)[0], stop)
        turn_regions = re.findall(r"<region(\d+)>", text)
        mapping = {str(k): r for k, r in enumerate(turn_regions)}
        remapped = re.sub(r"\[([0-9]+)\]", lambda mt: f"[{mapping.get(mt.group(1), mt.group(1))}]", answer)
        self.conv.messages.pop()
        self.conv.append_message(self.conv.roles[1], answer)
        self.model_turns.append(remapped)
        return remapped
