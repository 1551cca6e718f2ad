"""A handle on the decoder's cached sequence, for ``past_key_values=`` of ``LlavaLlamaModel.generate`` / ``forward``.

The reference passes its KV cache around as tensors (HF ``DynamicCache`` / legacy tuples, grown by torch.cat,
modeling_llama.py:451-456) and, during generation, feeds only the rows after the cached prefix
(prepare_inputs_for_generation, modeling_llama.py:1112-1149).  Here the KV lives in the decoder's paged cache; the handle
records which sequence that cache holds, so a later call can prefill only the rows that are new.  Like a ``DynamicCache`` it
is mutated in place by the call it is passed to.

What the cache holds is decided by the INPUT rows: a call reuses the longest prefix of its spliced input-embedding rows that
is bitwise equal to the rows the handle recorded, so a different image, mask, depth map or text is never served from the
cache.  The decoder keeps one cached sequence; any other request on it (a plain generate, a batch, beam search, a cache
re-allocation) bumps its ``kv_epoch`` and makes older handles stale.
"""
from __future__ import annotations

from typing import Optional

import torch


class PagedKVCacheHandle:
    def __init__(self):
        self.decoder = None                    # the LlamaDecoder whose pages hold the sequence
        self.epoch: int = -1                   # decoder.kv_epoch when the handle was filled
        self.length: int = 0                   # positions [0, length) have final KV in the cache
        self.rows: Optional[torch.Tensor] = None  # input-embedding rows [>= length, H] of those positions (and possibly one more)
        self.last_reused: int = 0              # rows the last call took from the cache instead of prefilling them

    def get_seq_length(self) -> int:
        return self.length

    def is_live_for(self, decoder) -> bool:
        """True when the handle describes what `decoder`'s cache holds right now."""
        return self.decoder is not None and self.decoder is decoder and self.epoch == getattr(decoder, "kv_epoch", None) and self.length > 0

    def update(self, decoder, rows: torch.Tensor, length: int) -> None:
        self.decoder, self.epoch, self.rows, self.length = decoder, decoder.kv_epoch, rows, int(length)

    def __repr__(self) -> str:
        return f"PagedKVCacheHandle(length={self.length}, epoch={self.epoch}, last_reused={self.last_reused})"


def reusable_prefix(new_rows: torch.Tensor, cached_rows: Optional[torch.Tensor], cached_length: int, live: bool = True) -> int:
    """Rows of `new_rows` [S, H] whose KV can be taken from the cache: the first row index where `new_rows` and `cached_rows`
    differ bitwise, capped at `cached_length` (positions with final KV) and at S - 1 (the last prompt row is always prefilled, so
    the first new token has logits).  A stale (`live` False) or empty handle gives 0."""
    S = int(new_rows.shape[0])
    if not live or cached_rows is None or cached_length <= 0 or S <= 1:
        return 0
    m = min(S - 1, int(cached_length), int(cached_rows.shape[0]))
    if m <= 0:
        return 0
    if new_rows.shape[1:] != cached_rows.shape[1:] or new_rows.dtype != cached_rows.dtype:
        return 0
    a, b = new_rows[:m], cached_rows[:m].to(new_rows.device)
    if a.element_size() == 2:  # bitwise: -0.0 != +0.0 and NaN == NaN as the bits say
        a, b = a.view(torch.int16), b.view(torch.int16)
    diff = (a != b).reshape(m, -1).any(dim=1)
    idx = torch.nonzero(diff)
    return int(idx[0, 0]) if idx.numel() else m
