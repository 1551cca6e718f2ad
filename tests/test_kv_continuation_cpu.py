"""Host-side parts of KV continuation (past_key_values / chunked prefill) that need no GPU: argument rejection of the paged C
entries, the prefix rule that decides which cached rows are reused, and RegionChat's handle bookkeeping."""
from types import SimpleNamespace

import numpy as np
import pytest
import torch

from spatialrgpt_b200.kv_handle import PagedKVCacheHandle, reusable_prefix
from tests.golden.make_host_golden import ToyTokenizer


# ------------------------------------------------------------------------------------------ C entries: host validation
def test_paged_attention_rejects_bad_arguments_without_a_gpu():
    from spatialrgpt_b200 import _lib
    lib = _lib.load()
    buf = 1 << 12  # any non-null, 16-byte aligned address: validation returns before the launch
    ok = dict(q=buf, q_ld=4096, out=buf, o_ld=4096, kv=buf, pt=buf, pts=257, ps=16, n=1, cu=buf, sp=buf, mq=40, mc=430, nh=32, nkv=8,
              hd=128, scale=0.088, ws=None, wsb=0, st=None)

    def call(**over):
        a = dict(ok, **over)
        return lib.srgpt_attention_prefill_paged_bf16(a["q"], a["q_ld"], a["out"], a["o_ld"], a["kv"], a["pt"], a["pts"], a["ps"], a["n"], a["cu"],
                                                      a["sp"], a["mq"], a["mc"], a["nh"], a["nkv"], a["hd"], a["scale"], a["ws"], a["wsb"], a["st"])

    for bad in (dict(q=None), dict(kv=None), dict(pt=None), dict(cu=None), dict(sp=None), dict(out=None),
                dict(nh=30, nkv=8),            # heads not a multiple of kv heads
                dict(nh=32, nkv=2),            # GQA group 16 > 8
                dict(mc=20),                   # context shorter than the chunk
                dict(n=0), dict(pts=0), dict(q_ld=4100)):
        assert call(**bad) == -1, bad
        assert "invalid argument" in _lib.last_error()
    assert call(hd=64) == -3 and "head_dim" in _lib.last_error()
    assert call(ps=32) == -3 and "page_size" in _lib.last_error()
    # a split shape with a workspace that is too small
    need = lib.srgpt_attention_prefill_paged_workspace(1, 40, 430, 32, 8)
    assert need > 0
    assert call(ws=buf, wsb=need - 4) == -1


def test_paged_workspace_sizes():
    from spatialrgpt_b200 import _lib
    lib = _lib.load()
    assert lib.srgpt_attention_prefill_paged_workspace(1, 40, 430, 32, 8) > 0          # follow-up turn: 24 CTAs -> context split
    assert lib.srgpt_attention_prefill_paged_workspace(1, 512, 4096, 32, 8) == 0       # 256 CTAs: no split
    assert lib.srgpt_attention_prefill_paged_workspace(1, 40, 39, 32, 8) == -1
    assert lib.srgpt_attention_prefill_paged_workspace(0, 40, 430, 32, 8) == -1


def test_paged_layer_stack_rejects_bad_arguments_without_a_gpu():
    from spatialrgpt_b200 import _lib
    lib = _lib.load()
    b = 1 << 12
    args = [b, b, 1, b, b, b, b, None, 0, 40, 4096, 32, 8, 128, 14336, 1e-5, b, b, b, b, 257, 16, 1, b, 40, 430, None]
    for i, v in ((23, None), (18, None), (25, 39), (24, 41)):  # no cu_seqlens / start_pos, context < chunk, chunk > rows
        bad = list(args)
        bad[i] = v
        assert lib.srgpt_llama_prefill_layers_paged_bf16(*bad) == -1, i


# ------------------------------------------------------------------------------------------ the prefix rule
def _rows(n, seed=0, H=8):
    g = torch.Generator().manual_seed(seed)
    return torch.randn(n, H, generator=g).to(torch.bfloat16)


def test_prefix_is_the_first_differing_row():
    cached = _rows(10)
    new = torch.cat([cached[:6], _rows(5, seed=1)])
    assert reusable_prefix(new, cached, 10) == 6


def test_prefix_is_capped_at_length_and_at_s_minus_1():
    cached = _rows(10)
    new = torch.cat([cached, _rows(4, seed=1)])
    assert reusable_prefix(new, cached, 9) == 9          # the handle's last row has no final KV
    assert reusable_prefix(cached.clone(), cached, 10) == 9  # identical prompt: the last row is still prefilled (first logits)
    assert reusable_prefix(cached[:1].clone(), cached, 10) == 0
    assert reusable_prefix(cached[:5].clone(), cached, 3) == 3


def test_prefix_is_bitwise():
    cached = _rows(6)
    new = cached.clone()
    new[2, 3] = -new[2, 3] if float(new[2, 3]) != 0 else 1.0
    assert reusable_prefix(torch.cat([new, _rows(2, 3)]), cached, 6) == 2
    z = torch.zeros(4, 8, dtype=torch.bfloat16)
    nz = z.clone()
    nz[1, 0] = -0.0                                       # equal as numbers, different bits
    assert reusable_prefix(torch.cat([nz, z]), z, 4) == 1


def test_stale_or_empty_handle_reuses_nothing():
    cached = _rows(10)
    new = torch.cat([cached, _rows(3, 2)])
    assert reusable_prefix(new, cached, 10, live=False) == 0
    assert reusable_prefix(new, None, 0) == 0
    h = PagedKVCacheHandle()
    assert h.get_seq_length() == 0 and h.rows is None and not h.is_live_for(object())
    dec = SimpleNamespace(kv_epoch=3)
    h.update(dec, cached, 9)
    assert h.is_live_for(dec) and h.get_seq_length() == 9
    dec.kv_epoch += 1                                     # the decoder served another request
    assert not h.is_live_for(dec)
    assert not h.is_live_for(SimpleNamespace(kv_epoch=3))  # another decoder


def test_cached_length_rule():
    from spatialrgpt_b200.llama_decoder import LlamaDecoder
    # prompt S, n tokens returned: the prompt and decode steps 1..n-1 fed positions [0, S + n - 1)
    assert LlamaDecoder.cached_length(259, 1) == 259
    assert LlamaDecoder.cached_length(259, 128) == 386


# ------------------------------------------------------------------------------------------ RegionChat(reuse_kv=True)
def _chat_fixture():
    from PIL import Image
    from transformers import SiglipImageProcessor
    proc = SiglipImageProcessor(size={"height": 28, "width": 28})
    tok = ToyTokenizer()
    img = Image.fromarray(np.random.RandomState(0).randint(0, 255, (40, 50, 3), dtype=np.uint8))
    segs = [np.zeros((40, 50), dtype=np.uint8) for _ in range(3)]
    for i, s in enumerate(segs):
        s[5 * i:5 * i + 8, 4:20] = 1
    return proc, tok, img, segs


@pytest.mark.parametrize("reuse", [False, True])
def test_region_chat_passes_one_handle_per_conversation(reuse):
    from spatialrgpt_b200.chat import RegionChat
    proc, tok, img, segs = _chat_fixture()
    calls = []

    class Stub:
        device = torch.device("cpu")
        dtype = torch.bfloat16
        config = SimpleNamespace(image_aspect_ratio="resize", mm_use_im_start_end=False)

        def generate(self, input_ids, images=None, depths=None, masks=None, **kw):
            calls.append(kw)
            return torch.tensor([tok("fine </s>").input_ids[1:]])

    chat = RegionChat(Stub(), tok, proc, conv_mode="llava_v1", reuse_kv=reuse)
    chat.ask("What is <region0> ?", img, segs)
    chat.ask("And <region1> ?", img, segs, follow_up=True)
    chat.ask("And <region2> ?", img, segs, follow_up=True)
    chat.ask("What is <region1> ?", img, segs)             # a new first turn
    if not reuse:
        assert all("past_key_values" not in kw for kw in calls)
        return
    hs = [kw["past_key_values"] for kw in calls]
    assert all(isinstance(h, PagedKVCacheHandle) for h in hs)
    assert hs[0] is hs[1] is hs[2]                         # follow-ups continue the same handle
    assert hs[3] is not hs[0]                              # a first turn starts a new one
