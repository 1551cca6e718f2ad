"""Prefill over cached KV pages: the paged attention kernel against fp32 attention built from the same pages, chunked prefill
against one-shot prefill, the incremental forward(past_key_values=) and the multimodal generate(past_key_values=) against the fp32
oracle, and RegionChat(reuse_kv=True) end to end.  Needs a B200."""
import numpy as np
import pytest
import torch

from oracle import srgpt_oracle as O
from tests.golden.make_golden import CASES
from tests.test_gpu_pipeline import build_model
from tests.util import BF16_1ROUND, BF16_CHAIN, assert_close, write_synthetic_checkpoint

pytestmark = pytest.mark.gpu
DEV = "cuda"
PAGE = 16


@pytest.fixture(scope="module")
def ops():
    from spatialrgpt_b200 import _lib, ops as _ops
    _lib.load()
    assert _lib.device_info()[1] == 10
    return _ops


def _paged_problem(starts, rows, nh, nkv, dtype, seed):
    """Random q rows and a paged cache holding positions [0, start + rows) of every sequence on scattered pages; every other slot
    of the cache is NaN (a kernel that reads past its sequence's context poisons its output)."""
    hd = 128
    g = torch.Generator().manual_seed(seed)
    ctx = [s + r for s, r in zip(starts, rows)]
    need = [(c + PAGE - 1) // PAGE for c in ctx]
    n_pages = sum(need) + 7
    perm = torch.randperm(n_pages, generator=g).tolist()
    cap = max(need) + 1
    pts = torch.zeros(len(starts), cap, dtype=torch.int32)
    o = 0
    for b, n in enumerate(need):
        pts[b, :n] = torch.tensor(perm[o:o + n], dtype=torch.int32)
        o += n
    pages = torch.full((n_pages, 2, PAGE, nkv, hd), float("nan"))
    kv = []
    for b, c in enumerate(ctx):
        k = torch.randn(c, nkv, hd, generator=g).to(dtype)
        v = torch.randn(c, nkv, hd, generator=g).to(dtype)
        for p in range(c):
            pg = int(pts[b, p // PAGE])
            pages[pg, 0, p % PAGE], pages[pg, 1, p % PAGE] = k[p].float(), v[p].float()
        kv.append((k, v))
    q_ld = (nh + 2 * nkv) * hd
    q = torch.randn(sum(rows), q_ld, generator=g).to(dtype)
    cu = torch.tensor([0] + np.cumsum(rows).tolist(), dtype=torch.int32)
    return q, pages.to(dtype), pts, cu, kv


def _ref(q, kv, starts, rows, nh, nkv):
    hd, G = 128, nh // nkv
    out, o = [], 0
    for (k, v), s, r in zip(kv, starts, rows):
        qb = q[o:o + r, :nh * hd].float().view(r, nh, hd).transpose(0, 1)            # [nh, r, hd]
        kk = k.float().transpose(0, 1).repeat_interleave(G, 0)                       # [nh, c, hd]
        vv = v.float().transpose(0, 1).repeat_interleave(G, 0)
        att = qb @ kk.transpose(1, 2) * hd ** -0.5
        pos = s + torch.arange(r)
        att = att.masked_fill(torch.arange(k.shape[0])[None, :] > pos[:, None], float("-inf"))
        out.append((att.softmax(-1) @ vv).transpose(0, 1).reshape(r, nh * hd))
        o += r
    return torch.cat(out)


SINGLE = [(s, r) for s in (0, 1, 15, 16, 17, 250) for r in (1, 7, 64, 129)]
RAGGED = [([0, 17, 250], [7, 129, 1]), ([16, 1, 15], [64, 1, 37])]


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float16])
@pytest.mark.parametrize("group", [1, 2, 4, 8])
def test_paged_attention_against_fp32(ops, group, dtype):
    nkv = 2
    nh = group * nkv
    with ops.elem_dtype(dtype):
        for i, (starts, rows) in enumerate([([s], [r]) for s, r in SINGLE] + RAGGED):
            q, pages, pts, cu, kv = _paged_problem(starts, rows, nh, nkv, dtype, seed=100 + i)
            ref = _ref(q, kv, starts, rows, nh, nkv)
            qd = q.to(DEV)
            args = (pages.to(DEV), pts.to(DEV), PAGE, cu.to(DEV), torch.tensor(starts, dtype=torch.int32, device=DEV), max(rows),
                    max(s + r for s, r in zip(starts, rows)), nh, nkv, 128, 128 ** -0.5)
            for split in (True, False):
                out = ops.attention_prefill_paged(qd, *args, split=split)
                assert_close(out, ref, rel_rms=1e-2, rel_max=8e-2, what=f"paged G{group} starts {starts} rows {rows} split={split} {dtype}")


@pytest.mark.parametrize("rows", [[1], [7], [64], [129], [259, 1, 64, 130]])
def test_paged_attention_at_position_0_equals_varlen_prefill(ops, rows):
    """start_pos = 0 over the chunk's own pages = the existing causal prefill on the same rows, to one rounding."""
    nh, nkv, hd = 8, 2, 128
    q, pages, pts, cu, kv = _paged_problem([0] * len(rows), rows, nh, nkv, torch.bfloat16, seed=7)
    qkv = q.clone()
    o = 0
    for (k, v), r in zip(kv, rows):  # the K / V columns of the fused buffer hold what the pages hold
        qkv[o:o + r, nh * hd:(nh + nkv) * hd] = k.reshape(r, -1)
        qkv[o:o + r, (nh + nkv) * hd:] = v.reshape(r, -1)
        o += r
    d = qkv.to(DEV)
    ref = ops.attention_prefill_varlen(d[:, :nh * hd], d[:, nh * hd:(nh + nkv) * hd], d[:, (nh + nkv) * hd:], cu.to(DEV), max(rows), nh, nkv, hd,
                                       hd ** -0.5, True)
    out = ops.attention_prefill_paged(d, pages.to(DEV), pts.to(DEV), PAGE, cu.to(DEV), torch.zeros(len(rows), dtype=torch.int32, device=DEV), max(rows),
                                      max(rows), nh, nkv, hd, hd ** -0.5)
    assert_close(out, ref, **BF16_1ROUND, what=f"paged vs varlen rows {rows}")


# ------------------------------------------------------------------------------------------ decoder level
def _agree_where_decided(ids, ref_ids, ref_logits, noise, what=""):
    """Greedy ids agree with the reference up to the first step whose top-1 / top-2 margin is within 4 x the rms noise (a near
    tie may flip under any change of summation order; after a flip the sequences diverge)."""
    top2 = ref_logits.float().topk(2, -1).values
    margin = (top2[:, 0] - top2[:, 1]).tolist()
    for t, (a, b) in enumerate(zip(ids, ref_ids)):
        if margin[t] <= 4 * noise:
            return t
        assert a == b, f"{what}: step {t} id {a} != {b} with margin {margin[t]:.3f} > 4 x noise {noise:.3f}"
    return len(ids)


@pytest.mark.parametrize("chunk", [1, 16, 37, 64])
def test_chunked_prefill_matches_one_shot(chunk):
    kw = CASES["tiny_masks_gqa"][0]
    oc, sd, model = build_model(kw, 5)
    llm = model.llm
    S = 150
    x = llm.embed_tokens(torch.randint(3, oc.vocab - 3, (S,), generator=torch.Generator().manual_seed(1)))
    llm.release_all()
    one = llm.prefill_hidden(x, 0, 0).clone()
    pages = llm.cache.pages.clone()
    pt = list(llm.cache.owned[0])
    llm.release_all()
    parts = [llm.prefill_hidden(x[a:a + chunk], 0, a).clone() for a in range(0, S, chunk)]
    assert_close(torch.cat(parts), one, **BF16_CHAIN, what=f"final hidden, chunks of {chunk}")

    def gather(pg, owned):  # [layers, 2, S, nkv, hd] through the page list
        return torch.cat([pg[:, p] for p in owned], dim=2)[:, :, :S]
    assert_close(gather(llm.cache.pages, llm.cache.owned[0]), gather(pages, pt), **BF16_CHAIN, what="KV pages")
    # greedy continuation from the chunked cache vs from one shot
    ids_one, lg_one = llm.generate_from_embeds(x, 8, return_logits=True)
    llm.release_all()
    for a in range(0, S - 1, chunk):
        llm.prefill_hidden(x[a:min(a + chunk, S - 1)], 0, a)
    ids_ch, lg_ch = llm.generate_from_embeds(x, 8, return_logits=True, prefix_len=S - 1)
    noise = float((lg_ch - lg_one).pow(2).mean().sqrt())
    _agree_where_decided(ids_ch.tolist(), ids_one.tolist(), lg_one, noise, "chunked")
    assert int(ids_ch[0]) == int(ids_one[0]) or float((lg_one[0].topk(2).values[0] - lg_one[0].topk(2).values[1])) <= 4 * noise


@pytest.mark.parametrize("name", list(CASES))
def test_incremental_forward_matches_oracle_cache(name):
    from spatialrgpt_b200.kv_handle import PagedKVCacheHandle
    kw, n_regions, t_text, kind, n_new, depth_on = CASES[name]
    oc, sd, model = build_model(kw, 9)
    input_ids, images, depths, masks = O.synth_request(oc, n_regions, t_text, seed=1234, kind=kind)
    if not depth_on:
        depths = None
    out = model.forward(input_ids=input_ids.to(DEV), images=images.to(DEV), masks=[m.to(DEV) for m in masks],
                        depths=None if depths is None else depths.to(DEV), use_cache=True)
    h = out.past_key_values
    assert isinstance(h, PagedKVCacheHandle) and h.get_seq_length() == out.logits.shape[1]
    enc = O.encode_multimodal(oc, sd, images, depths, masks)
    emb = O.splice_embeddings(oc, sd["llm"]["model.embed_tokens.weight"].float(), input_ids, enc["image_features"], enc["mask_embeds"],
                              enc["depth_embeds"], None, depths_given=depths is not None)[0]
    ref, cache = O.llama_forward(oc, sd["llm"], emb, None)
    sigma = float(ref.std())
    assert (out.logits[0].cpu() - ref).abs().max().item() <= 0.06 * sigma
    g = torch.Generator().manual_seed(2)
    for n in (1, 5, 3):
        new = torch.randint(3, oc.vocab - 3, (1, n), generator=g)
        L = h.get_seq_length()
        o2 = model.forward(input_ids=new.to(DEV), past_key_values=h)
        assert o2.past_key_values is h and h.get_seq_length() == L + n and h.last_reused == L and o2.logits.shape == (1, n, oc.vocab)
        ref, cache = O.llama_forward(oc, sd["llm"], sd["llm"]["model.embed_tokens.weight"].float()[new[0]], cache)
        err = (o2.logits[0].cpu() - ref).abs().max().item()
        assert err <= 0.06 * sigma, f"{name}: incremental logits err {err:.4f} > 0.06 sigma ({sigma:.3f}) after {L} cached rows"
    with pytest.raises(NotImplementedError):
        model.forward(input_ids=input_ids.to(DEV), images=images.to(DEV), masks=[m.to(DEV) for m in masks], past_key_values=h)
    model.generate(input_ids[:, :5].to(DEV), max_new_tokens=2)  # another request: the handle is stale now
    with pytest.raises(ValueError):
        model.forward(input_ids=new.to(DEV), past_key_values=h)
    with pytest.raises(NotImplementedError):
        model.forward(input_ids=torch.cat([new, new]).to(DEV), past_key_values=PagedKVCacheHandle())


def test_multimodal_continuation_matches_full_reprefill():
    from spatialrgpt_b200.kv_handle import PagedKVCacheHandle
    kw, n_regions, t_text, kind, n_new, depth_on = CASES["tiny_masks_gqa"]
    oc, sd, model = build_model(kw, 11)
    ids1, images, depths, masks = O.synth_request(oc, n_regions, t_text, seed=1234, kind=kind)
    dev_args = dict(images=images.to(DEV), depths=depths.to(DEV), masks=[m.to(DEV) for m in masks], do_sample=False)
    S1 = ids1.shape[1] - 1 + model._tokens_per_image()
    follow = torch.randint(100, 130, (1, 9), generator=torch.Generator().manual_seed(4))  # text ids inside the 1003-row table

    def turn2(h, **kw):
        out1 = model.generate(ids1.to(DEV), max_new_tokens=6, past_key_values=h, **dev_args)
        full = torch.cat([ids1, out1.cpu(), follow], 1)
        return full, out1.shape[1], model.generate(full.to(DEV), max_new_tokens=n_new, past_key_values=h, **dev_args, **kw)

    h = PagedKVCacheHandle()
    full, n1, (ids, logits) = turn2(h, output_logits=True)
    assert h.last_reused >= S1, (h.last_reused, S1)       # bitwise reuse: the encoders reproduced the first turn's rows
    assert h.last_reused == S1 + n1 - 1                   # everything but the last answer token (cached_length)
    ref_ids, enc = O.generate(oc, sd, full, images, depths, masks, n_new, return_all=True)
    sigma = float(enc["logits"].std())
    err = (logits[0].cpu() - enc["logits"]).abs().max().item()
    assert err <= 0.06 * sigma, f"continuation logits err {err:.4f} > 0.06 sigma ({sigma:.3f})"
    noise = float((logits[0].cpu() - enc["logits"]).pow(2).mean().sqrt())
    _agree_where_decided(ids[0].tolist(), ref_ids.tolist(), enc["logits"], noise, "continuation vs oracle re-prefill")
    # graph decode after a continuation = eager decode
    h2 = PagedKVCacheHandle()
    _, _, ids_graph = turn2(h2)
    assert h2.last_reused == h.last_reused and ids_graph[0].tolist() == ids[0].tolist()
    # sampling after a continuation
    h3 = PagedKVCacheHandle()
    out1 = model.generate(ids1.to(DEV), max_new_tokens=6, past_key_values=h3, **dev_args)
    full3 = torch.cat([ids1, out1.cpu(), follow], 1)
    samp = {k: v for k, v in dev_args.items() if k != "do_sample"}
    ids_s = model.generate(full3.to(DEV), max_new_tokens=n_new, past_key_values=h3, do_sample=True, temperature=0.8, top_p=0.9, seed=5, **samp)
    assert h3.last_reused == h.last_reused and ids_s.shape == (1, n_new) and int(ids_s.min()) >= 0 and int(ids_s.max()) < oc.vocab
    # a stale handle falls back to a full prefill; batch > 1 and beams are refused
    model.generate(ids1.to(DEV), max_new_tokens=2, **dev_args)
    model.generate(full3.to(DEV), max_new_tokens=2, past_key_values=h3, **dev_args)
    assert h3.last_reused == 0
    with pytest.raises(NotImplementedError):
        model.generate(full3.to(DEV), max_new_tokens=2, past_key_values=h3, num_beams=2, **dev_args)


def test_region_chat_reuse_kv_end_to_end(tmp_path):
    from PIL import Image

    from llava.model.builder import load_pretrained_model
    from spatialrgpt_b200.chat import RegionChat

    oc = O.OracleConfig(**CASES["tiny_masks_gqa"][0])
    sd = O.make_weights(oc, seed=3)
    root = str(tmp_path / "SpatialRGPT-tiny")
    write_synthetic_checkpoint(root, oc, sd, generation_eos=[2])
    tokenizer, model, image_processor, _ = load_pretrained_model(root, "SpatialRGPT-tiny", None)
    model.to(dtype=torch.bfloat16)
    model.config.image_processor = image_processor
    rng = np.random.RandomState(3)
    image = Image.fromarray(rng.randint(0, 255, (90, 120, 3), dtype=np.uint8))
    depth = Image.fromarray(np.repeat(rng.randint(0, 255, (90, 120, 1), dtype=np.uint8), 3, axis=2))
    segs = [np.zeros((90, 120), dtype=np.uint8) for _ in range(4)]
    for i, s in enumerate(segs):
        s[10 + 15 * i:50 + 15 * i, 20 + 10 * i:70 + 10 * i] = 1
    turns = [("How far is <region0> from <region1> ?", False), ("And <region2> ?", True), ("Is <region3> left of <region0> ?", True)]
    answers, reused = {}, []
    for reuse in (False, True):
        chat = RegionChat(model, tokenizer, image_processor, conv_mode="llava_v1", max_new_tokens=8, reuse_kv=reuse)
        answers[reuse] = []
        for text, follow in turns:
            answers[reuse].append(chat.ask(text, image, segs, depth_image=depth, follow_up=follow))
            if reuse:
                reused.append(chat.kv.last_reused)
    assert answers[True][0] == answers[False][0]          # turn 1 runs the plain path
    assert answers[True] == answers[False]                # follow-ups: the same answers from the cached prefix (no near-ties here)
    assert reused[0] == 0 and all(r > 0 for r in reused[1:]), reused
    print(f"chat reuse_kv: rows reused per turn {reused}; answers {answers}")
