"""Follow-up turn of a region chat at the c2 dims (SigLIP@448 + Llama-3-8B, seeded random weights as bench.py builds them):
time to first token of turn 2 with the KV of turn 1 reused (generate(..., past_key_values=h)) against re-prefilling the whole
conversation (the reference's behaviour, RegionChat's default), alternated in one process; and the paged prefill-attention kernel
alone at the follow-up shape and at a 512-row chunk at the end of a 4096-position context.

    python tools/followup_turn.py [--reps 7] [--out FILE.json]

Turn 1 = the c2 request (1 image, 8 regions, depth on, 128 new tokens); turn 2 = turn 1 + its answer + a 40-token follow-up that
names 2 more regions.  Every reuse repetition re-runs turn 1 first (untimed) so the cache holds exactly turn 1 again.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

NEW_TOKENS, T_TEXT, N_REGIONS, FOLLOW = 128, 64, 8, 40


def card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else "unknown"


def attn_flops(n_heads: int, start: int, rows: int, hd: int = 128) -> float:
    """QK^T and P.V over the causal context of every row: row i sees start + i + 1 positions, 2 x 2 x hd flops per (head, position)."""
    seen = rows * start + rows * (rows + 1) // 2
    return 4.0 * n_heads * hd * seen


def kv_bytes(n_kv: int, ctx: int, hd: int = 128, elem: int = 2) -> float:
    """K and V of every position of the context, read once per kv head group (the kernel's one pass per q tile is L2-served)."""
    return 2.0 * ctx * n_kv * hd * elem


def time_kernel(ops, nh, nkv, start, rows, iters=200):
    dev = "cuda"
    ctx = start + rows
    n_pages = (ctx + 15) // 16
    g = torch.Generator().manual_seed(0)
    pages = (torch.randn(n_pages, 2, 16, nkv, 128, generator=g) * 0.5).to(torch.bfloat16).to(dev)
    pt = torch.randperm(n_pages, generator=g).to(torch.int32)[None].to(dev)
    q = torch.randn(rows, (nh + 2 * nkv) * 128, generator=g).to(torch.bfloat16).to(dev)
    cu = torch.tensor([0, rows], dtype=torch.int32, device=dev)
    sp = torch.tensor([start], dtype=torch.int32, device=dev)
    out = torch.empty(rows, nh * 128, dtype=torch.bfloat16, device=dev)
    ws = ops.attention_prefill_paged_workspace(1, rows, ctx, nh, nkv, dev)
    lib = ops._lib.load()

    def launch():
        ops.check(lib.srgpt_attention_prefill_paged_bf16(q.data_ptr(), q.stride(0), out.data_ptr(), out.stride(0), pages.data_ptr(), pt.data_ptr(),
                                                         pt.stride(0), 16, 1, cu.data_ptr(), sp.data_ptr(), rows, ctx, nh, nkv, 128, 128 ** -0.5,
                                                         None if ws is None else ws.data_ptr(), 0 if ws is None else ws.numel() * 4,
                                                         torch.cuda.current_stream().cuda_stream), "paged attention")
    for _ in range(10):
        launch()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        launch()
    e1.record()
    torch.cuda.synchronize()
    us = e0.elapsed_time(e1) * 1e3 / iters
    fl, by = attn_flops(nh, start, rows), kv_bytes(nkv, ctx)
    return dict(rows=rows, start_pos=start, context=ctx, split=ws is not None, us_per_layer=round(us, 2), kv_MB=round(by / 1e6, 3),
                GB_per_s=round(by / us / 1e3, 1), GFLOP=round(fl / 1e9, 3), TFLOP_per_s=round(fl / us / 1e6, 2))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    from spatialrgpt_b200 import baseline_config, ops
    from spatialrgpt_b200.kv_handle import PagedKVCacheHandle
    from spatialrgpt_b200.llava_llama import LlavaLlamaModel
    from spatialrgpt_b200.synth import synth_request
    from spatialrgpt_b200.weights import random_init

    assert torch.cuda.is_available(), "needs a B200"
    dev = torch.device("cuda", 0)
    cfg = baseline_config("c2")
    model = LlavaLlamaModel(cfg, random_init(cfg, dev, seed=0, n_tower_layers=cfg.vision.num_hidden_layers - 1), max_seq_len=1024)
    d = cfg.llama
    ids1, images, depths, masks8 = synth_request(cfg, N_REGIONS, T_TEXT, 1234)
    _, _, _, masks10 = synth_request(cfg, N_REGIONS + 2, T_TEXT, 1234)  # same generator: the first 8 masks are the same, 2 more follow
    assert torch.equal(masks10[0][:N_REGIONS], masks8[0])
    g = torch.Generator().manual_seed(77)
    follow = torch.randint(1000, 30000, (1, FOLLOW), generator=g)
    for p in (5, 20):  # "... <mask> <depth> ..." twice: the follow-up names 2 more regions
        follow[0, p], follow[0, p + 1] = cfg.llm_mask_token_id, cfg.llm_depth_token_id
    kw1 = dict(images=images.to(dev), depths=depths.to(dev), masks=[masks8[0].to(dev)], do_sample=False, eos_token_id=None)
    kw2 = dict(images=images.to(dev), depths=depths.to(dev), masks=[masks10[0].to(dev)], do_sample=False, eos_token_id=None, max_new_tokens=1)

    def turn1(h):
        return model.generate(ids1.to(dev), max_new_tokens=NEW_TOKENS, past_key_values=h, **kw1)

    out1 = turn1(None)
    full2 = torch.cat([ids1, out1.cpu(), follow], 1).to(dev)
    S2 = full2.shape[1] - 1 + model._tokens_per_image()

    def timed(fn):
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        r = fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1), r

    ttft = {"reprefill": [], "reuse": []}
    prefill_cont = []
    reused = None
    for rep in range(args.reps + 1):  # the first round warms up both paths (graph capture, lazy kernel attributes)
        ms, ids_off = timed(lambda: model.generate(full2, **kw2))
        if rep:
            ttft["reprefill"].append(ms)
        h = PagedKVCacheHandle()
        turn1(h)
        ms, ids_on = timed(lambda: model.generate(full2, past_key_values=h, **kw2))
        reused = h.last_reused
        if rep:
            ttft["reuse"].append(ms)
        # the continuation prefill alone (rows [L, S2) at position L; rewrites the same KV slots with the same values)
        emb = model._last_packed[0]
        ms, _ = timed(lambda: model.llm.prefill_hidden(emb[reused:], 0, reused))
        if rep:
            prefill_cont.append(ms)
    k_follow = time_kernel(ops, d.num_attention_heads, d.num_key_value_heads, S2 - (S2 - reused), S2 - reused)
    k_chunk = time_kernel(ops, d.num_attention_heads, d.num_key_value_heads, 4096 - 512, 512)
    med = {k: statistics.median(v) for k, v in ttft.items()}
    res = dict(
        card=card(),
        config="c2 dims (SigLIP@448 + Llama-3-8B, random weights seed 0), bf16",
        turn1=dict(prompt_rows=ids1.shape[1] - 1 + model._tokens_per_image(), new_tokens=NEW_TOKENS),
        turn2=dict(prompt_rows=S2, rows_reused=reused, rows_prefilled=S2 - reused, follow_up_tokens=FOLLOW, regions_total=N_REGIONS + 2),
        ttft_ms=dict(reprefill_median=round(med["reprefill"], 3), reuse_median=round(med["reuse"], 3),
                     reprefill_all=[round(x, 3) for x in ttft["reprefill"]], reuse_all=[round(x, 3) for x in ttft["reuse"]]),
        continuation_prefill_ms_median=round(statistics.median(prefill_cont), 3),
        paged_attention_kernel=dict(follow_up=k_follow, chunk_512_at_4096=k_chunk),
        paged_attention_share_of_continuation_prefill=round(k_follow["us_per_layer"] * d.num_hidden_layers / 1e3 / statistics.median(prefill_cont), 4),
        same_first_token=bool(int(ids_on[0, 0]) == int(ids_off[0, 0])),
        formulas=dict(flops="4 * n_heads * 128 * sum_i(start_pos + i + 1)", bytes="2 (K,V) * context * n_kv_heads * 128 * 2 bytes"),
    )
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
