#!/usr/bin/env python
"""bench.py — BASELINE.json's headline metric on its config c2:

    generated tokens/sec, SpatialRGPT-VILA1.5-8B shape (SigLIP-so400m @448 px + Llama-3-8B), one image,
    8 mask regions, depth branch ON, 64-token prompt, 128 greedy tokens, batch 1 per GPU.

A "step" is one complete request through the hot path (2 tower passes, deconv refinement, mask
pooling, projector, splice, Llama prefill, 128 greedy tokens).  Synthetic inputs / random-init weights
of the named architecture (no checkpoints offline).

  python bench.py --gpus N --steps K --warmup W            # our sm_100a path (one rank per GPU under torchrun)
  python bench.py --impl reference --steps K --warmup W    # the reference algorithm (oracle port) on the host cores
  python bench.py --steps K --dump-outputs DIR             # also writes the last timed step's token ids to DIR/tokens.npy

Prints ONE JSON line (rank 0).  See DESIGN.md "Measurement" for the definitions of value / e2e / roofline.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

N_REGIONS, T_TEXT, NEW_TOKENS = 8, 64, 128
C3_BATCH, C3_REGIONS = 32, 4
METRIC = "generated_tokens_per_sec"
UNIT = "tokens/s"
WORKLOAD = ("c2: SigLIP-so400m@448px + Llama-3-8B, 1 image, 8 mask regions, depth ON, 64-token prompt "
            "(S=259 after splice), 128 greedy tokens, batch 1 per GPU")


def ncu_traffic():
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the dominant kernel, from the committed ncu capture."""
    p = os.path.join(ROOT, "profiles", "r01_ncu_traffic.json")
    try:
        return int(json.load(open(p))["decode_gemv_gateup_dram_bytes_per_launch"])
    except Exception:
        return None


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return (float(d["hbm_gbs"]), float(d["bf16_tflops"]), "measured (MEASURED_PEAKS.json)",
                float(d.get("bf16_tflops_sustained", d["bf16_tflops"])))
    return 6650.0, 1590.0, "fallback (B200_PROFILING.md)", 1590.0


# --------------------------------------------------------------------------------------------------
# clocks: sample nvidia-smi during the timed region
# --------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.idx = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200",
                                          "-i", str(self.idx)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for n, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# --------------------------------------------------------------------------------------------------
# synthetic request (SURVEY.md §8d), generated once on the host
# --------------------------------------------------------------------------------------------------
def make_request(cfg, seed):
    from spatialrgpt_b200.synth import synth_request
    return synth_request(cfg, N_REGIONS, T_TEXT, seed)


def make_batch(cfg, n_requests, n_regions, seed):
    """n_requests synthetic requests stacked into one generate() batch (config c3: 32 images, 4 regions each)."""
    from spatialrgpt_b200.synth import synth_request
    reqs = [synth_request(cfg, n_regions, T_TEXT, seed + 1000 * i) for i in range(n_requests)]
    return (torch.cat([r[0] for r in reqs]), torch.cat([r[1] for r in reqs]), torch.cat([r[2] for r in reqs]), [r[3][0] for r in reqs])


def algorithmic_numbers(cfg):
    """Per-request FLOPs / bytes (SURVEY.md §8d formulas)."""
    v, l = cfg.vision, cfg.llama
    T, Dv, Iv, Lv = v.grid ** 2, v.hidden_size, v.intermediate_size, v.num_hidden_layers - 1
    f_vit = Lv * (2 * T * (4 * Dv * Dv + 2 * Dv * Iv) + 4 * T * T * Dv) + 2 * T * 3 * v.patch_size ** 2 * Dv
    f_ref = 2 * T * Dv * 4 * Dv + 2 * 4 * T * Dv * 4 * Dv
    H, I, nh, nkv, hd, V = l.hidden_size, l.intermediate_size, l.num_attention_heads, l.num_key_value_heads, l.head_dim, l.vocab_size
    f_proj = 196 * 2 * (4 * Dv * H + H * H)
    f_tok = l.num_hidden_layers * 2 * (H * nh * hd + 2 * H * nkv * hd + nh * hd * H + 3 * H * I)
    S = T_TEXT - 1 + 196
    f_prefill = S * f_tok + l.num_hidden_layers * 2 * S * S * nh * hd + 2 * H * V
    w_stream = (l.num_hidden_layers * (H * (nh + 2 * nkv) * hd + nh * hd * H + 3 * H * I + 2 * H) + H + V * H) * 2
    kv_per_tok = l.num_hidden_layers * 2 * nkv * hd * 2
    return dict(S=S, flops_ttft=2 * f_vit + f_ref + f_proj + f_prefill, w_stream=w_stream, kv_per_tok=kv_per_tok,
                gateup_bytes=2 * I * H * 2)


# --------------------------------------------------------------------------------------------------
# our arm
# --------------------------------------------------------------------------------------------------
def run_ours(args):
    import torch.distributed as dist

    from spatialrgpt_b200 import baseline_config, ops
    from spatialrgpt_b200.distributed import aggregate_throughput
    from spatialrgpt_b200.llava_llama import LlavaLlamaModel
    from spatialrgpt_b200.weights import random_init

    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))
    # NCCL's log (incl. the "nranks N" init lines the driver reads) must reach stderr, never stdout: rank 0 prints ONE JSON line.
    # NCCL_DEBUG_FILE=/dev/stderr does NOT do that when stderr is a file (NCCL fopen()s it with "w": every rank truncates the
    # shared file and the log is lost - seen on the 2-GPU pre-flight), so each rank logs to its own temporary file and copies it to
    # stderr when it is done.  A caller who sets NCCL_DEBUG_FILE keeps their own destination.
    # The GPU boxes export NCCL_DEBUG=VERSION, which prints only a version banner (to stdout): levels below INFO are raised to
    # INFO / INIT so that the communicator's "rank r nranks N" lines exist; a caller's INFO / TRACE setting is kept.
    if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION", "WARN"):
        os.environ["NCCL_DEBUG"] = "INFO"
        os.environ.setdefault("NCCL_DEBUG_SUBSYS", "INIT")
    nccl_log = None
    if world > 1 and "NCCL_DEBUG_FILE" not in os.environ:
        import tempfile
        nccl_log = os.path.join(tempfile.gettempdir(), f"srgpt_nccl_rank{rank}_{os.getpid()}.log")
        os.environ["NCCL_DEBUG_FILE"] = nccl_log

    def forward_nccl_log():
        if nccl_log is not None and os.path.exists(nccl_log):
            try:
                with open(nccl_log, errors="replace") as f:
                    sys.stderr.write(f.read())
                sys.stderr.flush()
                os.remove(nccl_log)
            except OSError:
                pass
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    cfg = baseline_config("c2")
    wdtype = {"bf16": torch.bfloat16, "fp16": torch.float16}[args.dtype]
    from spatialrgpt_b200 import _lib
    _lib.set_elem({"bf16": "bf16", "fp16": "f16"}[args.dtype])  # process-wide: the per-kernel timing below calls ops.* directly
    model = LlavaLlamaModel(cfg, random_init(cfg, dev, seed=0, n_tower_layers=cfg.vision.num_hidden_layers - 1, dtype=wdtype), max_seq_len=1024)
    nums = algorithmic_numbers(cfg)
    hbm_peak, tensor_peak, peak_src, tensor_sustained = load_peaks()

    input_ids, images, depths, masks = make_request(cfg, 1234 + rank)
    pin = lambda t: t.pin_memory()  # noqa: E731
    h_ids, h_img, h_dep, h_msk = pin(input_ids), pin(images), pin(depths), pin(masks[0])
    d_ids, d_img, d_dep, d_msk = (t.to(dev) for t in (h_ids, h_img, h_dep, h_msk))
    gen_kw = dict(do_sample=False, max_new_tokens=NEW_TOKENS, use_cache=True)

    def step_device():
        return model.generate(d_ids, images=d_img, depths=d_dep, masks=[d_msk], **gen_kw)

    def step_e2e():
        ids = h_ids.to(dev, non_blocking=True)
        im = h_img.to(dev, non_blocking=True)
        de = h_dep.to(dev, non_blocking=True)
        mk = h_msk.to(dev, non_blocking=True)
        out = model.generate(ids, images=im, depths=de, masks=[mk], **gen_kw)
        return out.cpu()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        """Returns (ms, tokens, output of the last step)."""
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        n_tok = 0
        for _ in range(steps):
            out = fn()
            n_tok += int(out.numel())
        e1.record()
        barrier()
        ms, n_tok, _ = aggregate_throughput(e0.elapsed_time(e1), n_tok, dev)  # max over ranks; tokens all-gathered
        return ms, n_tok, out

    for _ in range(max(args.warmup, 3)):
        step_device()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    ops.LAUNCHES = 0
    ms, n_tok, last_ids = timed(step_device, args.steps)
    launches = ops.LAUNCHES
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        # token ids [1, NEW_TOKENS] of the last timed step; float64 holds every int64 id below 2^53 exactly
        import numpy as np
        os.makedirs(args.dump_outputs, exist_ok=True)
        np.save(os.path.join(args.dump_outputs, "tokens.npy"), last_ids.cpu().numpy().astype(np.float64))
    for _ in range(2):
        step_e2e()
    ms_e2e, n_tok_e2e, _ = timed(step_e2e, args.steps)

    # ---- the mode the reference's driver actually runs (eval_spatial.py:223-237): an EOS id plus KeywordsStoppingCriteria,
    #      inspected after every token.  Stop checks are asynchronous in our decoder (llama_decoder._decode_loop), so this
    #      should cost (almost) nothing; reported beside the headline, not instead of it.
    from types import SimpleNamespace

    from spatialrgpt_b200.mm_utils import KeywordsStoppingCriteria

    class _StubTokenizer:  # no tokenizer files offline: ids <-> "t<id>" words, enough for the real criterion class to run
        bos_token_id = 1

        def __call__(self, text):
            return SimpleNamespace(input_ids=[1] + [cfg.llama.vocab_size - 4 for _ in text.split()])

        def batch_decode(self, ids, skip_special_tokens=True):
            return [" ".join(f"t{int(i)}" for i in row) for row in ids]

    crit = KeywordsStoppingCriteria(["</s>"], _StubTokenizer(), h_ids)

    def step_stop():
        ids = h_ids.to(dev, non_blocking=True)
        out = model.generate(ids, images=h_img.to(dev, non_blocking=True), depths=h_dep.to(dev, non_blocking=True),
                             masks=[h_msk.to(dev, non_blocking=True)], eos_token_id=cfg.llama.vocab_size - 3, stopping_criteria=[crit], **gen_kw)
        return out.cpu()
    step_stop()
    ms_stop, n_tok_stop, _ = timed(step_stop, args.steps)

    # ---- TTFT (2 tower passes + refinement + pooling + projector + splice + Llama prefill + first token): the
    #      "prefill TFLOPS vs roofline" half of BASELINE.json's metric, algorithmic FLOPs of SURVEY.md §8d
    def step_ttft():
        return model.generate(d_ids, images=d_img, depths=d_dep, masks=[d_msk], do_sample=False, max_new_tokens=1)
    step_ttft()
    ms_ttft, _, _ = timed(step_ttft, args.steps)
    ttft_ms = ms_ttft / args.steps

    # ---- per-kernel roofline of the dominant kernel, timed live with CUDA events: the gate/up GEMV
    roof = None
    if rank == 0:
        llm = model.llm
        evs = []
        n_steps = 4
        for _ in range(n_steps):
            d, w = llm.dims, llm.w
            for l, lw in enumerate(w.layers):
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                ops.gemv(llm.h, lw.gateup_w, llm.act_buf, norm_weight=lw.post_norm, eps=d.rms_norm_eps, mode=ops.GEMV_SWIGLU)
                b.record()
                evs.append((a, b))
        torch.cuda.synchronize()
        dur = [a.elapsed_time(b) for a, b in evs][len(w.layers):]  # drop the first (warm) pass
        avg_ms = sum(dur) / len(dur)
        achieved = nums["gateup_bytes"] / avg_ms / 1e6
        # whole decode step, for context (graph replay timed with events)
        llm._ensure_graph(0)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        llm.step.zero_(); llm.pos.fill_(nums["S"])
        a.record()
        for _ in range(32):
            llm._graph.replay()
        b.record(); torch.cuda.synchronize()
        step_ms = a.elapsed_time(b) / 32
        step_bytes = nums["w_stream"] + nums["kv_per_tok"] * (nums["S"] + 16)
        roof = {"kernel": "gemv_kernel<SWIGLU> (rmsnorm + gate/up_proj 4096->2x14336 + SwiGLU), decode", "bound": "hbm",
                "achieved": round(achieved, 1), "peak": hbm_peak, "unit": "GB/s", "frac": round(achieved / hbm_peak, 4),
                "traffic": ncu_traffic(), "peak_source": peak_src, "bytes_per_launch": nums["gateup_bytes"], "avg_launch_ms": round(avg_ms, 5),
                "decode_step": {"ms": round(step_ms, 4), "algorithmic_GBps": round(step_bytes / step_ms / 1e6, 1),
                                "frac_hbm": round(step_bytes / step_ms / 1e6 / hbm_peak, 4), "kernels": llm.kernels_per_decode_step}}

    # ---- config c3: batch of 32 images x 4 regions, prefill only (generate(max_new_tokens=1)): every GEMM of the tower and
    #      of the Llama prefill runs over the whole batch (64 x 1024 ViT rows, 32 x 259 prompt rows) -> tensor-core bound
    c3 = None
    if not args.no_c3:
        b_ids, b_img, b_dep, b_msk = make_batch(cfg, C3_BATCH, C3_REGIONS, 4321 + rank)
        b_ids, b_img, b_dep = b_ids.to(dev), b_img.to(dev), b_dep.to(dev)
        b_msk = [m.to(dev) for m in b_msk]

        def step_c3():
            return model.generate(b_ids, images=b_img, depths=b_dep, masks=b_msk, do_sample=False, max_new_tokens=1)
        for _ in range(2):
            step_c3()
        l0 = ops.LAUNCHES
        ms_c3, n_c3, _ = timed(step_c3, args.steps)
        c3_launches = (ops.LAUNCHES - l0) // args.steps
        c3_ms = ms_c3 / args.steps
        c3_flops = C3_BATCH * nums["flops_ttft"]
        c3 = {"workload": f"c3: {C3_BATCH} images x {C3_REGIONS} mask regions, depth ON, 64-token prompts, prefill + first token, per GPU",
              "ms_per_batch": round(c3_ms, 2), "algorithmic_tflop": round(c3_flops / 1e12, 2),
              "tflops_per_gpu": round(c3_flops / c3_ms / 1e9, 1), "peak_tflops": tensor_peak, "peak_tflops_sustained": tensor_sustained,
              "frac_tensor": round(c3_flops / c3_ms / 1e9 / tensor_peak, 4),
              "frac_tensor_sustained": round(c3_flops / c3_ms / 1e9 / tensor_sustained, 4), "requests_per_s": round(C3_BATCH * world / (c3_ms / 1e3), 1),
              "gpu_launches_per_batch": int(c3_launches)}
        # batched decode of the same 32 requests (llama_decoder._decode_batched): every step streams each weight once for all 32
        # sequences (tcgen05 GEMMs over 32 rows, tall stream-K configuration) -> tokens/s per GPU grows ~32x over batch 1
        n_dec = 33

        def step_c3_dec():
            return model.generate(b_ids, images=b_img, depths=b_dep, masks=b_msk, do_sample=False, max_new_tokens=n_dec)
        step_c3_dec()
        # a differential measurement (33-token request - 1-token request) / 32: both terms are medians of 3 individually timed runs
        # (one sample of each made the step time swing by +-1 ms between runs of the same build)
        t_dec = sorted(timed(step_c3_dec, 1)[0] for _ in range(3))[1]
        t_pre = sorted(timed(step_c3, 1)[0] for _ in range(3))[1]
        step_ms_b = (t_dec - t_pre) / (n_dec - 1)
        c3["batched_decode"] = {"sequences": C3_BATCH, "new_tokens_per_sequence": n_dec, "ms_per_step": round(step_ms_b, 4),
                                "tokens_per_s_per_gpu": round(C3_BATCH / step_ms_b * 1e3, 1),
                                "algorithmic_GBps": round((nums["w_stream"] + C3_BATCH * nums["kv_per_tok"] * (nums["S"] + n_dec // 2)) / step_ms_b / 1e6, 1)}
        del b_ids, b_img, b_dep, b_msk

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        forward_nccl_log()
        return
    cpu = cpu_reference_sample()
    line = {
        "metric": METRIC, "value": round(n_tok / (ms / 1e3), 2), "unit": UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": max(args.warmup, 3), "ms_per_step": round(ms / args.steps, 3), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": args.dtype, "data": "synthetic",
        "config": {"workload": WORKLOAD, "requests_per_step_per_gpu": 1, "new_tokens": NEW_TOKENS, "parallelism": f"replicas x{world}",
                   "l2": "working set per step (16 GB of weights) exceeds the 126 MB L2; no flush needed",
                   "ttft_flops": nums["flops_ttft"]},
        "clocks": clocks,
        "e2e": {"value": round(n_tok_e2e / (ms_e2e / 1e3), 2), "unit": UNIT,
                "h2d_bytes_per_step": int(sum(t.numel() * t.element_size() for t in (h_ids, h_img, h_dep, h_msk))),
                "d2h_bytes_per_step": NEW_TOKENS * 8, "ms_per_step": round(ms_e2e / args.steps, 3)},
        "with_stop_checks": {"value": round(n_tok_stop / (ms_stop / 1e3), 2), "unit": UNIT, "tokens_per_step": n_tok_stop // max(args.steps * world, 1),
                             "ms_per_step": round(ms_stop / args.steps, 3),
                             "what": "e2e with eos_token_id + KeywordsStoppingCriteria inspected after every token (asynchronous stop checks)"},
        "gpu_launches": int(launches) * world,  # every rank launches the same kernels (replicas)
        "prefill": {"ttft_ms": round(ttft_ms, 3), "algorithmic_tflop": round(nums["flops_ttft"] / 1e12, 3),
                    "tflops": round(nums["flops_ttft"] / ttft_ms / 1e9, 1), "peak_tflops": tensor_peak,
                    "frac_tensor": round(nums["flops_ttft"] / ttft_ms / 1e9 / tensor_peak, 4),
                    "peak_tflops_sustained": tensor_sustained,
                    "frac_tensor_sustained": round(nums["flops_ttft"] / ttft_ms / 1e9 / tensor_sustained, 4),
                    "note": "S=259 rows per Llama GEMM: weight-streaming bound (15 GB), not tensor bound",
                    "batch32": c3},
        "roofline": roof,
        "cpu_baseline": cpu,
    }
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()
    forward_nccl_log()


# --------------------------------------------------------------------------------------------------
# CPU reference (oracle port), bounded sample of the same workload
# --------------------------------------------------------------------------------------------------
_CPU_STATE = {}


def _aliased_full_depth_weights(O):
    """Full-depth c2 state dicts for TIMING: every tower / decoder layer key aliases the tensors of one seeded layer (fp32) and
    lm_head aliases the token table, so the 8 B-parameter model costs 4 GB of host memory and seconds to build.  The arithmetic
    the oracle executes is the full 26 + 26 + 32 layers; only the VALUES repeat (CPU GEMM time does not depend on them)."""
    small = O.OracleConfig(v_layers=1, layers=1)
    w = O.make_weights(small, seed=0, dtype=torch.float32)
    full = O.OracleConfig()
    vt, llm = w["vision_tower"], w["llm"]
    for i in range(1, full.v_layers):
        for k in [k for k in list(vt) if ".layers.0." in k]:
            vt[k.replace(".layers.0.", f".layers.{i}.")] = vt[k]
    for i in range(1, full.layers):
        for k in [k for k in list(llm) if ".layers.0." in k]:
            llm[k.replace(".layers.0.", f".layers.{i}.")] = llm[k]
    return full, w


def cpu_reference_sample(decode_tokens: int = 6):
    """The reference algorithm (oracle/srgpt_oracle.py, the pinned CPU restatement of the reference's PyTorch path) timed on the
    host cores on ONE REAL c2 request at FULL depth: 26 SigLIP layers x 2 images (rgb + depth), refinement, mask pooling,
    projectors, splice, 32 Llama-3-8B layers of prefill at S = 259 with lm_head over all rows (modeling_llama.py:1044), then
    `decode_tokens` greedy decode steps through all 32 layers.  fp32 compute.  Nothing is scaled by layer counts; the only
    extrapolation is the decode tail: 128 tokens = TTFT + 127 x the measured per-token time (SURVEY.md §8d allows
    "prefill + 8 decode tokens extrapolated, clearly labelled")."""
    from oracle import srgpt_oracle as O

    cores = os.cpu_count() or 1
    if "w" not in _CPU_STATE:
        torch.set_num_threads(min(cores, 32))
        oc, w = _aliased_full_depth_weights(O)
        _CPU_STATE["oc"], _CPU_STATE["w"] = oc, w
        _CPU_STATE["req"] = O.synth_request(oc, N_REGIONS, T_TEXT, seed=1234)
        # the reference (torch on the host) gets the thread count that serves it best: on many-core hosts torch's intra-op
        # pool is slower with every core than with a subset (measured on the 128-core GPU box).  Probe = one decoder layer.
        one = O.OracleConfig(v_layers=1, layers=1)
        tab = w["llm"]["model.embed_tokens.weight"]
        best = (None, 1e30)
        # score = the request's own mix: 127 x one FULL-DEPTH decode token (all 32 layers, best of 3) + the 259-row prompt (one layer,
        # best of 2, x 32).  One-layer probes of a few ms picked 8, 16 or 32 threads at random on the same box (2.9 .. 4.7 tokens/s)
        for t in sorted({cores, 64, 32, 16, 8}):
            if t > cores:
                continue
            torch.set_num_threads(t)
            t_dec, t_pre = 1e30, 1e30
            with torch.no_grad():
                O.llama_forward(one, w["llm"], tab[5][None], None)
                for _ in range(3):
                    t0 = time.perf_counter()
                    O.llama_forward(oc, w["llm"], tab[5][None], None)
                    t_dec = min(t_dec, time.perf_counter() - t0)
                for _ in range(2):
                    t0 = time.perf_counter()
                    O.llama_forward(one, w["llm"], tab[:259], None)
                    t_pre = min(t_pre, (time.perf_counter() - t0) * oc.layers)
            dt = (NEW_TOKENS - 1) * t_dec + t_pre
            if dt < best[1]:
                best = (t, dt)
        _CPU_STATE["threads"] = best[0]
    threads = _CPU_STATE["threads"]
    torch.set_num_threads(threads)
    oc, w, (input_ids, images, depths, masks) = _CPU_STATE["oc"], _CPU_STATE["w"], _CPU_STATE["req"]
    st = {}

    def timed(name, fn):
        t0 = time.perf_counter()
        r = fn()
        st[name] = time.perf_counter() - t0
        return r

    with torch.no_grad():
        tf = timed("tower_rgb_26_layers", lambda: O.vision_tower_forward(oc, w["vision_tower"], images))
        df = timed("tower_depth_26_layers", lambda: O.vision_tower_forward(oc, w["vision_tower"], depths))
        hres, lres = timed("refinement", lambda: O.feature_refinement(oc, w["region_extractor"], tf))
        me, de = timed("mask_pool_project", lambda: O.region_extractor_forward(oc, w["region_extractor"], hres, df, masks))
        feats = timed("mm_projector", lambda: O.mm_projector_forward(oc, w["mm_projector"], lres))
        emb = timed("splice", lambda: O.splice_embeddings(oc, w["llm"]["model.embed_tokens.weight"], input_ids, feats, me, de)[0])
        logits, cache = timed("llama_prefill_32_layers", lambda: O.llama_forward(oc, w["llm"], emb, None))
        tab = w["llm"]["model.embed_tokens.weight"]
        per_tok = []
        nxt = int(torch.argmax(torch.nan_to_num(logits[-1])))
        for _ in range(decode_tokens):
            t0 = time.perf_counter()
            logits, cache = O.llama_forward(oc, w["llm"], tab[nxt][None], cache)
            nxt = int(torch.argmax(torch.nan_to_num(logits[-1])))
            per_tok.append(time.perf_counter() - t0)
    ttft = sum(st.values())
    t_tok = statistics.median(per_tok)
    t_request = ttft + (NEW_TOKENS - 1) * t_tok
    st["decode_per_token_32_layers"] = t_tok
    return {"value": round(NEW_TOKENS / t_request, 4), "unit": UNIT, "cores": threads, "kind": "port",
            "sample": (f"oracle port, fp32, {threads} of {cores} host threads: ONE c2 request at full depth (2 x 26 SigLIP layers, "
                       f"refinement, pooling, projectors, splice, 32-layer Llama prefill at S=259) measured = TTFT {ttft:.1f} s, plus "
                       f"{decode_tokens} full-depth decode steps (median {t_tok * 1e3:.0f} ms/token); 128-token request = TTFT + 127 x "
                       f"per-token = {t_request:.1f} s.  Layer weights are aliased copies of one seeded layer (timing only)"),
            "stage_s": {k: round(v, 3) for k, v in st.items()}, "ttft_s": round(ttft, 2),
            "sample_cpu_seconds": round(ttft + sum(per_tok), 1)}


def run_reference(args):
    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    if rank != 0:
        return
    steps, warm = args.steps, args.warmup
    res = None
    for _ in range(min(warm, 1)):  # one warm-up sample is enough for the host (each is a full-depth request prefix)
        res = cpu_reference_sample(decode_tokens=3)
    vals, t0 = [], time.perf_counter()
    for _ in range(steps):
        res = cpu_reference_sample(decode_tokens=3)
        vals.append(res["value"])
    wall = time.perf_counter() - t0
    v = statistics.median(vals)
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": world, "steps": steps, "warmup": warm,
            "ms_per_step": round(wall / max(steps, 1) * 1e3, 1), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "fp32 (CPU)", "data": "synthetic", "config": {"workload": WORKLOAD},
            "cpu_baseline": {**res, "value": v},
            "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-c3", action="store_true", help="skip the batch-32 prefill-only measurement (config c3)")
    ap.add_argument("--dtype", default="bf16", choices=["bf16", "fp16"],
                    help="compute dtype: bf16 (how the reference's eval_spatial.py runs the model; the graded default) or fp16 (the loader default)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the token ids rank 0's last timed step returned to DIR/tokens.npy (float64); "
                         "inputs and weights are seeded, so runs with the same arguments can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs applies to the CUDA path (--impl ours)")
    if args.impl == "reference":
        run_reference(args)
    else:
        world = int(os.environ.get("WORLD_SIZE", 1))
        if args.gpus > 1 and world == 1:
            # convenience: re-launch under torchrun, one rank per GPU
            cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}",
                   "--master-addr", "127.0.0.1", "--master-port", "29511", os.path.abspath(__file__), "--gpus", str(args.gpus),
                   "--steps", str(args.steps), "--warmup", str(args.warmup), "--dtype", args.dtype]
            if args.dump_outputs:
                cmd += ["--dump-outputs", os.path.abspath(args.dump_outputs)]
            sys.exit(subprocess.call(cmd))
        run_ours(args)


if __name__ == "__main__":
    main()
