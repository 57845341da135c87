#!/usr/bin/env python
"""bench.py — NVILA-8B single-image request (BASELINE.json configs[1]) on B200, plus the blocks the
other BASELINE configs need (all in ONE JSON line, printed by rank 0).

One "step" = one request through the hot path: 1 x 448^2 synthetic image -> SigLIP tower ->
mm_projector -> text/media splice -> Qwen2-7B prefill (S = 257 visual + 22 text = 279) -> first token
(TTFT) -> 127 more greedy tokens (CUDA-graph decode).  Random-init weights of the named architecture
(no checkpoints / network), bf16.

  value           decode tokens/s (README "decode throughput"), inputs resident in HBM, CUDA events
  ttft_ms         time to first token for the same request, inputs resident in HBM
  e2e             the same two numbers through the public API (LlavaLlamaModel.generate) with HOST
                  buffers: pinned pixels + ids copied H2D and the new ids read back D2H inside the region
  roofline        dominant kernel = the gate/up decode GEMV; algorithmic bytes = N*K*2 per launch
  decode_kernels  every kernel of the decode step timed live (CUDA events, back to back over all
                  layers' weights): achieved GB/s and fraction of the measured HBM peak
  ttft_roofline   flops / bytes / floor of the TTFT path and the achieved fraction
  video_decode    BASELINE configs[2] follow-up: 64-frame prefill (S = 16.5K) then 128 greedy tokens
                  through LlavaLlamaModel.generate: decode tok/s at ctx 16.5K with its HBM roofline
  batched_decode  serving follow-up: 8 concurrent copies of the request, continuous batching over one
                  shared paged pool (vila_b200/serving.py): aggregate tok/s
  tiled_image     BASELINE configs[3]: a dynamic-S2 tiled image (35 tiles of 448^2 -> tower -> S2 merge ->
                  projector) through encode_images, with its tensor-core floor (N = 1 runs only; last block of the run)
  sp_prefill      BASELINE configs[4]: LongVILA 256 frames (S = 65,814), sequence-parallel over ALL
                  ranks of this launch through LlavaLlamaModel.generate(max_new_tokens=1) with
                  vila_b200.sp enabled; first-token id + last-token logits top-5 / checksum so runs at
                  N = 1/2/4/8 can be compared from the driver's SCALE file alone (strong scaling)
  cpu_baseline    the oracle (PyTorch port of the reference's modules) on the host cores: the FULL
                  26-layer tower + projector + 28-layer prefill once, then a bounded number of decode
                  tokens through all 28 layers (no extrapolation); thread count swept and stated

`--dump-outputs DIR`    after the timed steps, rank 0 writes what the last timed request computed as DIR/<name>.npy
                        (last_step_outputs): inputs are seeded, so two builds can be compared output for output.
`--impl reference`      the same CPU port as its own arm (rank 0 only).
`--impl reference_gpu`  informational: HF transformers (SigLIP + Qwen2, sdpa, bf16, eager) on the same
                        B200 for the same request — the library path the reference would run.
Launch with torchrun for N > 1: the decode request does not shard at bs=1 ("replicas only",
SURVEY §8e): every rank serves its own replica, value = all ranks' tokens / max-over-ranks time; the
sp_prefill block is the part that really shards.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

if "--impl" in sys.argv and "reference" in sys.argv and os.environ.get("OMP_NUM_THREADS") == "1":
    # torch.distributed.run exports OMP_NUM_THREADS=1; the CPU arm sets its thread count explicitly
    os.environ.pop("OMP_NUM_THREADS")

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

PROMPT_TEXT_TOKENS = 22
NEW_TOKENS = 128


# ------------------------------------------------------------------------------------------------
def read_peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        d = json.loads(p.read_text())
        return {"hbm_gbs": float(d["hbm_gbs"]), "bf16_tflops": float(d["bf16_tflops"]),
                "bf16_tflops_sustained": float(d.get("bf16_tflops_sustained", d["bf16_tflops"])),
                "source": "measured (MEASURED_PEAKS.json)"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0,
            "source": "fallback (B200_PROFILING.md)"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int, period: float = 0.2):
        self.index = index
        self.period = period
        self.samples = []
        self._stop = threading.Event()
        self._t = threading.Thread(target=self._run, daemon=True)

    def _run(self):
        while not self._stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                      "-i", str(self.index)], capture_output=True, text=True, timeout=5).stdout
                self.samples.append([x.strip() for x in out.strip().split(",")])
            except Exception:
                pass
            self._stop.wait(self.period)

    def __enter__(self):
        self._t.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        self._t.join(timeout=3)

    def summary(self):
        sm = sorted(int(float(s[0])) for s in self.samples if s and s[0].replace(".", "").isdigit())
        mx = [int(float(s[1])) for s in self.samples if len(s) > 1 and s[1].replace(".", "").isdigit()]
        pw = [float(s[2]) for s in self.samples if len(s) > 2 and s[2].replace(".", "").isdigit()]
        reasons = set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for s in self.samples:
            for i, n in enumerate(names):
                if len(s) > 3 + i and s[3 + i].lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_mhz_min": sm[0] if sm else None,
                "sm_max_mhz": max(mx) if mx else None, "power_w_max": max(pw) if pw else None,
                "reasons": sorted(reasons), "samples": len(self.samples)}


# ------------------------------------------------------------------------------------------------
def make_request(cfg, seed=1):
    import torch
    g = torch.Generator().manual_seed(seed)
    S = cfg.vision_tower_cfg.image_size
    pixels = torch.randn(3, S, S, generator=g).to(torch.bfloat16)
    ids = torch.randint(0, 151643, (PROMPT_TEXT_TOKENS,), generator=g).tolist()
    ids.insert(14, cfg.image_token_id)  # "<system/user text> <image> <question>"
    return pixels, torch.tensor([ids], dtype=torch.long)


def last_step_outputs(emb, hid, dec):
    """Host copies of what one request_device() step computed (8 MB for NVILA-8B): the spliced prompt
    embeddings [S, hidden], the prefill's final hidden states [S, hidden] (before the last RMSNorm) and
    the NEW_TOKENS greedy ids (float64, exact).  Must run before the next request reuses these buffers
    (the prefill output is a static CUDA-graph buffer)."""
    return {"inputs_embeds": emb[0].float().cpu().numpy(),
            "prefill_hidden": hid.float().cpu().numpy(),
            "output_ids": dec.hist[:NEW_TOKENS].double().cpu().numpy()}


def write_outputs(outputs, out_dir):
    import numpy as np
    out = Path(out_dir)
    out.mkdir(parents=True, exist_ok=True)
    for name, arr in outputs.items():
        np.save(out / f"{name}.npy", arr)


def llm_weight_bytes(lc):
    layer_w = (lc.hidden_size * (lc.num_attention_heads + 2 * lc.num_key_value_heads) * lc.head_dim
               + lc.hidden_size * lc.num_attention_heads * lc.head_dim + 3 * lc.hidden_size * lc.intermediate_size)
    return 2 * (lc.num_hidden_layers * layer_w + lc.vocab_size * lc.hidden_size)


def decode_kernel_ledger(model, peaks, ctx=280):
    """Every kernel of one decode step, timed live with CUDA events: each kernel is launched back to
    back over ALL layers' weights (7.6 GB of gate/up weights etc. >> the 126 MB L2, so every launch
    streams from HBM; PDL lets launch i+1 prefetch under launch i exactly as in the decode graph)."""
    import torch

    from vila_b200 import ops
    llm = model.llm
    lc = llm.config
    Hq, Hkv, D = lc.num_attention_heads, lc.num_key_value_heads, lc.head_dim
    dev = llm.device
    x = torch.randn(lc.hidden_size, device=dev).to(torch.bfloat16)
    xa = torch.randn(Hq * D, device=dev).to(torch.bfloat16)
    xi = torch.randn(lc.intermediate_size, device=dev).to(torch.bfloat16)
    qkv = torch.empty((Hq + 2 * Hkv) * D, device=dev, dtype=torch.bfloat16)
    y = torch.empty(lc.hidden_size, device=dev, dtype=torch.bfloat16)
    act = torch.empty(lc.intermediate_size, device=dev, dtype=torch.bfloat16)
    key = torch.zeros(1, device=dev, dtype=torch.int64)
    dec = llm.decoder(NEW_TOKENS)
    cache = dec.cache if dec.cache is not None else dec.cache_for(ctx + NEW_TOKENS)
    pos = torch.tensor([ctx], dtype=torch.int32, device=dev)
    layers = list(llm.model.layers)
    ev = lambda: torch.cuda.Event(enable_timing=True)

    def per_layer(fn, reps=4, n=None):
        for li, l in enumerate(layers):
            fn(li, l)
        torch.cuda.synchronize()
        a, b = ev(), ev()
        a.record()
        for _ in range(reps):
            for li, l in enumerate(layers):
                fn(li, l)
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b) * 1e3 / (reps * (n or len(layers)))

    rows = []

    def add(name, nbytes, us):
        gbs = nbytes / us / 1e3
        rows.append({"kernel": name, "algorithmic_bytes": int(nbytes), "us": round(us, 2),
                     "gbs": round(gbs, 1), "frac": round(gbs / peaks["hbm_gbs"], 4)})

    nq = (Hq + 2 * Hkv) * D
    add("gemv qkv (+RMSNorm, +bias) N=%d K=%d" % (nq, lc.hidden_size), 2 * nq * lc.hidden_size,
        per_layer(lambda li, l: ops.gemv(x, l._qkv_w, bias=l._qkv_b, norm_w=l.input_layernorm.weight,
                                         norm_eps=lc.rms_norm_eps, out=qkv, static_w=True)))
    add("decode_attn ctx=%d splits=%d (RoPE + KV append + attention; 0 = one CTA per query head)" % (ctx, dec.num_splits),
        2 * 2 * (ctx + 1) * Hkv * D,
        per_layer(lambda li, l: ops.decode_attention(qkv, pos, cache.k(li), cache.v(li), cache.page_table,
                                                     xa, dec.ws, dec.counters, llm.inv_freq, Hq, Hkv, D,
                                                     dec.num_splits, D ** -0.5)))
    add("gemv o_proj (+residual) N=%d K=%d" % (lc.hidden_size, Hq * D), 2 * lc.hidden_size * Hq * D,
        per_layer(lambda li, l: ops.gemv(xa, l.self_attn.o_proj.weight, residual=x, out=y, static_w=True)))
    add("gemv gate/up (+RMSNorm, SwiGLU) N=%d K=%d" % (2 * lc.intermediate_size, lc.hidden_size),
        2 * 2 * lc.intermediate_size * lc.hidden_size,
        per_layer(lambda li, l: ops.gemv(x, l._gu_w, norm_w=l.post_attention_layernorm.weight,
                                         norm_eps=lc.rms_norm_eps, swiglu=True, out=act, static_w=True)))
    add("gemv down (+residual) N=%d K=%d" % (lc.hidden_size, lc.intermediate_size),
        2 * lc.hidden_size * lc.intermediate_size,
        per_layer(lambda li, l: ops.gemv(xi, l.mlp.down_proj.weight, residual=x, out=y, static_w=True)))
    add("gemv lm_head (+RMSNorm, argmax) N=%d K=%d" % (lc.vocab_size, lc.hidden_size),
        2 * lc.vocab_size * lc.hidden_size,
        per_layer(lambda li, l: ops.gemv(x, llm.lm_head.weight, norm_w=llm.model.norm.weight,
                                         norm_eps=lc.rms_norm_eps, argmax_key=key, write_out=False,
                                         static_w=True), reps=1, n=len(layers)))
    return rows


def video_decode_block(model, peaks, frames_n=64, reps=3):
    """NVILA-Video follow-up to the headline: decode right after a 64-frame prefill (ctx 16.5K).
    Through LlavaLlamaModel.generate with device-resident frames; decode tok/s = 127 tokens /
    (t(128 new tokens) - t(1 new token))."""
    import torch
    cfg = model.config
    lc = cfg.llm_cfg
    g = torch.Generator(device="cuda").manual_seed(77)
    S_img = cfg.vision_tower_cfg.image_size
    frames = torch.randn(frames_n, 3, S_img, S_img, device="cuda", generator=g).to(torch.bfloat16)
    ids = torch.randint(0, 151643, (PROMPT_TEXT_TOKENS,), generator=torch.Generator().manual_seed(8)).tolist()
    ids.insert(14, cfg.video_token_id)
    ids = torch.tensor([ids], dtype=torch.long)
    ev = lambda: torch.cuda.Event(enable_timing=True)

    def run(n_new):
        a, b = ev(), ev()
        a.record()
        out = model.generate(input_ids=ids, media={"video": [frames]}, media_config={"video": {}},
                             max_new_tokens=n_new, eos_token_id=None)
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b), out

    run(1); run(NEW_TOKENS)
    t1 = sum(run(1)[0] for _ in range(reps)) / reps
    tn = sum(run(NEW_TOKENS)[0] for _ in range(reps)) / reps
    S = frames_n * 257 + PROMPT_TEXT_TOKENS
    ms_tok = (tn - t1) / (NEW_TOKENS - 1)
    kv_bytes = 2 * 2 * (S + NEW_TOKENS // 2) * lc.num_key_value_heads * lc.head_dim * lc.num_hidden_layers
    byts = llm_weight_bytes(lc) + kv_bytes
    del frames
    return {"workload": "NVILA-Video-8B: %d frames x 448^2 -> S=%d prefill, then %d greedy tokens (bs=1)"
                        % (frames_n, S, NEW_TOKENS),
            "decode_tok_s": round(1e3 / ms_tok, 2), "decode_ms_per_token": round(ms_tok, 4),
            "ttft_ms": round(t1, 2), "splits": model.llm.decoder(NEW_TOKENS).num_splits,
            "bytes_per_token": int(byts), "kv_bytes_per_token": int(kv_bytes),
            "achieved_gbs": round(byts / ms_tok / 1e6, 1),
            "frac_of_hbm_peak": round(byts / ms_tok / 1e6 / peaks["hbm_gbs"], 4)}


def tiled_image_block(peaks, reps=5):
    """BASELINE.json configs[3]: one dynamic-S2 tiled image — 1 + 4 + 5x6 = 35 tiles of 448^2 (what the tiler
    makes of a wide 4K frame at max_tiles 12, SURVEY §8d) -> SigLIP tower -> multi-scale merge to the
    largest scale (C = 3456) -> mm_projector -> re-stitched token grid [7680, 3584].  Vision + projector only:
    the model is built with the dynamic-S2 configuration and a 2-layer LLM stub (encode_images never touches
    the LLM layers).  Same call and shapes as tests/test_fullsize_gpu.py::test_cfg4_matches_oracle_full_depth."""
    import dataclasses

    import torch

    from vila_b200.model import LlavaLlamaModel, nvila_8b_dynamic_s2
    cfg = nvila_8b_dynamic_s2()
    cfg.llm_cfg = dataclasses.replace(cfg.llm_cfg, num_hidden_layers=2)
    model = LlavaLlamaModel(cfg, device="cuda").init_random(0, device_rng=True)
    bs = (5, 6)
    n_tiles = 1 + 4 + bs[0] * bs[1]
    g = torch.Generator(device="cuda").manual_seed(5)
    tiles = torch.randn(n_tiles, 3, 448, 448, device="cuda", generator=g).to(torch.bfloat16)
    tiles_pin = tiles.cpu().pin_memory()
    ev = lambda: torch.cuda.Event(enable_timing=True)

    def run(from_host):
        a, b = ev(), ev()
        a.record()
        x = tiles_pin.to("cuda", non_blocking=True) if from_host else tiles
        out = model.encode_images(x, block_sizes=[bs])
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b), out

    for _ in range(3):
        run(False)
    ms = sum(run(False)[0] for _ in range(reps)) / reps
    ms_h2d, out = 0.0, None
    for _ in range(reps):
        t, out = run(True)
        ms_h2d += t / reps
    tokens = int(out.shape[1])
    C, Hd = cfg.vision_tower_cfg.hidden_size, cfg.llm_cfg.hidden_size
    flops = n_tiles * (936e9 + 1.39e9) + bs[0] * bs[1] * 256 * (2 * 12 * C * Hd + 2 * Hd * Hd)
    floor_ms = flops / (peaks["bf16_tflops_sustained"] * 1e12) * 1e3
    del model, tiles
    torch.cuda.empty_cache()
    return {"workload": "dynamic-S2 tiled image: %d tiles x 448^2 (1 + 2x2 + %dx%d) -> tower -> S2 merge (C=%d) -> projector "
                        "-> %d tokens (BASELINE.json configs[3])" % (n_tiles, bs[0], bs[1], 3 * C, tokens),
            "api": "LlavaLlamaModel.encode_images(tiles, block_sizes=[(5, 6)])", "tiles": n_tiles, "tokens_out": tokens,
            "ms": round(ms, 3), "ms_with_h2d_of_tiles": round(ms_h2d, 3), "h2d_bytes": int(tiles_pin.numel() * 2),
            "tiles_per_s": round(n_tiles / (ms / 1e3), 1), "flops": flops, "floor_ms": round(floor_ms, 3),
            "frac_of_sustained_tensor_peak": round(floor_ms / ms, 4), "finite": bool(torch.isfinite(out.float()).all())}


def batched_decode_block(model, peaks, ids_h, pixels_d, slots=8):
    """Serving follow-up (SURVEY §8 f3): `slots` copies of the headline request decoded together with
    continuous batching over one shared paged pool (vila_b200/serving.py): aggregate tok/s; the weights
    are streamed once per step for all slots."""
    import torch

    from vila_b200.serving import BatchedDecoder
    lc = model.config.llm_cfg
    emb, _, _ = model._embed(ids_h, {"image": [pixels_d]}, {"image": {}}, None, None)
    prompt = emb[0].clone()
    S = prompt.shape[0]
    dec = BatchedDecoder(model.llm, slots=slots, max_tokens_per_slot=1024, max_new=NEW_TOKENS)
    dec.capture()
    ev = lambda: torch.cuda.Event(enable_timing=True)
    times = []
    for rep in range(3):
        for s_ in range(slots):
            dec.admit(s_, prompt)
        torch.cuda.synchronize()
        a, b = ev(), ev()
        a.record()
        dec.run(NEW_TOKENS - 1)
        b.record()
        torch.cuda.synchronize()
        times.append(a.elapsed_time(b))
        first = [dec.generated(s_)[:4] for s_ in range(slots)]
        for s_ in range(slots):
            dec.release(s_)
    ms = sum(times[1:]) / len(times[1:])
    step_ms = ms / (NEW_TOKENS - 1)
    kv = 2 * 2 * (S + NEW_TOKENS // 2) * lc.num_key_value_heads * lc.head_dim * lc.num_hidden_layers * slots
    byts = llm_weight_bytes(lc) + kv
    del dec
    return {"workload": "%d concurrent copies of the headline request (S=%d, %d greedy tokens each), continuous "
                        "batching over one shared paged pool" % (slots, S, NEW_TOKENS),
            "slots": slots, "aggregate_tok_s": round(slots * (NEW_TOKENS - 1) / (ms / 1e3), 1),
            "ms_per_step": round(step_ms, 4), "per_request_tok_s": round(1e3 / step_ms, 1),
            "bytes_per_step": int(byts), "achieved_gbs": round(byts / step_ms / 1e6, 1),
            "frac_of_hbm_peak": round(byts / step_ms / 1e6 / peaks["hbm_gbs"], 4),
            "all_slots_agree": bool(all(f == first[0] for f in first))}


def sp_prefill_block(model, args, peaks, rank, world, local):
    """BASELINE configs[4] through the public API with sequence parallelism over this launch's ranks."""
    import torch
    import torch.distributed as dist

    from vila_b200 import sp
    cfg = model.config
    lc = cfg.llm_cfg
    F = args.frames
    S_img = cfg.vision_tower_cfg.image_size
    g = torch.Generator(device="cuda").manual_seed(1234)  # the SAME video on every rank and for every N
    frames = torch.randn(F, 3, S_img, S_img, device="cuda", generator=g).to(torch.bfloat16)
    ids = torch.randint(0, 151643, (PROMPT_TEXT_TOKENS,), generator=torch.Generator().manual_seed(7)).tolist()
    ids.insert(14, cfg.video_token_id)
    ids = torch.tensor([ids], dtype=torch.long)
    S = F * 257 + PROMPT_TEXT_TOKENS
    sp.set_sequence_parallel_group(None)
    ev = lambda: torch.cuda.Event(enable_timing=True)
    vis_events = []
    orig = model._encode_frames

    def timed_encode(fr, batch=32):
        a, b = ev(), ev()
        a.record()
        r = orig(fr, batch)
        b.record()
        vis_events.append((a, b))
        return r

    model._encode_frames = timed_encode
    runner = model._sp_runner()
    pre_events = []
    orig_prefill = runner.prefill_hidden

    def timed_prefill(*a, **k):
        e0, e1 = ev(), ev()
        e0.record()
        r = orig_prefill(*a, **k)
        e1.record()
        pre_events.append((e0, e1))
        return r

    runner.prefill_hidden = timed_prefill

    def step():
        a, b = ev(), ev()
        a.record()
        out = model.generate(input_ids=ids, media={"video": [frames]}, media_config={"video": {}},
                             max_new_tokens=1, eos_token_id=None)
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b), int(out[0, 0])

    try:
        est = 0.0
        for _ in range(max(3, args.warmup) if not args.profile else 1):
            est = step()[0]
        # at least --sp-steps steps, and long enough for >= 20 nvidia-smi clock samples (a query takes
        # ~0.75 s on an 8-GPU box): ~20 s of timed steps, capped at 80 steps; same count on every rank
        n_steps = torch.tensor([max(args.sp_steps, min(80, int(20000.0 / max(est, 1.0)) + 1))], device="cuda")
        dist.all_reduce(n_steps, op=dist.ReduceOp.MAX)
        n_steps = int(n_steps)
        dist.barrier(); torch.cuda.synchronize()
        vis_events.clear()
        pre_events.clear()
        rows = []
        with ClockSampler(local, period=0.1) as clocks:
            for _ in range(n_steps):
                rows.append(step())
            dist.barrier(); torch.cuda.synchronize()
        tot = torch.tensor([sum(r[0] for r in rows) / len(rows),
                            sum(a.elapsed_time(b) for a, b in vis_events) / max(1, len(vis_events)),
                            sum(a.elapsed_time(b) for a, b in pre_events) / max(1, len(pre_events))],
                           device="cuda", dtype=torch.float64)
        dist.all_reduce(tot, op=dist.ReduceOp.MAX)
        ms, vis_ms, pre_ms = float(tot[0]), float(tot[1]), float(tot[2])
        tok = rows[-1][1]
        toks = torch.tensor([tok], device="cuda")
        all_toks = [torch.zeros_like(toks) for _ in range(world)]
        dist.all_gather(all_toks, toks)
        logits = model.llm.logits_from_hidden(model.llm.last_prefill_hidden[None])[0].float()
        top = torch.topk(logits, 5)
    finally:
        model._encode_frames = orig
        runner.prefill_hidden = orig_prefill
        sp.set_sequence_parallel_group(None, enabled=False)
    gemm_flops = 2.0 * 6.525e9 * S
    attn_flops = 2.0 * S * S * lc.num_attention_heads * lc.head_dim * lc.num_hidden_layers
    vit_flops = F * 936e9
    tf_gpu = (gemm_flops + attn_flops + vit_flops) / world / (ms / 1e3) / 1e12
    plan = sp.make_plan(S, world, rank)
    return {"workload": "LongVILA-8B %d frames x 448^2, S=%d tokens: vision tower sharded by frames + zigzag "
                        "SP-%d prefill + first token (BASELINE.json configs[4])" % (F, S, world),
            "api": "vila_b200.sp.set_sequence_parallel_group(); LlavaLlamaModel.generate(media={'video': [...]}, max_new_tokens=1)",
            "scaling": "strong", "n_gpus": world, "steps": n_steps, "warmup": max(3, args.warmup),
            "ms_per_step": round(ms, 2), "tok_s": round(S / (ms / 1e3), 1),
            "phase_ms_max_over_ranks": {"vision_tower_projector_gather": round(vis_ms, 2),
                                        "sp_prefill_28_layers": round(pre_ms, 2),
                                        "splice_host_glue_first_token": round(ms - vis_ms - pre_ms, 2)},
            "padded_len": plan.padded_len, "chunk": plan.chunk,
            "first_token_id": tok, "first_token_ids_all_ranks": [int(t) for t in all_toks],
            "logits_top5_ids": [int(i) for i in top.indices], "logits_top5": [round(float(v), 4) for v in top.values],
            "logits_checksum": {"sum": round(float(logits.sum()), 3), "l2": round(float(logits.norm()), 4)},
            "achieved_tflops_per_gpu": round(tf_gpu, 1),
            "frac_of_sustained_bf16_peak": round(tf_gpu / peaks["bf16_tflops_sustained"], 4),
            "clocks": clocks.summary()}


def run_ours(args):
    import torch
    import torch.distributed as dist

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if "RANK" not in os.environ:  # plain `python bench.py`: a 1-rank group (the SP block needs one)
        os.environ.update({"RANK": "0", "WORLD_SIZE": "1", "MASTER_ADDR": "127.0.0.1",
                           "MASTER_PORT": os.environ.get("MASTER_PORT", "29533")})
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    from vila_b200 import _lib, ops
    from vila_b200.model import LlavaLlamaModel, nvila_8b

    cfg = nvila_8b()
    model = LlavaLlamaModel(cfg, device="cuda").init_random(0, device_rng=True)
    llm = model.llm
    pixels_h, ids_h = make_request(cfg, seed=1 + rank)
    pixels_pin = pixels_h.pin_memory()
    ids_pin = ids_h.pin_memory()
    pixels_d = pixels_h.cuda()
    media_cfg = {"image": {}}
    ev = lambda: torch.cuda.Event(enable_timing=True)

    vision_ms = []
    last = {}  # the latest request_device() results, for --dump-outputs

    def request_device():
        """inputs resident in HBM; returns (t_ttft_ms, t_decode_ms)."""
        e0, e1, e2, ea = ev(), ev(), ev(), ev()
        e0.record()
        emb, _, _ = model._embed(ids_h, {"image": [pixels_d]}, media_cfg, None, None)
        ea.record()
        dec = llm.decoder(NEW_TOKENS)
        cache = dec.cache_for(emb.shape[1] + NEW_TOKENS)
        hid = llm.prefill_hidden_graphed(emb[0], cache)
        dec.start(hid[-1], cache)
        e1.record()
        dec.run(NEW_TOKENS)
        e2.record()
        torch.cuda.synchronize()
        vision_ms.append(e0.elapsed_time(ea))  # SigLIP tower + projector + splice
        last.update(emb=emb, hid=hid, dec=dec)
        return e0.elapsed_time(e1), e1.elapsed_time(e2), emb.shape[1]

    def request_e2e(n_new):
        """public API with host buffers (pinned): H2D of pixels/ids and D2H of ids inside the region."""
        e0, e1 = ev(), ev()
        e0.record()
        out = model.generate(input_ids=ids_pin, media={"image": [pixels_pin]}, media_config=media_cfg,
                             max_new_tokens=n_new, eos_token_id=None)
        out_h = out.cpu()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1), out_h

    def barrier():
        dist.barrier()
        torch.cuda.synchronize()

    # ---- warm-up (graph capture, allocator, TMA descriptors) ----
    n_warm = 1 if args.profile else max(3, args.warmup)
    for _ in range(n_warm):
        request_device()
    request_e2e(1)
    request_e2e(NEW_TOKENS)

    # ---- timed: exactly K steps, device-resident ----
    launches0 = _lib.LAUNCHES
    barrier()
    ttfts, decs = [], []
    vision_ms.clear()
    with ClockSampler(local) as clocks:
        t_wall0 = time.perf_counter()
        for _ in range(args.steps):
            a, b, S = request_device()
            ttfts.append(a)
            decs.append(b)
        barrier()
        t_wall = time.perf_counter() - t_wall0
        launches_timed = _lib.LAUNCHES - launches0
        outputs = last_step_outputs(**last) if args.dump_outputs else None
        # e2e through the public API (host buffers)
        e2e_full, e2e_first = [], []
        for _ in range(args.steps):
            t, _ = request_e2e(NEW_TOKENS)
            e2e_full.append(t)
            t1, _ = request_e2e(1)
            e2e_first.append(t1)
    clock_summary = clocks.summary()
    peaks = read_peaks()
    # TTFT anatomy (outside the timed region): each stage alone, 10 repetitions, CUDA events around
    # the host call (so host-side Python that is not hidden behind GPU work shows up)
    def stage(fn, reps=10):
        fn(); torch.cuda.synchronize()
        a, b = ev(), ev()
        a.record()
        for _ in range(reps):
            fn()
        b.record(); torch.cuda.synchronize()
        return a.elapsed_time(b) / reps
    emb0, _, _ = model._embed(ids_h, {"image": [pixels_d]}, media_cfg, None, None)
    emb0 = emb0[0].clone()
    dec0 = llm.decoder(NEW_TOKENS)
    cache0 = dec0.cache_for(emb0.shape[0] + NEW_TOKENS)
    def _prefill():
        cache0.length = 0
        return llm.prefill_hidden_graphed(emb0, cache0)
    hid0 = _prefill()
    anatomy = {"encode_images_graph": round(stage(lambda: model.encode_images(pixels_d[None])), 3),
               "embed_total (encoders + host index table + splice)": round(stage(lambda: model._embed(ids_h, {"image": [pixels_d]}, media_cfg, None, None)), 3),
               "prefill_graph": round(stage(_prefill), 3),
               "first_token (lm_head GEMV + finalize)": round(stage(lambda: dec0.start(hid0[-1], cache0)), 3)}
    ledger = decode_kernel_ledger(model, peaks, ctx=S)
    video = None
    if not (args.profile or args.no_video):
        try:
            video = video_decode_block(model, peaks)
        except Exception as e:  # the headline line must survive a failure of an extra block
            video = {"error": "%s: %s" % (type(e).__name__, str(e)[:300])}
            torch.cuda.synchronize()

    batched = None
    if not (args.profile or args.no_video):
        try:
            batched = batched_decode_block(model, peaks, ids_h, pixels_d, slots=8)
            batched["more_slots"] = [
                {k: v for k, v in batched_decode_block(model, peaks, ids_h, pixels_d, slots=n).items()
                 if k in ("slots", "aggregate_tok_s", "ms_per_step", "frac_of_hbm_peak", "all_slots_agree")}
                for n in (32,)]
        except Exception as e:
            batched = {"error": "%s: %s" % (type(e).__name__, str(e)[:300])}
            torch.cuda.synchronize()

    step_ms = [a + b for a, b in zip(ttfts, decs)]
    local_stats = torch.tensor([sum(step_ms) / len(step_ms), sum(decs) / len(decs), sum(ttfts) / len(ttfts),
                                sum(e2e_full) / len(e2e_full), sum(e2e_first) / len(e2e_first)],
                               device="cuda", dtype=torch.float64)
    dist.all_reduce(local_stats, op=dist.ReduceOp.MAX)
    ms_step, ms_dec, ms_ttft, ms_e2e_full, ms_e2e_first = local_stats.tolist()

    sp_block = None
    if not args.no_sp and not args.profile:
        try:
            sp_block = sp_prefill_block(model, args, peaks, rank, world, local)
        except Exception as e:  # the headline line must survive a failure of the extra block
            sp_block = {"error": "%s: %s" % (type(e).__name__, str(e)[:300])}
            torch.cuda.synchronize()

    if rank != 0:
        dist.destroy_process_group()
        return
    decode_tok_s = world * (NEW_TOKENS - 1) / (ms_dec / 1e3)
    e2e_decode_tok_s = world * (NEW_TOKENS - 1) / ((ms_e2e_full - ms_e2e_first) / 1e3)
    lc = cfg.llm_cfg
    weight_bytes_token = llm_weight_bytes(lc)
    gu = next(r for r in ledger if r["kernel"].startswith("gemv gate/up"))
    gemv_bytes, gemv_ms, achieved = gu["algorithmic_bytes"], gu["us"] / 1e3, gu["gbs"]
    ncu_file = ROOT / "profiles" / "ncu_dominant_kernel.json"
    traffic = None
    if ncu_file.exists():
        try:
            traffic = json.loads(ncu_file.read_text()).get("dram_bytes_per_launch")
        except Exception:
            traffic = None
    vis_avg = sum(vision_ms[:args.steps]) / max(1, min(len(vision_ms), args.steps))
    # TTFT floor: tower (26 evaluated layers) + projector on the tensor pipe, prefill at the ridge
    vit_flops, proj_flops = 936e9 + 1.39e9, 15.0e9
    prefill_flops = 2.0 * 6.525e9 * S + 2.0 * lc.vocab_size * lc.hidden_size
    tf = peaks["bf16_tflops_sustained"] * 1e12
    floor_vis = (vit_flops + proj_flops) / tf * 1e3
    floor_llm = max(prefill_flops / tf, weight_bytes_token / (peaks["hbm_gbs"] * 1e9)) * 1e3
    cpu = None
    if not args.no_cpu and world == 1:
        cpu = cpu_reference(cfg, seconds_budget=args.cpu_budget)["cpu_baseline"]
    dec_obj = llm.decoder(NEW_TOKENS)
    tiled = None
    if world == 1 and not (args.profile or args.no_video):
        try:  # last GPU work of the run; the headline line must survive a failure of this extra block
            tiled = tiled_image_block(peaks)
        except Exception as e:
            tiled = {"error": "%s: %s" % (type(e).__name__, str(e)[:300])}
    line = {
        "metric": "NVILA-8B decode tokens/sec (1 img 448^2, bs=1, 128 new tokens); TTFT reported as ttft_ms",
        "value": round(decode_tok_s, 2), "unit": "tok/s", "n_gpus": world, "steps": args.steps,
        "warmup": max(3, args.warmup), "ms_per_step": round(ms_step, 3), "higher_is_better": True,
        "scaling": "weak", "vs_baseline": round(decode_tok_s / world / 82.1, 3),
        "baseline_ref": "BASELINE.md: NVILA-8B FP16 PyTorch decode 82.1 tok/s on A100 (README.md:65); other hardware",
        "dtype": "bf16", "data": "synthetic (random-init weights of the named architecture, randn pixels, random ids)",
        "ttft_ms": round(ms_ttft, 3), "decode_ms_per_token": round(ms_dec / (NEW_TOKENS - 1), 4),
        "ttft_breakdown_ms": {"vision_projector_splice": round(vis_avg, 3),
                              "llm_prefill_first_token": round(ms_ttft - vis_avg, 3)},
        "ttft_anatomy_ms": anatomy,
        "config": {"workload": "NVILA-8B bf16, 1x448^2 image, prefill S=%d + %d-token greedy decode, bs=1 "
                               "(BASELINE.json configs[1])" % (S, NEW_TOKENS),
                   "vision": "SigLIP-so400m/14-448 (26 of 27 layers evaluated: hidden_states[-2])",
                   "projector": cfg.mm_projector_type, "llm": "Qwen2.5-7B architecture",
                   "parallelism": "replicas x%d (decode does not shard at bs=1); sp_prefill block: sp%d" % (world, world),
                   "l2_policy": "no flush needed: each decode step streams %.2f GB of weights (>> 126 MB L2)"
                                % (weight_bytes_token / 1e9)},
        "e2e": {"value": round(e2e_decode_tok_s, 2), "unit": "tok/s",
                "ttft_ms": round(ms_e2e_first, 3), "request_ms": round(ms_e2e_full, 3),
                "request_tok_s": round(world * NEW_TOKENS / (ms_e2e_full / 1e3), 2),
                # pixels (bf16) + the int32 splice index table built from the host ids
                "h2d_bytes_per_step": int(pixels_pin.numel() * 2 + S * 4),
                # token history (int32) read back once at the end + the returned LongTensor copied to host
                "d2h_bytes_per_step": int(NEW_TOKENS * 4 + NEW_TOKENS * 8),
                "api": "LlavaLlamaModel.generate(input_ids=<pinned host>, media={'image': [<pinned host>]})"},
        "gpu_launches": int(launches_timed + args.steps * (NEW_TOKENS - 1) * dec_obj.launches_per_step),
        "gpu_launches_note": "timed region (K device-resident requests): %d C-ABI kernel launches issued from Python "
                             "(vision, projector, splice, first token; the prefill replays a CUDA graph of ~230 "
                             "more that are not counted) + CUDA-graph replays of %d kernels per decoded token"
                             % (launches_timed, dec_obj.launches_per_step),
        "clocks": clock_summary,
        "roofline": {"kernel": "gemv_tma_kernel (gate/up SwiGLU GEMV, N=%d K=%d, fused RMSNorm prologue)"
                               % (2 * lc.intermediate_size, lc.hidden_size),
                     "bound": "hbm", "achieved": round(achieved, 1), "peak": peaks["hbm_gbs"], "unit": "GB/s",
                     "frac": round(achieved / peaks["hbm_gbs"], 4), "traffic": traffic,
                     "peak_source": peaks["source"], "algorithmic_bytes_per_launch": gemv_bytes,
                     "launch_ms": round(gemv_ms, 5)},
        "decode_kernels": ledger,
        "decode_step_roofline": {"weight_bytes_per_token": weight_bytes_token,
                                 "achieved_gbs": round(weight_bytes_token / (ms_dec / (NEW_TOKENS - 1) / 1e3) / 1e9, 1),
                                 "frac_of_hbm_peak": round(weight_bytes_token / (ms_dec / (NEW_TOKENS - 1) / 1e3) / 1e9
                                                           / peaks["hbm_gbs"], 4)},
        "ttft_roofline": {"vit_projector_flops": vit_flops + proj_flops, "prefill_flops": prefill_flops,
                          "prefill_weight_bytes": weight_bytes_token,
                          "floor_ms": {"vision": round(floor_vis, 3), "llm_prefill": round(floor_llm, 3),
                                       "total": round(floor_vis + floor_llm, 3)},
                          "peaks": "sustained bf16 %.0f TFLOP/s, HBM %.0f GB/s" % (peaks["bf16_tflops_sustained"], peaks["hbm_gbs"]),
                          "frac": round((floor_vis + floor_llm) / ms_ttft, 4),
                          "frac_vision": round(floor_vis / vis_avg, 4),
                          "frac_llm": round(floor_llm / max(ms_ttft - vis_avg, 1e-6), 4)},
        "video_decode": video,
        "batched_decode": batched,
        "tiled_image": tiled,
        "sp_prefill": sp_block,
        "cpu_baseline": cpu,
        "wall_s_timed_region": round(t_wall, 3),
    }
    if outputs is not None:
        write_outputs(outputs, args.dump_outputs)
    print(json.dumps(line))
    dist.destroy_process_group()


# ------------------------------------------------------------------------------------------------
class CpuReference:
    """The reference's PyTorch path (oracle port) on the host cores at FULL size: 26 SigLIP layers +
    projector + 28 Qwen2-7B layers + lm_head in fp32 (~36 GB).  Weights: one randomly initialised
    layer per module type, the other layers are scaled copies written by a parallel multiply (so
    every layer owns distinct, touched memory; initialising 8 G parameters with the serial CPU RNG
    would take minutes and is not what is being measured)."""

    def __init__(self, cfg):
        import torch

        from oracle import vila_oracle as O
        self.O, self.torch, self.cfg = O, torch, cfg
        lc, vc = cfg.llm_cfg, cfg.vision_tower_cfg
        g = torch.Generator().manual_seed(0)

        def w(*shape, std=0.02):
            return torch.randn(*shape, generator=g) * std

        D, Hq, Hkv, Hd, I = lc.head_dim, lc.num_attention_heads, lc.num_key_value_heads, lc.hidden_size, lc.intermediate_size
        base = {"self_attn.q_proj.weight": w(Hq * D, Hd), "self_attn.q_proj.bias": w(Hq * D),
                "self_attn.k_proj.weight": w(Hkv * D, Hd), "self_attn.k_proj.bias": w(Hkv * D),
                "self_attn.v_proj.weight": w(Hkv * D, Hd), "self_attn.v_proj.bias": w(Hkv * D),
                "self_attn.o_proj.weight": w(Hd, Hq * D), "mlp.gate_proj.weight": w(I, Hd),
                "mlp.up_proj.weight": w(I, Hd), "mlp.down_proj.weight": w(Hd, I),
                "input_layernorm.weight": torch.ones(Hd), "post_attention_layernorm.weight": torch.ones(Hd)}
        p = {}
        for i in range(lc.num_hidden_layers):
            f = 1.0 + 0.01 * ((i * 7) % 5 - 2)
            for k, v in base.items():
                p[f"model.layers.{i}.{k}"] = v if i == 0 else v * f
        p["model.norm.weight"] = torch.ones(Hd)
        head = w(8192, Hd)
        reps = (lc.vocab_size + 8191) // 8192
        p["lm_head.weight"] = torch.cat([head * (1.0 + 0.003 * r) for r in range(reps)])[:lc.vocab_size].contiguous()
        p["model.embed_tokens.weight"] = p["lm_head.weight"]
        self.llm = p
        self.lcfg = O.Qwen2Cfg(Hd, I, lc.num_hidden_layers, Hq, Hkv, lc.vocab_size, lc.rms_norm_eps,
                               lc.rope_theta, D)
        C, Iv = vc.hidden_size, vc.intermediate_size
        sc = (2.0 / (2 * C)) ** 0.5
        vbase = {}
        for n in ("q_proj", "k_proj", "v_proj", "out_proj"):
            vbase[f"self_attn.{n}.weight"], vbase[f"self_attn.{n}.bias"] = w(C, C, std=sc), w(C)
        vbase["layer_norm1.weight"] = vbase["layer_norm2.weight"] = torch.ones(C)
        vbase["layer_norm1.bias"] = vbase["layer_norm2.bias"] = torch.zeros(C)
        vbase["mlp.fc1.weight"], vbase["mlp.fc1.bias"] = w(Iv, C, std=sc), w(Iv)
        vbase["mlp.fc2.weight"], vbase["mlp.fc2.bias"] = w(C, Iv, std=sc), w(C)
        vp = {}
        for i in range(vc.num_hidden_layers):
            for k, v in vbase.items():
                vp[f"vision_model.encoder.layers.{i}.{k}"] = v if i == 0 else v * (1.0 + 0.01 * (i % 3))
        vp["vision_model.embeddings.patch_embedding.weight"] = w(C, 3, vc.patch_size, vc.patch_size)
        vp["vision_model.embeddings.patch_embedding.bias"] = w(C)
        vp["vision_model.embeddings.position_embedding.weight"] = w(vc.num_patches, C)
        self.vision = vp
        self.vcfg = O.SiglipCfg(C, Iv, vc.num_hidden_layers, vc.num_attention_heads, vc.image_size, vc.patch_size)
        mm = 4 * C
        self.proj = {"layers.1.weight": torch.ones(mm), "layers.1.bias": torch.zeros(mm),
                     "layers.2.weight": w(Hd, mm), "layers.2.bias": w(Hd),
                     "layers.4.weight": w(Hd, Hd), "layers.4.bias": w(Hd)}
        self.pixels = torch.randn(1, 3, vc.image_size, vc.image_size, generator=g)
        self.text = torch.randn(PROMPT_TEXT_TOKENS + 1, Hd, generator=g) * 0.02
        self.past = None
        self.x = torch.randn(1, Hd, generator=g) * 0.02

    def ttft(self):
        """tower + projector + splice + 28-layer prefill + first-token logits; returns seconds"""
        O, torch = self.O, self.torch
        t0 = time.perf_counter()
        with torch.no_grad():
            feats = O.siglip_tower(self.pixels, self.vision, self.vcfg, -2)
            tok = O.projector(feats, self.proj, "mlp_downsample")[0]
            emb = torch.cat([self.text[:14], tok, self.text[14:]], 0)
            logits, self.past = O.qwen2_forward(emb, self.llm, self.lcfg, last_only=True)
            int(torch.argmax(logits[-1]))
        return time.perf_counter() - t0, emb.shape[0]

    def decode(self, n_tokens):
        """n greedy-decode steps through all 28 layers at the current context; past is NOT grown across
        calls beyond n tokens (each call restarts from the prefill's cache) so every sample is the same work"""
        O, torch = self.O, self.torch
        past = self.past
        t0 = time.perf_counter()
        with torch.no_grad():
            x = self.x
            for _ in range(n_tokens):
                logits, past = O.qwen2_forward(x, self.llm, self.lcfg, past=past, last_only=True)
                tok = int(torch.argmax(logits[-1]))
                x = self.llm["model.embed_tokens.weight"][tok][None, :]
        return time.perf_counter() - t0


def pick_threads(ref, candidates=None):
    """CPU decode is a memory-bound GEMV chain: more threads than memory channels need only adds
    synchronisation cost (128 threads on the 128-CPU B200 host: 26 s per token; 16 threads: 0.18 s).
    Sweep thread counts upwards on one decode token each, keep the fastest, and stop as soon as a count
    is more than 2x slower than the best so far (so the sweep itself stays cheap)."""
    import torch
    n = os.cpu_count() or 1
    cand = candidates or sorted({c for c in (8, 16, 32, 64, n // 2, n) if 1 <= c <= n})
    timings = {}
    best_t = None
    for c in cand:
        torch.set_num_threads(c)
        t = ref.decode(1)            # first token at this count (also the warm-up)
        if best_t is None or t < 2.0 * best_t:
            t = min(t, ref.decode(1), ref.decode(1))
        timings[c] = t
        if best_t is not None and t > 2.0 * best_t:
            break
        best_t = t if best_t is None else min(best_t, t)
    best = min(timings, key=timings.get)
    torch.set_num_threads(best)
    return best, {str(k): round(v, 4) for k, v in timings.items()}


def cpu_reference(cfg, seconds_budget=25.0, steps=1, warmup=0, tokens_per_step=8):
    """Returns {"cpu_baseline": {...}, "ttft_s": ..., "tok_s": ...}: the full-size CPU port, measured."""
    import torch
    t_build0 = time.perf_counter()
    ref = CpuReference(cfg)
    t_build = time.perf_counter() - t_build0
    torch.set_num_threads(os.cpu_count() or 1)
    t_ttft, S = ref.ttft()       # also builds the KV cache the decode samples start from
    best, sweep = pick_threads(ref)
    t_ttft2, _ = ref.ttft()      # with the chosen thread count
    ttft = min(t_ttft, t_ttft2)
    per_tok = ref.decode(2) / 2
    tokens_per_step = max(2, min(tokens_per_step, int(seconds_budget / max(1, steps + warmup) / max(per_tok, 1e-3))))
    for _ in range(warmup):
        ref.decode(tokens_per_step)
    times = [ref.decode(tokens_per_step) for _ in range(max(1, steps))]
    tok_s = tokens_per_step * len(times) / sum(times)
    cb = {"value": round(tok_s, 4), "unit": "tok/s", "cores": best, "kind": "port",
          "host_cpus": os.cpu_count(), "thread_sweep_s_per_token": sweep,
          "ttft_s": round(ttft, 3), "weights_build_s": round(t_build, 1),
          "sample": "oracle (fp32 PyTorch port of the reference modules) at FULL size on the host: %d-layer SigLIP "
                    "tower + projector + %d-layer LLM prefill at S=%d measured once (ttft_s), then %d x %d greedy "
                    "decode tokens through all %d layers + full-vocab lm_head at ctx %d (no extrapolation); "
                    "threads = fastest of the sweep"
                    % (cfg.vision_tower_cfg.num_hidden_layers - 1, cfg.llm_cfg.num_hidden_layers, S, len(times),
                       tokens_per_step, cfg.llm_cfg.num_hidden_layers, S)}
    return {"cpu_baseline": cb, "ttft_s": ttft, "tok_s": tok_s, "tokens_per_step": tokens_per_step,
            "step_s": sum(times) / len(times)}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from vila_b200.model import nvila_8b
    cfg = nvila_8b()
    r = cpu_reference(cfg, seconds_budget=max(60.0, args.cpu_budget * 4), steps=args.steps, warmup=args.warmup)
    cpu, v = r["cpu_baseline"], r["tok_s"]
    line = {
        "impl": "reference",
        "metric": "NVILA-8B decode tokens/sec (1 img 448^2, bs=1, 128 new tokens); TTFT reported as ttft_ms",
        "value": round(v, 4), "unit": "tok/s", "n_gpus": int(os.environ.get("WORLD_SIZE", "1")),
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(1e3 * r["step_s"], 1),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic", "ttft_ms": round(r["ttft_s"] * 1e3, 1),
        "config": {"workload": "NVILA-8B, 1x448^2 image, prefill S=279 + greedy decode, bs=1 (BASELINE.json "
                               "configs[1]); each step = %d decode tokens of the 128 (bounded CPU sample), TTFT "
                               "measured once at full size; see cpu_baseline.sample" % r["tokens_per_step"]},
        "cpu_baseline": cpu,
        "e2e": {"value": round(v, 4), "unit": "tok/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "note": "the reference CLI cannot run on CPU unmodified (flash-attn-only SigLIP, .cuda(), fp16; "
                "SURVEY §0.5) and llava.model does not import here; this arm is the oracle port of its modules",
    }
    print(json.dumps(line))


def run_reference_gpu(args):
    """Informational arm: the library path the reference runs (HF transformers SigLIP + Qwen2, torch
    sdpa attention, cuBLAS GEMMs, eager launches) on the same B200 for the same request.  The
    reference's own vendored SigLIP lives under /root/reference (absent on the GPU box); transformers'
    SiglipVisionModel is the same architecture.  Random-init weights on the device."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    try:
        import torch
        from transformers import Qwen2Config, Qwen2ForCausalLM, SiglipVisionConfig, SiglipVisionModel

        from oracle import vila_oracle as O
        from vila_b200.model import nvila_8b
        cfg = nvila_8b()
        lc, vc = cfg.llm_cfg, cfg.vision_tower_cfg
        torch.cuda.set_device(0)
        dev = torch.device("cuda")
        attn = "sdpa"
        with torch.device(dev):
            hf_l = Qwen2Config(hidden_size=lc.hidden_size, intermediate_size=lc.intermediate_size,
                               num_hidden_layers=lc.num_hidden_layers, num_attention_heads=lc.num_attention_heads,
                               num_key_value_heads=lc.num_key_value_heads, vocab_size=lc.vocab_size,
                               rms_norm_eps=lc.rms_norm_eps, rope_theta=lc.rope_theta,
                               max_position_embeddings=32768, tie_word_embeddings=False)
            hf_l._attn_implementation = attn
            llm = Qwen2ForCausalLM(hf_l).to(torch.bfloat16).eval()
            hf_v = SiglipVisionConfig(hidden_size=vc.hidden_size, intermediate_size=vc.intermediate_size,
                                      num_hidden_layers=vc.num_hidden_layers, num_attention_heads=vc.num_attention_heads,
                                      image_size=vc.image_size, patch_size=vc.patch_size)
            hf_v._attn_implementation = attn
            vit = SiglipVisionModel(hf_v).to(torch.bfloat16).eval()
            mm = 4 * vc.hidden_size
            proj = {"layers.1.weight": torch.ones(mm), "layers.1.bias": torch.zeros(mm),
                    "layers.2.weight": torch.randn(lc.hidden_size, mm) * 0.01, "layers.2.bias": torch.zeros(lc.hidden_size),
                    "layers.4.weight": torch.randn(lc.hidden_size, lc.hidden_size) * 0.01,
                    "layers.4.bias": torch.zeros(lc.hidden_size)}
            proj = {k: v.to(torch.bfloat16) for k, v in proj.items()}
        pixels_h, ids_h = make_request(cfg, seed=1)
        pixels = pixels_h.cuda()[None]
        text_ids = torch.tensor([i for i in ids_h[0].tolist() if i != cfg.image_token_id], device=dev)
        nl = torch.tensor(list(cfg.newline_token_ids), device=dev)
        ev = lambda: torch.cuda.Event(enable_timing=True)

        @torch.inference_mode()
        def request(n_new):
            a, b = ev(), ev()
            a.record()
            hs = vit(pixel_values=pixels, output_hidden_states=True).hidden_states[-2]
            tok = O.projector(hs, proj, "mlp_downsample")[0]
            table = llm.get_input_embeddings()
            emb = torch.cat([table(text_ids[:14]), tok, table(nl), table(text_ids[14:])], 0)[None]
            out = llm.generate(inputs_embeds=emb, attention_mask=torch.ones(emb.shape[:2], device=dev, dtype=torch.long),
                               max_new_tokens=n_new, min_new_tokens=n_new, do_sample=False, pad_token_id=0)
            out.cpu()
            b.record()
            torch.cuda.synchronize()
            return a.elapsed_time(b), emb.shape[1]

        for _ in range(max(1, min(args.warmup, 3))):
            request(1); request(NEW_TOKENS)
        t1 = tn = 0.0
        reps = max(1, min(args.steps, 5))
        with ClockSampler(0) as clocks:
            for _ in range(reps):
                a, S = request(1)
                b, _ = request(NEW_TOKENS)
                t1 += a / reps
                tn += b / reps
        v = (NEW_TOKENS - 1) / ((tn - t1) / 1e3)
        line = {"impl": "reference_gpu",
                "metric": "NVILA-8B decode tokens/sec (1 img 448^2, bs=1, 128 new tokens); TTFT reported as ttft_ms",
                "value": round(v, 2), "unit": "tok/s", "n_gpus": 1, "steps": reps, "warmup": args.warmup,
                "ms_per_step": round(tn, 2), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "bf16", "data": "synthetic", "ttft_ms": round(t1, 2),
                "config": {"workload": "NVILA-8B bf16, 1x448^2 image, prefill S=%d + %d greedy tokens, bs=1; HF transformers "
                                       "%s SiglipVisionModel + Qwen2ForCausalLM.generate(inputs_embeds=...), attn=%s, eager"
                                       % (S, NEW_TOKENS, __import__("transformers").__version__, attn)},
                "e2e": {"value": round(v, 2), "unit": "tok/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": NEW_TOKENS * 8},
                "clocks": clocks.summary(),
                "note": "library baseline (cuBLAS / sdpa / ATen through HF eager), not the product"}
    except Exception as e:
        line = {"impl": "reference_gpu", "unavailable": "%s: %s" % (type(e).__name__, str(e)[:300])}
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference", "reference_gpu"])
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-sp", action="store_true", help="skip the sp_prefill block")
    ap.add_argument("--no-video", action="store_true", help="skip the video_decode block")
    ap.add_argument("--cpu-budget", type=float, default=25.0)
    ap.add_argument("--frames", type=int, default=256, help="frames of the sp_prefill block")
    ap.add_argument("--sp-steps", type=int, default=10)
    ap.add_argument("--profile", action="store_true",
                    help="profiling aid (ncu): 1 warm-up, 8 new tokens, no extra blocks; NOT a valid bench number")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the last timed request's embeddings, prefill hidden states and ids as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    if args.profile:
        global NEW_TOKENS
        NEW_TOKENS = 8
        args.no_cpu = True
    if args.impl == "reference":
        run_reference(args)
    elif args.impl == "reference_gpu":
        run_reference_gpu(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
