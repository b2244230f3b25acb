#!/usr/bin/env python
"""bench.py — LiveCC streaming hot path on B200 (see DESIGN.md §Measurement).

One *step* = one full pass of the hot path over one synthetic 2 fps clip stream: the 6-frame first
chunk, then 2-frame chunks, each chunk = ViT -> prefill -> <=16 greedy decode steps with
repetition_penalty 1.05 (REF/demo/infer.py:62-180, REF/demo/cli.py:13-24).  Default workload =
BASELINE.json configs[1]: LiveCC-7B dims, 60 s clip (120 frames, 58 chunks) at 448x448, bf16, synthetic
checkpoint (no weights exist offline) and synthetic frames.

  value : tokens/s of the whole job with the chunk inputs already resident in HBM
  e2e   : the same metric through the public API (LiveCCDemoInfer.live_cc) with HOST frames:
          host patchify, pinned H2D of pixel rows + ids, D2H of the generated ids every chunk
  roofline      : the dominant kernel (decode gate/up GEMV) timed with CUDA events on its launch stream
  roofline_step : the whole decode step (CUDA-graph replay) timed inside the timed region
  cpu_baseline  : the reference's own eager CPU path (HF transformers fp32) on a bounded sample

`--impl reference` times only that CPU path (rank 0), same metric/config keys.
`--impl hf_gpu [--liger]` times the reference's own GPU path (installed transformers, bf16, flash_attention_2, through
oracle/hf_oracle.py) on the same clip and config: the "kernel to beat" line, printed with per-phase device time.
`--dump-outputs DIR` writes what the last timed step of the device-resident arm returned to its caller (rank 0), as .npy
files, so that two builds can be compared output for output on the same seeded inputs (see dump_outputs).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True  # the benchmark leaves the tree it runs from untouched (it may be read-only)

import torch  # noqa: E402

METRIC = "commentary tokens/sec + frames/sec at 7B 2fps 448x448; p50 per-frame latency"


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="native", choices=["native", "reference", "hf_gpu"],
                    help="native: this repo; reference: the reference's CPU path (driver arm); hf_gpu: the reference's GPU "
                         "path (HF bf16 + flash_attention_2, optionally --liger) on the same B200 = the kernel to beat")
    ap.add_argument("--liger", action="store_true", help="hf_gpu: apply_liger_kernel_to_qwen2_vl() first (REF/demo/infer.py:2-3)")
    ap.add_argument("--model", default="7b", choices=["7b", "small"])
    ap.add_argument("--seconds", type=int, default=60, help="clip length in seconds of video (2 fps)")
    ap.add_argument("--size", type=int, default=448)
    ap.add_argument("--max-new-tokens", type=int, default=16)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-batch", action="store_true", help="skip the multi-stream (generate_batch) sweep")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the outputs of the last timed step as DIR/<name>.npy (rank 0)")
    return ap.parse_args()


def get_config(name):
    from livecc_b200.config import LiveCCConfig

    return LiveCCConfig.livecc_7b() if name == "7b" else LiveCCConfig.small()


# ------------------------------------------------------------------------------------------------
# clocks sampler (B200_PROFILING.md "clocks line")
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    def __init__(self, index: int):
        self.index, self.samples, self._stop, self._thr = index, [], threading.Event(), None

    def start(self):
        def run():
            q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
                 "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
                 "clocks_event_reasons.sw_power_cap")
            while not self._stop.is_set():
                try:
                    out = subprocess.run(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}",
                                          "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                    parts = [p.strip() for p in out.strip().split(",")]
                    if len(parts) >= 7:
                        self.samples.append(parts)
                except Exception:
                    pass
                self._stop.wait(0.2)
        self._thr = threading.Thread(target=run, daemon=True)
        self._thr.start()

    def stop(self):
        self._stop.set()
        if self._thr:
            self._thr.join(timeout=3)
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        sm = sorted(float(s[0]) for s in self.samples)
        reasons = []
        for i, name in enumerate(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]):
            if any(s[3 + i].lower().startswith("active") for s in self.samples):
                reasons.append(name)
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": float(self.samples[0][1]), "reasons": reasons,
                "power_w_max": max(float(s[2]) for s in self.samples), "samples": len(self.samples)}


# ------------------------------------------------------------------------------------------------
# workload
# ------------------------------------------------------------------------------------------------
def build_chunks(cfg, seconds, size, seed):
    """Pre-processes one synthetic stream into per-chunk host inputs (what live_cc does per chunk)."""
    from livecc_b200.livecc_utils import get_smart_resized_clip, get_smart_resized_video_reader
    from livecc_b200.processing import StubProcessor

    proc = StubProcessor(cfg)
    nframes = seconds * 2
    path = f"synthetic://{nframes * 15}x{size}x{size}@30?seed={seed}"
    reader, H, W = get_smart_resized_video_reader(path, 384 * 28 * 28)
    reader.get_frame_timestamp(0)
    pts = torch.from_numpy(reader._frame_pts[:, 1])
    ts_all = torch.arange(0.0, seconds, 0.5)
    clip, ts, idxs = get_smart_resized_clip(reader, H, W, ts_all, pts, 0)
    chunks = [clip[:6]] + list(clip[6:].split(2))
    tss = [ts[:6]] + list(ts[6:].split(2))
    out = []
    off = None
    for i, (c, t) in enumerate(zip(chunks, tss)):
        content = [{"type": "text", "text": f"Time={t[0].item():.1f}-{t[-1].item() + 0.5:.1f}s"},
                   {"type": "video", "video": c}]
        if i == 0:
            content.append({"type": "text", "text": "Please describe the video."})
        text = proc.apply_chat_template([{"role": "user", "content": content}], tokenize=False, add_generation_prompt=True)
        if off is None:
            off = text.index("<|im_start|>user")
        if i > 0:
            text = "<|im_end|>\n" + text[off:]
        out.append(proc(text=text, videos=[c], return_attention_mask=False))
    return out, path


def run_stream_device(eng, chunks_dev, max_new, keep_cache=False):
    """Device-resident inputs: one generate() per chunk, ids threaded on the device. keep_cache: the last chunk's
    GenerateOutput (its cache not released) is returned as a fifth value."""
    cache, past_ids = None, None
    n_tok = n_frames = 0
    lat = []
    for ch in chunks_dev:
        t0 = time.perf_counter()
        ids = ch["input_ids"] if past_ids is None else torch.cat([past_ids, ch["input_ids"]], dim=1)
        out = eng.generate(input_ids=ids, pixel_values_videos=ch["pixel_values_videos"],
                           video_grid_thw=ch["video_grid_thw"], past_key_values=cache, return_dict_in_generate=True,
                           do_sample=False, repetition_penalty=1.05, max_new_tokens=max_new,
                           pad_token_id=eng.config.eos_token_id)
        cache, past_ids = out.past_key_values, out.sequences[:, :-1]
        n_tok += out.sequences.shape[1] - ids.shape[1]
        n_frames += ch["frames"]
        lat.append((time.perf_counter() - t0) / ch["frames"])
    kv = cache.get_seq_length()
    if keep_cache:
        return n_tok, n_frames, lat, kv, out
    cache.release()
    return n_tok, n_frames, lat, kv


def run_streams_batched(eng, chunks_dev, max_new, B, n_chunks=None):
    """B concurrent streams on ONE GPU through generate_batch (SURVEY.md §8(f) rank 2): per chunk the ViT and the prefill
    run per stream, the decode steps run batched in the persistent kernel (weights read once per step for all B)."""
    caches, pasts = [None] * B, [None] * B
    n_tok = n_frames = 0
    for ch in chunks_dev[:n_chunks]:
        reqs = []
        for b in range(B):
            ids = ch["input_ids"] if pasts[b] is None else torch.cat([pasts[b], ch["input_ids"]], dim=1)
            reqs.append(dict(input_ids=ids, pixel_values_videos=ch["pixel_values_videos"], video_grid_thw=ch["video_grid_thw"],
                             past_key_values=caches[b]))
        outs = eng.generate_batch(reqs, repetition_penalty=1.05, max_new_tokens=max_new, do_sample=False)
        for b, o in enumerate(outs):
            caches[b], pasts[b] = o.past_key_values, o.sequences[:, :-1]
            n_tok += o.sequences.shape[1] - reqs[b]["input_ids"].shape[1]
            n_frames += ch["frames"]
    for c in caches:
        c.release()
    return n_tok, n_frames


_E2E_RUN = [0]


def run_stream_e2e(infer, path, seconds, max_new):
    """The public API, driven like REF/demo/cli.py:13-24; frames start on the host. Every run is a new
    stream = a new video path (the reference caches readers and pts per path)."""
    _E2E_RUN[0] += 1
    path = f"{path}{_E2E_RUN[0]:03d}"
    state = {"video_path": path}
    n_tok = n_frames = 0
    h2d = d2h = 0
    lat = []
    n0 = len(infer.timings)
    for t in range(seconds + 1):
        state["video_timestamp"] = t
        for (_s, _e), _resp, state in infer.live_cc(message="Please describe the video.", state=state,
                                                    max_pixels=384 * 28 * 28, repetition_penalty=1.05,
                                                    do_sample=False, max_new_tokens=max_new):
            pass
        if state.get("video_end", False):
            break
    for rec in infer.timings[n0:]:
        n_tok += rec["new_tokens"]
        n_frames += rec["frames"]
        lat.append((rec["generate_s"] + rec["preprocess_s"] + rec["ingest_s"]) / rec["frames"])
    v = infer.model.config.vision_config
    for rec in infer.timings[n0:]:
        h2d += rec["frames"] * 3 * infer._last_hw[0] * infer._last_hw[1] + 8 * 64  # uint8 frames + new ids
        d2h += 8 * (rec["new_tokens"] + 1) + 32
    kv = state["past_key_values"].get_seq_length()
    state["past_key_values"].release()
    return n_tok, n_frames, lat, kv, h2d, d2h


KV_SAMPLE_TOKENS = 256


def dump_outputs(out_dir, out):
    """What one stream's last generate() call hands its caller: `sequences` (every prompt and generated id of the whole
    stream, as the ids are threaded through the chunks) and the KV cache. The cache is sampled: the K and V rows of
    KV_SAMPLE_TOKENS positions drawn with a fixed seed, all layers and heads, [layers, kv_heads, tokens, 128] (7B: 29 MB
    in all). Everything is written as float64 (ids, positions) or float32 (cache, exact for bf16)."""
    import numpy as np

    os.makedirs(out_dir, exist_ok=True)
    cache = out.past_key_values
    n = cache.get_seq_length()
    g = torch.Generator().manual_seed(0)
    pos = torch.randperm(n, generator=g)[:min(KV_SAMPLE_TOKENS, n)].sort().values
    idx = pos.to(cache.pool.device)
    ks, vs = zip(*(cache.gather(layer) for layer in range(cache.pool.layers)))
    arrays = {"sequences": out.sequences.double(), "kv_positions": pos.double(),
              "kv_keys_sample": torch.stack([k[:, idx] for k in ks]).float(),
              "kv_values_sample": torch.stack([v[:, idx] for v in vs]).float()}
    total = sum(a.numel() * a.element_size() for a in arrays.values())
    assert total <= 64 << 20, f"output dump of {total} bytes exceeds 64 MB"
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), a.cpu().numpy())


# ------------------------------------------------------------------------------------------------
# roofline of the dominant kernel
# ------------------------------------------------------------------------------------------------
def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def recorded_pool_peak():
    """The driver-measured HBM figure BASELINE.md §2 quotes from MEASURED_PEAKS.json (GB/s), or None. Only used to annotate
    the roofline blocks when MEASURED_PEAKS.json itself is absent from the snapshot (the fractions then use the fallback)."""
    import re

    try:
        m = re.search(r"HBM copy bandwidth\s*\|\s*([0-9.]+)\s*GB/s", open(os.path.join(ROOT, "BASELINE.md")).read())
        return float(m.group(1)) if m else None
    except OSError:
        return None


def time_gateup_kernel(eng, iters=5):
    """decode gate/up GEMV (gemv_rows_kernel<2,true,SWIGLU>): fused RMSNorm + [2I,H] weight stream + SwiGLU.
    Algorithmic bytes/launch = 2I*H*2 (weights) + H*2 (x) + H*2 (norm w) + I*2 (out). Cycles through all layers
    so every launch streams a different 271 MB (7B) weight, i.e. inputs >> L2."""
    t = eng.config.text_config
    H, I = t.hidden_size, t.intermediate_size
    x = torch.randn(H, device=eng.device).to(torch.bfloat16)
    stream = torch.cuda.current_stream()
    for lw in eng.weights.layers:  # warm-up
        eng.ctx.gemv_norm_swiglu(lw.gate_up_w, x, lw.ln2_w, t.rms_norm_eps)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    n = 0
    e0.record(stream)
    for _ in range(iters):
        for lw in eng.weights.layers:
            eng.ctx.gemv_norm_swiglu(lw.gate_up_w, x, lw.ln2_w, t.rms_norm_eps)
            n += 1
    e1.record(stream)
    torch.cuda.synchronize()
    sec = e0.elapsed_time(e1) / 1e3 / n
    nbytes = 2 * I * H * 2 + 2 * H * 2 + I * 2
    return nbytes, sec



def time_persistent_kernel(eng, chunks_dev, max_new, iters=20):
    """The persistent decode kernel (decode_mega_kernel; what every batched step runs): one launch = one decode step of one
    stream (28 layers + lm_head).
    Timed alone with CUDA events on its launch stream (the sub-range hook of the C ABI launches exactly the kernel the
    CUDA-graph step contains, without the token selection, so the stream state does not advance and every launch
    re-reads the same bytes): algorithmic bytes per launch = all decoder weights + lm_head + the stream's KV at the
    clip's final length (SURVEY.md §8(d)); inputs (14 GB) >> L2 (126 MB)."""
    from livecc_b200 import _cabi

    t = eng.config.text_config
    _, _, _, kv, out = run_stream_device(eng, chunks_dev, max_new, keep_cache=True)
    cache = out.past_key_values
    with torch.inference_mode():
        cache.scalars[_cabi.SC_FINISHED] = 0
    st = [cache.stream_state()]
    L = t.num_hidden_layers
    stream = torch.cuda.current_stream()
    for _ in range(3):
        eng._native.decode_mega_debug(st, 0, L, 31, 1)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(iters):
        eng._native.decode_mega_debug(st, 0, L, 31, 1)
    e1.record(stream)
    torch.cuda.synchronize()
    sec = e0.elapsed_time(e1) / 1e3 / iters
    err = eng._native.mega_error()
    cache.release()
    weight_bytes = (L * ((t.num_attention_heads + 2 * t.num_key_value_heads) * 128 * t.hidden_size + t.hidden_size * t.hidden_size
                         + 3 * t.intermediate_size * t.hidden_size + 2 * t.hidden_size) + t.hidden_size
                    + t.vocab_size * t.hidden_size) * 2
    kv_bytes = 2 * L * t.num_key_value_heads * 128 * 2 * kv
    return weight_bytes + kv_bytes, sec, kv, err


def time_ingest_kernel(eng, peak, iters=20):
    """GPU frame ingest (SURVEY.md §8(f) rank 1): resize_bicubic_aa_u8_kernel on a 2-frame 1080p chunk -> 448x796 (what
    get_smart_resized_clip does for a 16:9 source, video_process_patch.py:150-155), rotated over > L2 of distinct clips,
    CUDA events; beside it the reference's host call (torchvision, all host threads) on the same clip, and whether the
    two results are identical. Algorithmic bytes = source + destination planes; the kernel is fp32-issue bound."""
    import time

    from torchvision.transforms import InterpolationMode
    from torchvision.transforms import functional as TF

    T, h, w, H, W = 2, 1080, 1920, 448, 796
    ctx = eng.ctx
    g = torch.Generator().manual_seed(0)
    host = torch.randint(0, 256, (T, 3, h, w), generator=g, dtype=torch.uint8)
    n = int(160e6 // host.numel()) + 1
    clips = [host.cuda()] + [torch.randint(0, 256, (T, 3, h, w), dtype=torch.uint8, device="cuda") for _ in range(n - 1)]
    out = ctx.resize_bicubic_aa_u8(clips[0], (H, W))
    for c in clips:
        ctx.resize_bicubic_aa_u8(c, (H, W), out=torch.empty_like(out))
    torch.cuda.synchronize()
    stream = torch.cuda.current_stream()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    scratch = torch.empty_like(out)
    e0.record(stream)
    for i in range(iters):
        ctx.resize_bicubic_aa_u8(clips[i % n], (H, W), out=scratch)
    e1.record(stream)
    torch.cuda.synchronize()
    us = e0.elapsed_time(e1) * 1e3 / iters
    TF.resize(host, [H, W], interpolation=InterpolationMode.BICUBIC, antialias=True)
    t0 = time.perf_counter()
    ref = TF.resize(host, [H, W], interpolation=InterpolationMode.BICUBIC, antialias=True)
    cpu_ms = (time.perf_counter() - t0) * 1e3
    nbytes = T * 3 * (h * w + H * W)
    return {"kernel": "resize_bicubic_aa_u8_kernel (bicubic antialias uint8 resize, both passes fused)",
            "workload": "2 frames 3x1080x1920 -> 3x448x796 uint8", "us_per_launch": us, "bytes_per_launch": nbytes,
            "achieved": nbytes / us / 1e3, "unit": "GB/s", "frac": nbytes / us / 1e3 / peak, "bound": "fp32 issue (22 taps/pixel); HBM frac reported",
            "host_torchvision_ms": cpu_ms, "host_threads": torch.get_num_threads(),
            "identical_to_torchvision": bool(torch.equal(out.cpu(), ref))}


# ------------------------------------------------------------------------------------------------
# CPU reference arm (HF eager fp32 on host cores)
# ------------------------------------------------------------------------------------------------
def cpu_reference_sample(cfg, size, max_new=16, steps=1, warmup=0, budget_s=150.0):
    """The reference's own CPU path: transformers Qwen2VLForConditionalGeneration, fp32, eager attention, through
    oracle/hf_oracle.py. Bounded sample = one steady-state streaming second: a fresh stream's turn with ONE 2-frame
    chunk at size x size (ViT on 1024 patches + prefill of ~281 tokens) and `max_new` = 16 greedy tokens
    (repetition_penalty 1.05), i.e. the per-chunk work of REF/demo/infer.py:165-172 at KV length ~300 (the CPU cost per
    chunk is dominated by the 7B weights, not by the KV length, so this does not flatter the GPU arm). Threads:
    min(host cores, 32) — oversubscribing a 128-core box made the eager path several times slower. Stops early once
    `budget_s` of samples were timed."""
    from livecc_b200.checkpoint import synthetic_tensors
    from livecc_b200.processing import StubProcessor
    from oracle.hf_oracle import build_hf_model, hf_generate_chunk

    ncores = os.cpu_count() or 1
    nthreads = max(1, min(ncores, int(os.environ.get("LIVECC_CPU_THREADS", "32"))))
    torch.set_num_threads(nthreads)
    gen_dev = "cuda" if torch.cuda.is_available() else "cpu"
    model = build_hf_model(cfg, synthetic_tensors(cfg, 1234, torch.float32, "cpu", gen_device=gen_dev),
                           dtype=torch.float32, device="cpu", attn_implementation="eager")
    proc = StubProcessor(cfg)
    g = torch.Generator().manual_seed(0)
    clip = torch.randint(0, 256, (2, 3, size, size), generator=g, dtype=torch.uint8)
    content = [{"type": "text", "text": "Time=0.0-1.0s"}, {"type": "video", "video": clip},
               {"type": "text", "text": "Please describe the video."}]
    text = proc.apply_chat_template([{"role": "user", "content": content}], tokenize=False, add_generation_prompt=True)
    times, toks = [], 0
    spent = 0.0
    for i in range(warmup + steps):
        inputs = proc(text=text, videos=[clip], return_attention_mask=False)
        model.model.rope_deltas = None
        t0 = time.perf_counter()
        out, L = hf_generate_chunk(model, inputs, None, None, max_new_tokens=max_new)
        dt = time.perf_counter() - t0
        spent += dt
        if i >= warmup or spent > budget_s:
            times.append(dt)
            toks = out.sequences.shape[1] - L
        if spent > budget_s:
            break
    sec = sum(times) / len(times)
    return {"tokens_per_s": toks / sec, "frames_per_s": 2 / sec, "sec_per_sample": sec, "cores": nthreads,
            "host_cores": ncores, "tokens": toks, "timed_samples": len(times),
            "sample": f"one streaming chunk of a fresh stream: 2 frames {size}x{size} (ViT 1024 patches + prefill) + {toks} "
                      f"greedy tokens (max_new_tokens=16 as REF/demo/infer.py:170), fp32 eager, {nthreads} threads, "
                      f"{len(times)} timed sample(s); tokens/s = {toks} / seconds per chunk"}


# ------------------------------------------------------------------------------------------------
# "kernel to beat": the reference's own GPU path (HF bf16 + flash_attention_2 [+ liger]) on the same B200
# ------------------------------------------------------------------------------------------------
def run_hf_gpu(args, cfg, config, dev):
    """REF/demo/infer.py:43-47,165-172 with the installed transformers / flash-attn (/ liger_kernel) stack: same
    synthetic checkpoint, same clip, same per-chunk generate() arguments, inputs resident on the device. Per-phase device
    time from CUDA events around the vision tower and the language-model forwards (prefill = S > 1, decode = S == 1)."""
    from livecc_b200.checkpoint import synthetic_tensors
    from oracle.hf_oracle import build_hf_model, hf_generate_chunk, oracle_variant

    tensors = synthetic_tensors(cfg, 1234, torch.bfloat16, dev, gen_device=dev)
    impl = "flash_attention_2"
    try:
        model = build_hf_model(cfg, tensors, dtype=torch.bfloat16, device=dev, attn_implementation=impl, liger=args.liger)
    except Exception as e:  # noqa: BLE001
        print(json.dumps({"impl": "hf_gpu", "unavailable": f"{type(e).__name__}: {e}"}))
        return 0
    chunks, _ = build_chunks(cfg, args.seconds, args.size, seed=0)
    chunks = [dict(input_ids=c.input_ids.to(dev), pixel_values_videos=c.pixel_values_videos.to(dev),
                   video_grid_thw=c.video_grid_thw.to(dev), frames=int(c.video_grid_thw[0, 0]) * 2) for c in chunks]
    ev = {"vit": [], "prefill": [], "decode": []}

    def hook(kind_of):
        def pre(mod, a, kw):
            e = torch.cuda.Event(enable_timing=True)
            e.record()
            mod._lcc_e0 = (e, kind_of(a, kw))

        def post(mod, a, kw, out):
            e1 = torch.cuda.Event(enable_timing=True)
            e1.record()
            e0, kind = mod._lcc_e0
            ev[kind].append((e0, e1))
        return pre, post

    def lm_kind(a, kw):
        x = kw.get("inputs_embeds")
        x = x if x is not None else kw.get("input_ids")
        return "decode" if x is not None and x.shape[1] == 1 else "prefill"

    pre, post = hook(lambda a, kw: "vit")
    model.model.visual.register_forward_pre_hook(pre, with_kwargs=True)
    model.model.visual.register_forward_hook(post, with_kwargs=True)
    pre, post = hook(lm_kind)
    model.model.language_model.register_forward_pre_hook(pre, with_kwargs=True)
    model.model.language_model.register_forward_hook(post, with_kwargs=True)

    def one_stream():
        kv = past = None
        model.model.rope_deltas = None
        tok = frames = 0
        lat = []
        for ch in chunks:
            t0 = time.perf_counter()
            out, L = hf_generate_chunk(model, ch, kv, past, max_new_tokens=args.max_new_tokens)
            kv, past = out.past_key_values, out.sequences[:, :-1]
            tok += out.sequences.shape[1] - L
            frames += ch["frames"]
            torch.cuda.synchronize()
            lat.append((time.perf_counter() - t0) / ch["frames"])
        return tok, frames, lat, kv.get_seq_length()

    for _ in range(args.warmup):
        one_stream()
    for v in ev.values():
        v.clear()
    torch.cuda.synchronize()
    sampler = ClockSampler(dev.index or 0)
    sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    tok = frames = 0
    lat = []
    for _ in range(args.steps):
        a, b, c, kv_end = one_stream()
        tok += a
        frames += b
        lat += c
    e1.record()
    torch.cuda.synchronize()
    sec = e0.elapsed_time(e1) / 1e3
    clocks = sampler.stop()
    n_chunks = len(chunks) * args.steps
    ph = {k: sum(a.elapsed_time(b) for a, b in v) for k, v in ev.items()}
    lat.sort()
    line = {"impl": "hf_gpu", "variant": oracle_variant(impl), "metric": METRIC, "value": tok / sec, "unit": "tokens/s",
            "n_gpus": 1, "steps": args.steps, "warmup": args.warmup, "ms_per_step": sec / args.steps * 1e3,
            "higher_is_better": True, "dtype": "bf16", "data": "synthetic", "config": config,
            "frames_per_s": frames / sec, "p50_frame_latency_ms": lat[len(lat) // 2] * 1e3, "kv_len_end": kv_end,
            "clocks": clocks,
            "phases_ms_per_chunk": {"vit": ph["vit"] / n_chunks, "prefill": ph["prefill"] / n_chunks,
                                    "decode": ph["decode"] / n_chunks,
                                    "host_and_other": sec * 1e3 / n_chunks - sum(ph.values()) / n_chunks},
            "decode_ms_per_step": ph["decode"] / max(len(ev["decode"]), 1)}
    print(json.dumps(line))
    return 0


# ------------------------------------------------------------------------------------------------
def main():
    args = parse_args()
    from livecc_b200 import runner  # the repo's own multi-GPU plumbing (rank env, NCCL init, barrier + device sync)

    rank, world, local_rank = runner.dist_env()
    cfg = get_config(args.model)
    workload = (f"LiveCC-{'7B' if args.model == '7b' else 'small'} streaming 2fps {args.seconds}s clip "
                f"({args.seconds * 2} frames) {args.size}x{args.size} greedy decode bf16, one stream per GPU")
    config = {"workload": workload, "chunks": 1 + (args.seconds * 2 - 6) // 2, "max_new_tokens": args.max_new_tokens,
              "repetition_penalty": 1.05, "l2": "inputs larger than L2 (bf16 weights streamed once per token/chunk)",
              "parallelism": f"dp{world} (independent streams, no data-path collective)"}

    if args.impl == "reference":
        if rank != 0:
            return 0
        r = cpu_reference_sample(cfg, args.size, max_new=args.max_new_tokens, steps=max(1, args.steps), warmup=min(args.warmup, 1))
        line = {"impl": "reference", "metric": METRIC, "value": r["tokens_per_s"], "unit": "tokens/s", "n_gpus": args.gpus,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": r["sec_per_sample"] * 1e3,
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": config, "frames_per_s": r["frames_per_s"],
                "cpu_baseline": {"value": r["tokens_per_s"], "unit": "tokens/s", "cores": r["cores"], "kind": "reference",
                                 "sample": r["sample"]},
                "e2e": {"value": r["tokens_per_s"], "unit": "tokens/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "gpu_launches": 0}
        print(json.dumps(line))
        return 0

    assert torch.cuda.is_available(), "bench.py needs a B200; there is no CPU fallback for the native arm"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if args.impl == "hf_gpu":
        return run_hf_gpu(args, cfg, config, dev) if rank == 0 else 0
    import torch.distributed as dist

    runner.init_distributed("nccl", device=dev)  # no-op for one rank

    from livecc_b200.engine import LiveCCB200ForConditionalGeneration
    from livecc_b200.streaming import LiveCCDemoInfer

    eng = LiveCCB200ForConditionalGeneration.from_synthetic(cfg, seed=1234, device=f"cuda:{local_rank}")
    chunks, path = build_chunks(cfg, args.seconds, args.size, seed=rank)
    chunks_dev = [dict(input_ids=c.input_ids.to(dev), pixel_values_videos=c.pixel_values_videos.to(dev),
                       video_grid_thw=c.video_grid_thw, frames=int(c.video_grid_thw[0, 0]) * 2) for c in chunks]
    from livecc_b200.processing import StubProcessor

    infer = LiveCCDemoInfer(model=eng, processor=StubProcessor(cfg, emit_frames=True))  # uint8 frames, GPU ingest
    infer._last_hw = (args.size, args.size)

    barrier = runner.barrier  # dist.barrier() when initialised, then torch.cuda.synchronize()

    # ---- device-resident arm ----
    for _ in range(args.warmup):
        run_stream_device(eng, chunks_dev, args.max_new_tokens)
    barrier()
    sampler = ClockSampler(local_rank)
    sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    tok = frames = 0
    lat = []
    kv_end = 0
    for k in eng.phase_ms_total:
        eng.phase_ms_total[k] = 0
    launches0 = eng.kernel_launches()
    last_out = None
    for i in range(args.steps):
        keep = args.dump_outputs is not None and rank == 0 and i == args.steps - 1
        a, b, c, kv_end, *kept = run_stream_device(eng, chunks_dev, args.max_new_tokens, keep_cache=keep)
        last_out = kept[0] if kept else None
        tok += a
        frames += b
        lat += c
    e1.record()
    barrier()
    gpu_launches = eng.kernel_launches() - launches0  # counted at the library's launch sites (+ graph nodes per replay)
    sec = e0.elapsed_time(e1) / 1e3
    clocks = sampler.stop()
    phases = dict(eng.phase_ms_total)
    if last_out is not None:
        dump_outputs(args.dump_outputs, last_out)
        last_out.past_key_values.release()

    # ---- end-to-end arm (public API, host frames) ----
    e2e = None
    if not args.no_e2e:
        for _ in range(max(1, min(args.warmup, 1))):
            run_stream_e2e(infer, path, args.seconds, args.max_new_tokens)
        barrier()
        t0 = time.perf_counter()
        e_tok = e_frames = h2d = d2h = 0
        e_lat = []
        for _ in range(args.steps):
            a, b, c, _kv, hb, db = run_stream_e2e(infer, path, args.seconds, args.max_new_tokens)
            e_tok += a
            e_frames += b
            e_lat += c
            h2d += hb
            d2h += db
        barrier()
        e_sec = time.perf_counter() - t0
        e2e = dict(tok=e_tok, frames=e_frames, sec=e_sec, lat=e_lat, h2d=h2d // args.steps, d2h=d2h // args.steps)

    # ---- reduce over ranks: sum of units, max of time ----
    stats = torch.tensor([tok, frames, sec, e2e["tok"] if e2e else 0, e2e["frames"] if e2e else 0,
                          e2e["sec"] if e2e else 0], dtype=torch.float64, device=dev)
    if world > 1:
        allst = [torch.zeros_like(stats) for _ in range(world)]
        dist.all_gather(allst, stats)
        allst = torch.stack(allst)
    else:
        allst = stats[None]
    tot_tok, tot_frames = allst[:, 0].sum().item(), allst[:, 1].sum().item()
    max_sec = allst[:, 2].max().item()
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return 0

    lat_sorted = sorted(lat)
    p50 = lat_sorted[len(lat_sorted) // 2] * 1e3
    peak, peak_src = load_peaks()
    kbytes, ksec = time_gateup_kernel(eng)
    pk_bytes, pk_sec, pk_kv, pk_err = time_persistent_kernel(eng, chunks_dev, args.max_new_tokens)
    traffic, traffic_src = None, None
    try:  # dram bytes of the same kernel from the committed `ncu --set full` capture (7B dims only)
        if args.model == "7b":
            tr = json.load(open(os.path.join(ROOT, "profiles", "r01_gateup_ncu.json")))
            traffic = tr["dram_bytes_read"] + tr["dram_bytes_write"]
            traffic_src = "static: one `ncu --set full` capture of this kernel (profiles/r01_gateup_ncu.json), not measured in this run"
    except Exception:
        traffic = None
    t = cfg.text_config
    step_weight_bytes = (t.num_hidden_layers * ((t.num_attention_heads + 2 * t.num_key_value_heads) * 128 * t.hidden_size
                                                + t.hidden_size * t.hidden_size + 3 * t.intermediate_size * t.hidden_size
                                                + 2 * t.hidden_size) + t.hidden_size + t.vocab_size * t.hidden_size) * 2
    n_chunks = len(chunks)
    line = {
        "metric": METRIC, "value": tot_tok / max_sec, "unit": "tokens/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": max_sec / args.steps * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "bf16", "data": "synthetic (hash-filled checkpoint, synthetic frames and token ids)",
        "config": config, "frames_per_s": tot_frames / max_sec, "p50_frame_latency_ms": p50,
        "kv_len_end": kv_end, "clocks": clocks, "gpu_launches": int(gpu_launches),
        "roofline": {"kernel": "gemv_rows_kernel<2,NORM,SWIGLU> (decode gate/up + RMSNorm + SwiGLU; largest share of the decode step)",
                     "bound": "hbm",
                     "achieved": kbytes / ksec / 1e9, "peak": peak, "peak_source": peak_src, "unit": "GB/s",
                     "frac": kbytes / ksec / 1e9 / peak, "traffic": traffic, "traffic_source": traffic_src,
                     "bytes_per_launch": kbytes,
                     "us_per_launch": ksec * 1e6},
    }
    line["persistent_kernel"] = {"kernel": "decode_mega_kernel (one launch = 28 layers + lm_head; the batched-decode kernel), 1 stream, "
                                           "kv_len %d" % pk_kv, "bytes_per_launch": pk_bytes, "us_per_launch": pk_sec * 1e6,
                                 "achieved": pk_bytes / pk_sec / 1e9, "unit": "GB/s", "frac": pk_bytes / pk_sec / 1e9 / peak,
                                 "native_error": pk_err}
    if world == 1:
        try:
            line["ingest"] = time_ingest_kernel(eng, peak)
        except Exception as ex:
            line["ingest"] = {"error": f"{type(ex).__name__}: {ex}"}
    if e2e:
        tot_e_tok, tot_e_frames = allst[:, 3].sum().item(), allst[:, 4].sum().item()
        max_e_sec = allst[:, 5].max().item()
        el = sorted(e2e["lat"])
        line["e2e"] = {"value": tot_e_tok / max_e_sec, "unit": "tokens/s", "frames_per_s": tot_e_frames / max_e_sec,
                       "p50_frame_latency_ms": el[len(el) // 2] * 1e3, "h2d_bytes_per_step": int(e2e["h2d"]),
                       "d2h_bytes_per_step": int(e2e["d2h"]),
                       "api": "LiveCCDemoInfer.live_cc (host uint8 frames -> H2D -> fused normalize+patchify -> generate -> D2H ids)"}
    # decode-step roofline inside the timed region: every generated token after the first of a chunk is one
    # CUDA-graph replay streaming all decoder weights + the stream's KV
    kv_bytes_tok = 2 * t.num_hidden_layers * t.num_key_value_heads * 128 * 2
    dsteps = max(int(phases["decode_steps"]), 1)
    ms_per_dstep = phases["decode"] / dsteps
    bytes_avg = step_weight_bytes + (kv_end / 2) * kv_bytes_tok  # KV grows ~linearly over the clip: mean length ~ end/2
    line["phases_ms_per_chunk"] = {"vit": phases["vit"] / max(phases["calls"], 1), "prefill": phases["prefill"] / max(phases["calls"], 1),
                                   "decode": phases["decode"] / max(phases["calls"], 1), "host_and_sync": max_sec * 1e3 / (args.steps * n_chunks)
                                   - (phases["vit"] + phases["prefill"] + phases["decode"]) / max(phases["calls"], 1)}
    line["roofline_step"] = {"unit_def": "one decode step (CUDA-graph replay): all decoder weights + lm_head + the stream's KV, "
                                         "timed with CUDA events inside the timed region",
                             "bound": "hbm", "bytes_per_step_mean": int(bytes_avg), "ms_per_step": ms_per_dstep,
                             "achieved": bytes_avg / (ms_per_dstep / 1e3) / 1e9, "peak": peak, "unit": "GB/s",
                             "frac": bytes_avg / (ms_per_dstep / 1e3) / 1e9 / peak, "decode_steps": dsteps}
    if peak_src.startswith("fallback"):
        rec = recorded_pool_peak()
        if rec:
            note = (f"MEASURED_PEAKS.json absent: fractions use the {peak:.0f} GB/s fallback; against the driver-measured "
                    f"{rec} GB/s recorded in BASELINE.md they are ")
            line["roofline"]["peak_note"] = note + f"{line['roofline']['achieved'] / rec:.4f}"
            line["roofline_step"]["peak_note"] = note + f"{line['roofline_step']['achieved'] / rec:.4f}"
    if not args.no_batch and world == 1:
        # multi-stream batching on one GPU: aggregate tokens/s of B concurrent streams over the same clip
        ms = {}
        for B in (2, 4, 8):
            run_streams_batched(eng, chunks_dev, args.max_new_tokens, B, n_chunks=3)  # warm-up: graphs, workspace
            torch.cuda.synchronize()
            eng.phase_ms_total.update(decode=0.0, decode_steps=0)
            b0, b1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            b0.record()
            a, b = run_streams_batched(eng, chunks_dev, args.max_new_tokens, B)
            b1.record()
            torch.cuda.synchronize()
            bs = b0.elapsed_time(b1) / 1e3
            ms[f"B{B}"] = {"tokens_per_s": a / bs, "frames_per_s": b / bs, "speedup_vs_B1": a / bs / (tot_tok / max_sec),
                           "decode_ms_per_step": eng.phase_ms_total["decode"] / max(eng.phase_ms_total["decode_steps"], 1)}
        line["multi_stream"] = {"api": "LiveCCB200ForConditionalGeneration.generate_batch (B streams, one GPU, one clip pass each)",
                                **ms}
    if not args.no_cpu_baseline and world == 1:
        try:
            r = cpu_reference_sample(cfg, args.size, max_new=args.max_new_tokens, steps=1, warmup=0, budget_s=60.0)
            line["cpu_baseline"] = {"value": r["tokens_per_s"], "unit": "tokens/s", "frames_per_s": r["frames_per_s"],
                                    "cores": r["cores"], "kind": "reference", "sample": r["sample"]}
        except Exception as ex:  # the baseline must never take the GPU number down with it
            line["cpu_baseline"] = {"value": None, "unit": "tokens/s", "cores": os.cpu_count(), "kind": "reference",
                                    "sample": f"failed: {type(ex).__name__}: {ex}"}
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
