"""CPU suite, part 2: C-ABI exports, host orchestration (streaming mirror with a mock model, page pool,
livecc_utils surface) and the world_size-2 gloo path of the multi-GPU runner. No GPU compute."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from livecc_b200 import _cabi
from livecc_b200.config import LiveCCConfig
from livecc_b200.processing import StubProcessor

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_loads_and_exports_every_header_symbol():
    lib = _cabi.load_library()
    syms = _cabi.header_symbols()
    assert len(syms) >= 28 and "lcc_gemm_bf16" in syms and "lcc_decode_steps" in syms
    for s in syms:
        assert hasattr(lib, s), f"liblivecc_sm100a.so does not export {s}"
    assert lib.lcc_abi_version() == _cabi.ABI_VERSION
    # sm_100a code only, with the Blackwell instructions the design relies on
    sass = subprocess.run(["cuobjdump", "-sass", str(_cabi.LIB_PATH)], capture_output=True, text=True).stdout
    if sass:
        assert "sm_100a" in sass and "UTCHMMA" in sass and "UTMALDG" in sass and "LDTM" in sass


def test_product_path_fails_loudly_without_a_gpu():
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from livecc_b200.engine import LiveCCB200ForConditionalGeneration

    with pytest.raises(Exception):
        _cabi.Context(0)
    with pytest.raises(Exception):
        LiveCCB200ForConditionalGeneration.from_synthetic(LiveCCConfig.small(), device="cuda")
    # and nothing in the product imports the oracle
    for dirpath, _, files in os.walk(os.path.join(ROOT, "livecc_b200")):
        for f in files:
            if f.endswith(".py"):
                src = open(os.path.join(dirpath, f)).read()
                assert "import oracle" not in src and "from oracle" not in src, f


class MockCache:
    def __init__(self):
        self.n = 0

    def get_seq_length(self):
        return self.n


class MockModel:
    """Records generate() calls; emits 3 fixed tokens (the last one EOS)."""

    def __init__(self, cfg):
        self.config, self.device, self.calls = cfg, torch.device("cpu"), []
        self.prepare_inputs_for_generation = None

    def generate(self, input_ids=None, pixel_values_videos=None, video_grid_thw=None, past_key_values=None,
                 max_new_tokens=16, **kw):
        cache = past_key_values or MockCache()
        self.calls.append(dict(L=input_ids.shape[1], past=cache.n,
                               grid=video_grid_thw.tolist() if video_grid_thw is not None else [],
                               rows=pixel_values_videos.shape[0] if pixel_values_videos is not None else 0, kw=kw,
                               new=input_ids[0, cache.n:].tolist()))
        gen = torch.tensor([[1234, 1235, self.config.eos_token_id]])
        seq = torch.cat([input_ids, gen], 1)
        cache.n = seq.shape[1] - 1

        class Out:
            sequences = seq
        Out.past_key_values = cache
        return Out


def test_live_cc_chunk_schedule_and_state_contract():
    """REF/demo/infer.py:105-180 driven like REF/demo/cli.py:13-24."""
    from livecc_b200.streaming import LiveCCDemoInfer

    cfg = LiveCCConfig.small()
    model = MockModel(cfg)
    infer = LiveCCDemoInfer(model=model, processor=StubProcessor(cfg))
    state = {"video_path": "synthetic://300x112x140@30?seed=3"}  # 10 s of video
    outs = []
    for t in range(12):
        state["video_timestamp"] = t
        for (s, e), resp, state in infer.live_cc(message="Please describe the video.", state=state,
                                                  repetition_penalty=1.05, streaming_eos_base_threshold=0.0,
                                                  streaming_eos_threshold_step=0):
            outs.append((s, e, resp))
        if state.get("video_end", False):
            break
    frames = [c["grid"][0][0] * 2 for c in model.calls]
    assert frames[0] == 6 and all(f == 2 for f in frames[1:]) and sum(frames) == 20
    assert outs[0][:2] == (0.0, 3.0) and outs[1][:2] == (3.0, 4.0)
    n_calls = len(model.calls)
    state["video_timestamp"] = 30  # past the end: nothing more to process (REF/demo/infer.py:100-109)
    assert list(infer.live_cc(message="", state=state)) == [] and len(model.calls) == n_calls
    # ids: full history is re-sent every turn; cache length == len(past_ids)
    for prev, cur in zip(model.calls, model.calls[1:]):
        assert cur["past"] == prev["L"] + 2 and cur["L"] > cur["past"]
        assert cur["new"][:2] == [cfg.eos_token_id, cfg.newline_token_id]       # '<|im_end|>\n' glue
        assert cur["new"].count(cfg.video_token_id) == cur["rows"] // 4
    first = model.calls[0]
    # 112x140 is below VIDEO_MIN_PIXELS (100*28*28) -> smart_resize upscales to 252x336 (18x24 patches per frame pair)
    assert first["rows"] == 3 * 18 * 24 and first["new"].count(cfg.video_token_id) == first["rows"] // 4
    assert "logits_processor" in first["kw"] and first["kw"]["logits_processor"][0].token_id == infer.streaming_eos_token_id
    assert state["past_ids"].shape[1] == state["past_key_values"].get_seq_length()
    assert len(infer.timings) == len(model.calls)


def test_video_qa_and_offline_eval_variants():
    """REF/demo/infer.py:183-242 (video_qa) and :245-310 (live_cc_once_for_evaluation) on the mock model."""
    from livecc_b200.streaming import LiveCCDemoInfer

    cfg = LiveCCConfig.small()
    model = MockModel(cfg)
    infer = LiveCCDemoInfer(model=model, processor=StubProcessor(cfg))
    state = {"video_path": "synthetic://240x56x84@30?seed=5"}  # 8 s
    resp, state = infer.video_qa("What happens?", [], state)
    first = model.calls[-1]
    assert first["past"] == 0 and first["grid"][0][0] >= 2 and first["kw"]["do_sample"] is False
    n_video = first["new"].count(cfg.video_token_id)
    assert n_video == first["rows"] // 4 and "max_new_tokens" not in first["kw"]
    resp2, state = infer.video_qa("And then?", [], state)
    second = model.calls[-1]
    assert second["past"] == first["L"] + 2 and second["new"].count(cfg.video_token_id) == 0  # video only once
    assert state["past_ids"].shape[1] == state["past_key_values"].get_seq_length()

    model2 = MockModel(cfg)
    infer2 = LiveCCDemoInfer(model=model2, processor=StubProcessor(cfg))
    out = infer2.live_cc_once_for_evaluation("Describe.", "synthetic://300x56x84@30?seed=6", video_start=0, video_end=None)
    frames = [c["grid"][0][0] * 2 for c in model2.calls]
    assert frames[0] == 6 and all(f == 2 for f in frames[1:]) and len(out) == len(frames)
    assert out[0][:2] == [0, 3.0] and out[1][:2] == [3.0, 4.0]


def test_processor_frame_passthrough():
    cfg = LiveCCConfig.small()
    clip = torch.randint(0, 256, (3, 3, 56, 84), dtype=torch.uint8)
    text = StubProcessor(cfg).apply_chat_template([{"role": "user", "content": [{"type": "video", "video": clip}]}],
                                                  tokenize=False, add_generation_prompt=True)
    a = StubProcessor(cfg)(text=text, videos=[clip], return_attention_mask=False)
    b = StubProcessor(cfg, emit_frames=True)(text=text, videos=[clip], return_attention_mask=False)
    assert torch.equal(a.input_ids, b.input_ids) and torch.equal(a.video_grid_thw, b.video_grid_thw)
    assert b.video_frames.dtype == torch.uint8 and b.video_frames.shape == (3, 3, 56, 84) and "pixel_values_videos" not in b
    # float frames (video_qa path) fall back to host patch rows
    c = StubProcessor(cfg, emit_frames=True)(text=text, videos=[clip.float()], return_attention_mask=False)
    assert "pixel_values_videos" in c and torch.equal(c.pixel_values_videos, a.pixel_values_videos)


def test_livecc_utils_surface():
    import livecc_b200.livecc_utils as U

    assert set(U.__all__) == {"prepare_multiturn_multimodal_inputs_for_generation", "_read_video_decord_plus",
                              "_spatial_resize_video", "get_smart_resized_video_reader", "get_smart_resized_clip"}
    reader, H, W = U.get_smart_resized_video_reader("synthetic://90x448x448@30?seed=1", 384 * 28 * 28)
    assert (H, W) == (448, 448)
    reader.get_frame_timestamp(0)
    pts = torch.from_numpy(reader._frame_pts[:, 1])
    clip, ts, idxs = U.get_smart_resized_clip(reader, H, W, torch.arange(0.0, 2.5, 0.5), pts, 0)
    assert clip.shape == (6, 3, 448, 448) and clip.dtype == torch.uint8 and len(idxs) == 6  # padded to FRAME_FACTOR, then fits
    clip2, fps = U._read_video_decord_plus({"video": "synthetic://300x56x84@30?seed=2"})
    assert clip2.shape[0] % 2 == 0 and clip2.shape[1:] == (3, 56, 84)
    with pytest.raises(ValueError):
        U._read_video_decord_plus({"video": "/nonexistent.mp4", "remote_loader": None})
    # generation patch semantics (generation_patch.py:35-39)
    cfg = LiveCCConfig.small()

    class M:
        config = cfg
    cache = MockCache()
    cache.n = 4
    ids = torch.tensor([[1, 2, 3, 4, 5, cfg.video_token_id, 6]])
    out = U.prepare_multiturn_multimodal_inputs_for_generation(M, ids, past_key_values=cache, pixel_values_videos="px")
    assert out["pixel_values_videos"] == "px" and out["position_ids"] is None and out["input_ids"].shape[1] == 3
    out = U.prepare_multiturn_multimodal_inputs_for_generation(M, ids[:, :5], past_key_values=cache, pixel_values_videos="px")
    assert out["pixel_values_videos"] is None


def test_page_pool_and_cache_bookkeeping():
    from livecc_b200.kv_cache import PagedKVCache, PagePool

    pool = PagePool(layers=2, kv_heads=2, device="cpu", initial_pages=4)
    a, b = PagedKVCache(pool), PagedKVCache(pool)
    a.ensure_tokens(130)  # 3 pages
    b.ensure_tokens(64)   # 1 page
    assert len(a.pages) == 3 and len(b.pages) == 1 and not set(a.pages) & set(b.pages) and len(pool.free) == 0
    gen0 = pool.generation
    pool.k[0, a.pages[0], 0, 0, 0] = 7.0
    b.ensure_tokens(65)   # forces growth; old contents must survive
    assert pool.generation == gen0 + 1 and pool.num_pages >= 8 and float(pool.k[0, a.pages[0], 0, 0, 0]) == 7.0
    assert a.page_table[:3].tolist() == a.pages and b.page_table[:2].tolist() == b.pages
    key = a.graph_key()
    a.ensure_tokens(64 * 70)  # page table reallocation changes the graph key
    assert a.graph_key() != key and a.page_table[:70].tolist() == a.pages
    st = a.stream_state()
    assert st.layer_stride == pool.num_pages * 2 * 64 * 128 and st.k_pool == pool.k.data_ptr()
    n_free = len(pool.free)
    a.release()
    assert len(pool.free) == n_free + 70 and a.get_seq_length() == 0 and a.rope_delta is None


def test_runner_world_size_2_gloo(tmp_path):
    """N>1 path on CPU: torchrun-style env, gloo backend, barrier + all_gather_object of per-stream stats."""
    script = tmp_path / "worker.py"
    script.write_text(f"""
import sys, json, time
sys.path.insert(0, {ROOT!r})
from livecc_b200 import runner
rank, world = runner.init_distributed("gloo")
recs = runner.run_streams(list(range(5)), lambda sid: dict(tokens=10 + sid, frames=2 * sid))
if rank == 0:
    print(json.dumps(dict(world=world, recs=recs, summary=runner.summarize(recs, 2.0))))
import torch.distributed as dist
dist.destroy_process_group()
""")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
           "--master-port", "29617", str(script)]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=240)
    assert r.returncode == 0, r.stderr[-2000:]
    import json
    line = [l for l in r.stdout.splitlines() if l.startswith("{")][-1]
    d = json.loads(line)
    assert d["world"] == 2 and [x["stream"] for x in d["recs"]] == [0, 1, 2, 3, 4]
    assert [x["rank"] for x in d["recs"]] == [0, 1, 0, 1, 0]
    assert d["summary"]["tokens"] == sum(10 + i for i in range(5)) and d["summary"]["tokens_per_s"] == 30.0


def test_bench_reference_arm_contract_small():
    """`bench.py --impl reference` prints one JSON line with the contract keys (tiny config, CPU)."""
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--model", "small",
                        "--size", "56", "--steps", "1", "--warmup", "0"], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    import json
    d = json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][-1])
    assert d["impl"] == "reference" and d["unit"] == "tokens/s" and d["value"] > 0 and d["higher_is_better"] is True
    assert d["cpu_baseline"]["kind"] == "reference" and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and "workload" in d["config"]


def test_frame_selection_matches_the_reference_scan():
    """get_smart_resized_clip's vectorised frame selection == the forward scan specified at
    REF/livecc-utils/src/livecc_utils/video_process_patch.py:134-145 (spelled out here as the test's oracle),
    including the end-of-video and odd-count quirks."""
    import livecc_b200.livecc_utils.video_process_patch as V

    def scan(timestamps, pts, start):
        ts = timestamps.clone()
        while len(ts) % 2 != 0:
            ts = torch.cat([ts, ts[-1:] + 1 / 2.0])
        out, cur = [], start
        for t in ts:
            while cur < len(pts) and pts[cur] < t:
                cur += 1
            if cur >= len(pts):
                break
            out.append(cur)
        while len(out) % 2 != 0:
            out, ts = out[:-1], ts[:-1]
        return out, ts

    class FakeReader:
        def get_batch(self, idxs):
            return V._Batch(np.zeros((len(idxs), 28, 28, 3), np.uint8))

    rng = np.random.default_rng(0)
    for trial in range(200):
        n = int(rng.integers(1, 60))
        pts = np.sort(rng.uniform(0, 10, n)) if trial % 3 else np.arange(1, n + 1) / 29.97
        t0 = float(rng.uniform(-0.5, 9))
        k = int(rng.integers(1, 9))
        stamps = torch.arange(t0, t0 + 0.5 * k - 1e-9, 0.5)
        start = int(rng.integers(0, n + 2))
        want_idx, want_ts = scan(stamps, pts, start)
        clip, got_ts, got_idx = V.get_smart_resized_clip(FakeReader(), 28, 28, stamps, torch.from_numpy(pts), start)
        assert got_idx == want_idx, (trial, got_idx, want_idx)
        assert torch.allclose(got_ts.double(), want_ts.double()) and clip.shape[0] == len(want_idx)


def test_cv2_reader_on_an_encoded_video(tmp_path):
    """The decord stand-in on a real mp4 file, written here with OpenCV's MPEG-4 encoder: 25 s at 5 fps of a moving
    pattern at 540x960 (the aspect of the 1080p demo videos). Pts table, smart-resized streaming size for
    max_pixels = 384*28*28, and a 6-frame opening clip whose frames are the encoded ones (each decoded frame is closest
    to the frame written at its index, within the codec's loss)."""
    import cv2

    import livecc_b200.livecc_utils as U

    n, fps, h, w = 125, 5.0, 540, 960
    yy, xx = np.mgrid[0:h, 0:w]

    def frame(i):  # RGB, shifted by 8 / 4 / 6 levels per frame
        return np.stack([(xx + 8 * i) % 256, (yy + 4 * i) % 256, ((xx + yy) // 8 + 6 * i) % 256], -1).astype(np.uint8)

    path = str(tmp_path / "clip.mp4")
    writer = cv2.VideoWriter(path, cv2.VideoWriter_fourcc(*"mp4v"), fps, (w, h))
    assert writer.isOpened()
    for i in range(n):
        writer.write(cv2.cvtColor(frame(i), cv2.COLOR_RGB2BGR))
    writer.release()

    reader, H, W = U.get_smart_resized_video_reader(path, 384 * 28 * 28)
    assert (H, W) == (392, 728) and H % 28 == 0 and W % 28 == 0 and H * W <= 384 * 28 * 28
    reader.get_frame_timestamp(0)
    pts = torch.from_numpy(reader._frame_pts[:, 1])
    assert len(reader) == len(pts) == n and float(pts[-1]) == pytest.approx(n / fps) and bool((pts[1:] > pts[:-1]).all())
    clip, ts, idxs = U.get_smart_resized_clip(reader, H, W, torch.arange(0.0, 3.0, 0.5), pts, 0)
    assert clip.shape == (6, 3, 392, 728) and clip.dtype == torch.uint8 and len(idxs) == 6
    assert idxs == sorted(idxs) and float(clip.float().std()) > 5.0
    for i, got in zip(idxs, reader.get_batch(idxs).asnumpy()):
        err = {j: float(np.abs(got.astype(np.int16) - frame(j)).mean()) for j in (i - 1, i, i + 1)}
        assert err[i] < 4.0 and err[i] < min(err[i - 1], err[i + 1]), (i, err)
    px, grid = __import__("livecc_b200.processing", fromlist=["patchify_video"]).patchify_video(clip)
    assert grid.tolist() == [[3, 28, 52]] and px.shape == (3 * 28 * 52, 1176)


def test_op_wrappers_pass_as_many_arguments_as_the_header_declares():
    """ctypes does no arity checking: a wrapper that drifts from include/livecc_b200.h would corrupt the call
    silently. Drive the wrappers with a recording `call` and CPU tensors and compare with the prototypes."""
    import ctypes as C
    import re
    from pathlib import Path

    import torch

    from livecc_b200 import _cabi

    header = (Path(__file__).resolve().parents[1] / "include" / "livecc_b200.h").read_text()

    def declared(fn):
        return len(re.search(fn + r"\((.*?)\);", header, re.S).group(1).split(","))

    ctx = object.__new__(_cabi.Context)
    calls = []
    ctx.call = lambda name, *args: calls.append((name, len(args)))
    ctx.stream_ptr = lambda: C.c_void_p(0)
    bf = torch.bfloat16
    a, b = torch.zeros((4, 8), dtype=bf), torch.zeros((16, 8), dtype=bf)
    ctx.gemm(a, b)
    ctx.gemm(a, b, splitk_ws=torch.zeros(64))
    qkv, cu = torch.zeros((8, 3 * 2 * 80), dtype=bf), torch.tensor([0, 8], dtype=torch.int32)
    ctx.vit_attention(qkv, cu, 8, 2, 80)
    ctx.vit_attention(qkv, cu, 8, 2, 80, impl=1)
    q, kv = torch.zeros((3, 8 * 128), dtype=bf), torch.zeros((2, 2, 64, 128), dtype=bf)
    pt = torch.zeros(2, dtype=torch.int32)
    ctx.attn_prefill(q, kv, kv, pt, 4, 2, 0)
    ctx.attn_prefill(q, kv, kv, pt, 4, 2, 0, impl=1, split=True)

    class _FakeCudaU8:  # resize_bicubic_aa_u8 insists on a CUDA tensor; the arity check needs no device
        dtype, is_cuda, shape = torch.uint8, True, (2, 3, 8, 10)

        def is_contiguous(self): return True
        def dim(self): return 4
        def numel(self): return 2 * 3 * 8 * 10
        def data_ptr(self): return 0

    ctx.resize_plan = lambda *a: 1
    ctx.resize_bicubic_aa_u8(_FakeCudaU8(), (4, 6), out=_FakeCudaU8())
    assert len(calls) == 7
    for name, nargs in calls:
        assert nargs + 1 == declared(name), (name, nargs + 1, declared(name))  # + the ctx argument added by call()


def test_model_wrappers_pass_as_many_arguments_as_the_header_declares(monkeypatch):
    """Same check for the model-level entry points (prefill slot, batched decode, sub-range hook) and embed_gather."""
    import ctypes as C
    import re
    from pathlib import Path

    import torch

    from livecc_b200 import _cabi

    header = (Path(__file__).resolve().parents[1] / "include" / "livecc_b200.h").read_text()

    def declared(fn):
        return len(re.search(r"\b" + fn + r"\((.*?)\);", header, re.S).group(1).split(","))

    monkeypatch.setattr(_cabi.Context, "stream_ptr", staticmethod(lambda: C.c_void_p(0)))
    calls = []
    nm = object.__new__(_cabi.NativeModel)
    nm._call = lambda name, *args: calls.append((name, len(args)))
    st, sp = _cabi.StreamState(), _cabi.Sampling()
    ids, pos3 = torch.zeros(3, dtype=torch.int64), torch.zeros((3, 3), dtype=torch.int32)
    feats = torch.zeros((2, 8), dtype=torch.bfloat16)
    nm.prefill(st, ids, pos3, 3, 0, feats, sp, slot=2)
    nm.decode_steps(st, 1, 1, sp)
    nm.decode_batch([st, st], 1, sp)
    nm.decode_mega_debug([st], 0, 1, 31, 1)
    nm.vit_forward(torch.zeros((4, 1176)), 1, 2, 2, feats)
    nm.vit_forward_frames(torch.zeros((2, 3, 28, 28), dtype=torch.uint8), [0.0] * 3, [1.0] * 3, feats)
    ctx = object.__new__(_cabi.Context)
    ctx.call = lambda name, *args: calls.append((name, len(args)))
    ctx.embed_gather(ids, torch.zeros((10, 8), dtype=torch.bfloat16), feats, 9)
    assert len(calls) == 7
    for name, nargs in calls:
        assert nargs + 1 == declared(name), (name, nargs + 1, declared(name))  # + the model / ctx handle
