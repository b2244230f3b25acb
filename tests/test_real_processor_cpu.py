"""The real-processor branch (SURVEY.md §8 a4/B4): `AutoProcessor.from_pretrained(model_path, use_fast=False)`
(REF/demo/infer.py:48-49) with the UNMODIFIED transformers Qwen2VLProcessor / tokenizer / video processor, built offline by
tests/hf_tiny_processor.py, driving livecc_b200.streaming.LiveCCDemoInfer on a recording mock model, diffed against what
the unmodified reference orchestrator did on the same processor and mock (stored in tests/golden/orchestrator_golden.json
by tests/golden/make_reference_golden.py). Also pins the offline StubProcessor against it: identical pixel rows, grids and
placeholder counts."""
import os
import sys

import pytest
import torch

sys.path.insert(0, os.path.dirname(__file__))
from hf_tiny_processor import build_processor_dir, config_for  # noqa: E402

from livecc_b200.config import LiveCCConfig  # noqa: E402
from livecc_b200.processing import StubProcessor  # noqa: E402


@pytest.fixture(scope="module")
def real(tmp_path_factory):
    from transformers import AutoProcessor

    d = build_processor_dir(str(tmp_path_factory.mktemp("hfproc")))
    proc = AutoProcessor.from_pretrained(d, use_fast=False)
    return d, proc, config_for(proc, LiveCCConfig.small())


def test_load_processor_branches(real, tmp_path):
    from livecc_b200.streaming import LiveCCDemoInfer

    d, proc, cfg = real

    class M:
        config = cfg

    got = LiveCCDemoInfer._load_processor(d, M)
    assert type(got).__name__ == "Qwen2VLProcessor" and got.tokenizer(" ...").input_ids == proc.tokenizer(" ...").input_ids
    empty = tmp_path / "weights-only"
    empty.mkdir()
    with pytest.warns(UserWarning, match="no tokenizer files"):
        assert isinstance(LiveCCDemoInfer._load_processor(str(empty), M), StubProcessor)
    broken = tmp_path / "broken"
    broken.mkdir()
    (broken / "tokenizer_config.json").write_text("{ this is not json")
    with pytest.raises(Exception):     # a present-but-broken processor is an error, not a silent fallback
        LiveCCDemoInfer._load_processor(str(broken), M)


def test_stub_processor_agrees_with_the_real_one(real):
    d, proc, cfg = real
    stub = StubProcessor(cfg)
    g = torch.Generator().manual_seed(1)
    for frames, hw in [(2, (56, 84)), (6, (112, 112)), (3, (84, 56))]:
        clip = torch.randint(0, 256, (frames, 3, hw[0], hw[1]), generator=g, dtype=torch.uint8)
        conv = [{"role": "user", "content": [{"type": "text", "text": "Time=0.0-1.0s"}, {"type": "video", "video": clip},
                                             {"type": "text", "text": "Please describe the video."}]}]
        ta = proc.apply_chat_template(conv, tokenize=False, add_generation_prompt=True)
        tb = stub.apply_chat_template(conv, tokenize=False, add_generation_prompt=True)
        assert ta == tb
        a = proc(text=ta, images=None, videos=[clip], return_tensors="pt", return_attention_mask=False)
        b = stub(text=tb, images=None, videos=[clip], return_tensors="pt", return_attention_mask=False)
        assert torch.equal(a["pixel_values_videos"], b["pixel_values_videos"])       # bit-exact host patchify
        assert torch.equal(a["video_grid_thw"], b["video_grid_thw"])
        n = int(a["video_grid_thw"][0].prod()) // 4
        assert int((a["input_ids"] == cfg.video_token_id).sum()) == n == int((b["input_ids"] == cfg.video_token_id).sum())
        assert torch.equal(a["mm_token_type_ids"].bool(), a["input_ids"] == cfg.video_token_id)


REAL_PATH, REAL_SECONDS = "synthetic://240x112x140@30?seed=4", 9


def test_streaming_with_the_real_processor_equals_the_reference_orchestrator(real):
    """Both orchestrators on the real HF processor: same generate() calls, same yields (REF/demo/cli.py driving)."""
    from test_dropin_cpu import ZERO_THRESHOLD, RecordingModel, load_golden, record

    from livecc_b200.streaming import LiveCCDemoInfer

    d, proc, cfg = real
    own_model = RecordingModel(cfg)
    own = LiveCCDemoInfer(model=own_model, processor=proc)
    got = record(own, own_model, REAL_PATH, REAL_SECONDS, **ZERO_THRESHOLD)
    outs_own = got["outs"]
    assert len(outs_own) >= 6 and all(isinstance(o[2], str) for o in outs_own)
    first = got["calls"][0]
    assert first["new"].count(cfg.video_token_id) == first["rows"] // 4 and first["procs"][0][1] == own.streaming_eos_token_id
    assert own.streaming_eos_token_id == proc.tokenizer(" ...").input_ids[-1]
    for prev, cur in zip(got["calls"], got["calls"][1:]):
        assert cur["new"][:2] == [cfg.eos_token_id, cfg.newline_token_id]      # '<|im_end|>\n' glue through the real tokenizer
    ref = load_golden()["real_processor"]
    assert got["streaming_eos_token_id"] == ref["streaming_eos_token_id"]
    assert ref["outs"] == outs_own
    assert len(ref["calls"]) == len(got["calls"])
    for a, b in zip(ref["calls"], got["calls"]):
        assert a == b
