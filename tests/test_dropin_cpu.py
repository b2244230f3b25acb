"""Diffs livecc_b200.streaming.LiveCCDemoInfer against what the UNMODIFIED reference orchestrator (REF/demo/infer.py,
imported under the module swap INTEGRATION.md §A describes) did on the same recording mock model: every generate() call
(ids, cache length, pixel rows, kwargs incl. the ThresholdLogitsProcessor the canonical caller REF/demo/cli.py:16-19
asks for), every yielded ((start, stop), text) and the `state` contract. The reference's run is stored in
tests/golden/orchestrator_golden.json (tests/golden/make_reference_golden.py regenerates it from a reference checkout).
The model is a deterministic recording mock (this is the host-side boundary test for SURVEY.md §8 B1-B3; the arithmetic
behind generate() is covered by the `-m gpu` parity tests)."""
import hashlib
import json
import os
import types

import pytest
import torch

from livecc_b200.config import LiveCCConfig
from livecc_b200.processing import StubProcessor

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
CLASS_CONSTANTS = ("fps", "initial_fps_frames", "streaming_fps_frames", "initial_time_interval",
                   "streaming_time_interval", "frame_time_interval")
# the recorded drop-in runs: this clip, driven for 12 s, with the cli's zero threshold and with live_cc's defaults
DROPIN_PATH, DROPIN_SECONDS = "synthetic://330x140x112@30?seed=9", 12   # 11 s of video, non-square frames
ZERO_THRESHOLD = dict(streaming_eos_base_threshold=0.0, streaming_eos_threshold_step=0)


def load_golden():
    with open(os.path.join(GOLDEN_DIR, "orchestrator_golden.json")) as f:
        return json.load(f)


class _Cache:
    def __init__(self):
        self.n = 0

    def get_seq_length(self):
        return self.n


class RecordingModel:
    """generate() is a pure function of (call index, max_new_tokens); every argument is recorded."""

    def __init__(self, cfg):
        self.config, self.device, self.calls = cfg, torch.device("cpu"), []

    def generate(self, input_ids=None, past_key_values=None, max_new_tokens=16, **kw):
        cache = past_key_values or _Cache()
        k = len(self.calls)
        procs = kw.get("logits_processor")
        rec = dict(L=input_ids.shape[1], past=cache.n, new=input_ids[0, cache.n:].tolist(), max_new_tokens=max_new_tokens,
                   rows=kw["pixel_values_videos"].shape[0] if kw.get("pixel_values_videos") is not None else 0,
                   px_sum=float(kw["pixel_values_videos"].double().sum()) if kw.get("pixel_values_videos") is not None else 0.0,
                   grid=kw["video_grid_thw"].tolist() if kw.get("video_grid_thw") is not None else None,
                   do_sample=kw.get("do_sample"), repetition_penalty=kw.get("repetition_penalty"),
                   pad_token_id=kw.get("pad_token_id"), return_dict=kw.get("return_dict_in_generate"),
                   procs=None if procs is None else [(type(p).__name__, p.token_id, p.base_threshold, p.step) for p in procs],
                   other=sorted(set(kw) - {"pixel_values_videos", "video_grid_thw", "do_sample", "repetition_penalty",
                                           "pad_token_id", "return_dict_in_generate", "logits_processor"}))
        self.calls.append(rec)
        n = 3 + k % 4  # 3..6 tokens, the last one EOS on even calls (early stop) else a plain id (token budget)
        gen = [2000 + 7 * k + j for j in range(n)]
        if k % 2 == 0:
            gen[-1] = self.config.eos_token_id
        seq = torch.cat([input_ids, torch.tensor([gen], dtype=input_ids.dtype)], 1)
        cache.n = seq.shape[1] - 1
        return types.SimpleNamespace(sequences=seq, past_key_values=cache)


def _drive(infer, path, seconds, **kw):
    """REF/demo/cli.py:13-24."""
    state = {"video_path": path}
    outs = []
    for t in range(seconds + 1):
        state["video_timestamp"] = t
        for (s, e), resp, state in infer.live_cc(message="Please describe the video.", state=state,
                                                  max_pixels=384 * 28 * 28, repetition_penalty=1.05, **kw):
            outs.append((s, e, resp, float(state["last_timestamp"]), int(state["last_video_pts_index"]),
                         state["past_ids"][0].tolist(), state["past_key_values"].get_seq_length()))
        if state.get("video_end", False):
            break
    return outs, state


def record(infer, model, path, seconds, **kw):
    """Everything one orchestrator does on a RecordingModel, as JSON data: the constructor's derived ids, every yield,
    every generate() call, the final state, and what a call after the end of the stream yields / asks of the model.
    The id history of each yield is kept as a SHA-256 of its ids (every yield carries the whole history)."""
    outs, st = _drive(infer, path, seconds, **kw)
    outs = [(*o[:5], hashlib.sha256(json.dumps(o[5]).encode()).hexdigest(), o[6]) for o in outs]
    n_calls = len(model.calls)
    st["video_timestamp"] = 99
    after = list(infer.live_cc(message="", state=st))
    rec = dict(streaming_eos_token_id=infer.streaming_eos_token_id, system_prompt_offset=infer.system_prompt_offset,
               outs=outs, calls=model.calls[:n_calls], video_end=bool(st.get("video_end")), message=st["message"],
               yields_after_end=len(after), calls_after_end=len(model.calls) - n_calls)
    return json.loads(json.dumps(rec))


@pytest.mark.parametrize("thr", [ZERO_THRESHOLD, dict()])
def test_unmodified_reference_orchestrator_equals_streaming_mirror(thr, monkeypatch):
    from livecc_b200 import streaming
    from livecc_b200.streaming import LiveCCDemoInfer

    gold = load_golden()
    ref = gold["dropin_zero_threshold" if thr else "dropin_default_threshold"]
    cfg = LiveCCConfig.small()
    m_own = RecordingModel(cfg)
    loaded = {}

    def from_pretrained(path, **kw):
        loaded.update(path=path, **kw)
        return m_own

    monkeypatch.setattr(streaming.LiveCCB200ForConditionalGeneration, "from_pretrained", staticmethod(from_pretrained))
    own = LiveCCDemoInfer(model_path="synthetic-checkpoint", device="cpu", processor=StubProcessor(cfg))
    for key in ("torch_dtype", "device_map"):                      # REF/demo/infer.py:43-47
        assert loaded[key] == gold["from_pretrained_kwargs"][key], key
    assert callable(m_own.prepare_inputs_for_generation)          # REF/demo/infer.py:50 assigns it on the model
    for name in CLASS_CONSTANTS:
        assert getattr(LiveCCDemoInfer, name) == gold["class_constants"][name], name
    got = record(own, m_own, DROPIN_PATH, DROPIN_SECONDS, **thr)
    assert got["streaming_eos_token_id"] == ref["streaming_eos_token_id"]
    assert got["system_prompt_offset"] == ref["system_prompt_offset"]
    assert len(got["outs"]) == len(ref["outs"]) >= 9
    for a, b in zip(ref["outs"], got["outs"]):
        assert a == b
    assert len(got["calls"]) == len(ref["calls"]) == len(ref["outs"])
    for a, b in zip(ref["calls"], got["calls"]):
        pa, pb = a.pop("procs"), b.pop("procs")
        assert a == b
        if thr:
            assert pa is not None and pb is not None and pa == pb
            assert pb[0][0] == "ThresholdLogitsProcessor"
        else:
            assert pa is None and pb is None
    assert ref["calls"][0]["max_new_tokens"] == 16 and ref["calls"][0]["pad_token_id"] == cfg.eos_token_id
    assert got["video_end"] == ref["video_end"] and got["message"] == ref["message"]
    # nothing left to do once the stream ended: both generators are empty and make no further model calls
    assert got["yields_after_end"] == ref["yields_after_end"] == 0
    assert got["calls_after_end"] == ref["calls_after_end"] == 0


def test_reference_threshold_processor_is_the_golden_source():
    """The committed golden (tests/golden/threshold_golden.json, generated by executing the reference class) follows the
    reference's rule, spelled out here as the test's oracle: call k masks scores[token] to -inf when
    softmax(scores)[token] <= base + step * k, and the argmax is taken after the mask."""
    with open(os.path.join(GOLDEN_DIR, "threshold_golden.json")) as f:
        gold = json.load(f)
    for c in gold["cases"]:
        scores = torch.tensor(c["scores"])
        p = torch.softmax(scores, -1)[c["token"]]
        assert float(p) == pytest.approx(c["prob"], rel=1e-6, abs=0), c["name"]
        for k in range(c["n_calls"]):
            masked = bool(p <= c["base"] + c["step"] * k)
            s = scores.clone()
            if masked:
                s[c["token"]] = -float("inf")
            assert masked == c["masked"][k] and int(s.argmax()) == c["argmax"][k], (c["name"], k)
