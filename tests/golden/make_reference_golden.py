"""Runs the original LiveCC project and stores what the CPU tests compare this project against, so that the tests need
no checkout of it. Run from the repo root with the path of a checkout of showlab/livecc:

    python tests/golden/make_reference_golden.py /path/to/livecc

* orchestrator_golden.json: the UNMODIFIED demo orchestrator (demo/infer.py, imported under the module swap of
  INTEGRATION.md §A) driven like demo/cli.py on the recording mock model of tests/test_dropin_cpu.py, once per run the
  tests replay: the stub processor with the cli's zero threshold and with live_cc's defaults, and the real HF processor of
  tests/hf_tiny_processor.py. Read by tests/test_dropin_cpu.py and tests/test_real_processor_cpu.py.
* reference_video_crops.npz: one decoded frame (index n // 3, RGB, [3, h, w] uint8) of each demo video
  (demo/sources/*.mp4), cropped to the 135x240 block at rows 540, columns 720 of the 1080x1920 frame, with the size the
  block maps to when the whole frame is resized to the demo reader's 392x728 (max_pixels = 384*28*28): 49x91, the same
  scale factors. Read by tests/test_resize_cpu.py.
"""
import importlib
import importlib.util
import json
import os
import sys
import tempfile
import types
from unittest import mock

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))

from hf_tiny_processor import build_processor_dir, config_for  # noqa: E402
from test_dropin_cpu import (CLASS_CONSTANTS, DROPIN_PATH, DROPIN_SECONDS, ZERO_THRESHOLD,  # noqa: E402
                             RecordingModel, record)
from test_real_processor_cpu import REAL_PATH, REAL_SECONDS  # noqa: E402

from livecc_b200.config import LiveCCConfig  # noqa: E402
from livecc_b200.processing import StubProcessor  # noqa: E402

VIDEOS = ["cvpr25_vlog.mp4", "howto_fix_laptop_mute_1080p.mp4", "warriors_vs_rockets_2025wcr1_mute_1080p.mp4"]
CROP = (540, 720, 135, 240)          # y0, x0, h, w in the 1080x1920 frame
CROP_OUT = (49, 91)                  # 135 * 392 / 1080, 240 * 728 / 1920


def load_reference_class(infer_py, model, processor):
    """demo/infer.py imported verbatim; its third-party imports resolve to stand-ins that hand it `model` and
    `processor`, and livecc_utils resolves to this project's package."""
    real_tf = importlib.import_module("transformers")
    ours = importlib.import_module("livecc_b200.livecc_utils")

    class _Model:
        @classmethod
        def from_pretrained(cls, path, **kw):
            model.from_pretrained_kwargs = dict(path=path, **kw)
            return model

    class _Processor:
        @classmethod
        def from_pretrained(cls, path, **kw):
            return processor

    tf = types.ModuleType("transformers")
    tf.Qwen2VLForConditionalGeneration, tf.AutoProcessor = _Model, _Processor
    tf.LogitsProcessor, tf.logging = real_tf.LogitsProcessor, real_tf.logging
    liger, liger_t = types.ModuleType("liger_kernel"), types.ModuleType("liger_kernel.transformers")
    liger_t.apply_liger_kernel_to_qwen2_vl = lambda *a, **k: None
    liger.transformers = liger_t
    qvu = types.ModuleType("qwen_vl_utils")
    qvu.process_vision_info = lambda *a, **k: (None, None)
    stubs = {"transformers": tf, "liger_kernel": liger, "liger_kernel.transformers": liger_t, "qwen_vl_utils": qvu,
             "livecc_utils": ours}
    with mock.patch.dict(sys.modules, stubs):
        spec = importlib.util.spec_from_file_location("ref_demo_infer", infer_py)
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)
        infer = mod.LiveCCDemoInfer(model_path="synthetic-checkpoint", device="cpu")
    return mod, infer


def orchestrator_runs(ref_root):
    infer_py = os.path.join(ref_root, "demo", "infer.py")
    cfg = LiveCCConfig.small()
    out = {"source": "demo/infer.py of showlab/livecc, executed by tests/golden/make_reference_golden.py"}
    for key, thr in (("dropin_zero_threshold", ZERO_THRESHOLD), ("dropin_default_threshold", {})):
        model = RecordingModel(cfg)
        mod, infer = load_reference_class(infer_py, model, StubProcessor(cfg))
        assert callable(model.prepare_inputs_for_generation)
        out["class_constants"] = {name: getattr(mod.LiveCCDemoInfer, name) for name in CLASS_CONSTANTS}
        out["from_pretrained_kwargs"] = {k: v for k, v in model.from_pretrained_kwargs.items() if k != "path"}
        out[key] = record(infer, model, DROPIN_PATH, DROPIN_SECONDS, **thr)
    with tempfile.TemporaryDirectory() as d:
        from transformers import AutoProcessor

        proc = AutoProcessor.from_pretrained(build_processor_dir(d), use_fast=False)
        model = RecordingModel(config_for(proc, cfg))
        _, infer = load_reference_class(infer_py, model, proc)
        out["real_processor"] = record(infer, model, REAL_PATH, REAL_SECONDS, **ZERO_THRESHOLD)
    return out


def video_crops(ref_root):
    from livecc_b200.livecc_utils import video_process_patch as vpp

    y0, x0, h, w = CROP
    arrays = {}
    for name in VIDEOS:
        reader, H, W = vpp.get_smart_resized_video_reader(os.path.join(ref_root, "demo", "sources", name), 384 * 28 * 28)
        frame = reader.get_batch([len(reader) // 3]).asnumpy()[0]
        assert frame.shape == (1080, 1920, 3) and (H, W) == (392, 728), (name, frame.shape, H, W)
        arrays[name] = np.ascontiguousarray(frame[y0:y0 + h, x0:x0 + w].transpose(2, 0, 1))
    arrays["out_size"] = np.array(CROP_OUT)
    return arrays


def main():
    ref_root = sys.argv[1]
    with open(os.path.join(HERE, "orchestrator_golden.json"), "w") as f:
        json.dump(orchestrator_runs(ref_root), f, separators=(",", ":"))
    np.savez_compressed(os.path.join(HERE, "reference_video_crops.npz"), **video_crops(ref_root))


if __name__ == "__main__":
    torch.manual_seed(0)
    main()
