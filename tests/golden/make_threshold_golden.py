"""Generates tests/golden/threshold_golden.json by executing the reference's own ThresholdLogitsProcessor
(REF/demo/infer.py:10-23, pure torch) on fixed score vectors. Run with the path of a checkout of showlab/livecc:

    python tests/golden/make_threshold_golden.py /path/to/livecc

The GPU test (tests/test_ops_gpu.py::test_threshold_processor_matches_reference_golden) feeds the same scores to the
sampling kernel and must reproduce `masked` (scores[token] == -inf) and `argmax` for every call of every case.
Cases keep softmax(scores)[token] at least 1e-3 away from the threshold, except the two `uniform` cases where the
probability is exactly 2^-8 in any correct fp32 softmax (the `<=` boundary itself)."""
import json
import os
import sys

import torch

OUT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "threshold_golden.json")


def reference_class(ref):
    src = open(ref).read().splitlines()
    body = "\n".join(src[9:23])  # lines 10-23: the class definition, verbatim
    assert body.lstrip().startswith("class ThresholdLogitsProcessor(LogitsProcessor):"), body[:80]
    from transformers import LogitsProcessor

    ns = {"torch": torch, "LogitsProcessor": LogitsProcessor}
    exec(compile(body, ref, "exec"), ns)
    return ns["ThresholdLogitsProcessor"]


def main():
    Proc = reference_class(os.path.join(sys.argv[1], "demo", "infer.py"))
    V = 256
    g = torch.Generator().manual_seed(7)
    cases = []

    def add(name, scores, token, base, step, n_calls):
        proc = Proc(token, base, step)
        masked, argmax = [], []
        for _ in range(n_calls):
            s = proc(torch.zeros((1, 1), dtype=torch.long), scores.clone()[None])[0]
            masked.append(bool(torch.isinf(s[token]) and s[token] < 0))
            argmax.append(int(s.argmax()))
        p = torch.softmax(scores, -1)[token].item()
        for k in range(n_calls):
            thr = base + step * k
            assert name.startswith("uniform") or abs(p - thr) > 1e-3, (name, k, p, thr)
        cases.append(dict(name=name, scores=[float(x) for x in scores.tolist()], token=token, base=base, step=step,
                          n_calls=n_calls, prob=p, masked=masked, argmax=argmax))

    s1 = torch.randn(V, generator=g) * 3
    top = int(s1.argmax())
    p_top = torch.softmax(s1, -1)[top].item()
    add("cli_zero_threshold", s1, top, 0.0, 0.0, 3)                      # REF/demo/cli.py:16-19: never masks
    add("rising_threshold_crosses", s1, top, round(p_top - 0.055, 4), 0.02, 6)   # masks from the 3rd/4th call on
    add("always_mask", s1, top, 1.1, 0.0, 2)
    second = int(s1.topk(2).indices[1])
    add("mask_non_argmax_token", s1, second, 0.9, 0.0, 2)               # argmax unchanged
    u = torch.full((V,), 1.5)
    add("uniform_boundary_equal", u, 5, 1.0 / V, 0.0, 1)                 # p == thr  ->  masked (<=)
    add("uniform_boundary_below", u, 5, (1.0 / V) * (1 - 2.0 ** -10), 0.0, 1)   # thr just below p -> kept
    json.dump(dict(source="REF/demo/infer.py:10-23 executed verbatim", V=V, cases=cases), open(OUT, "w"))
    for c in cases:
        print(c["name"], "p=%.5f" % c["prob"], c["masked"], c["argmax"])


if __name__ == "__main__":
    main()
