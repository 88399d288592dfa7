"""Generates tests/golden/live_ref.npz: what the reference-comparison tests compare the product and the oracle with,
produced by running the REFERENCE's own code (loaded by path, see oracle/refcheck.py; build container only) on the same
seeded inputs the tests build:

  dbnet_*, parseq<k>_*   DBNet.forward / PARSeq.forward + ParseqTokenizer.decode of oracle.refcheck.main's model cases
                         (tests/test_oracle_golden.py::test_oracle_against_reference_modules_live); PARSeq logits are
                         (B, T, ~7k) per case, so they are kept as argmax ids, per-row max / mean and a seeded sample
  flow_<case>_*          TextRecognizer.__call__ with the stand-in PARSeq (tests/flow_standins.py)
                         (tests/test_reference_flow.py::test_product_flow_matches_reference_live)
  detflow<i>_*           TextDetector.preprocess (shape, sums and a seeded sample of the tensor) and __call__ with the
                         stand-in DBNet (tests/test_reference_flow.py::test_detector_flow_matches_reference_live)
  rtdetr_b2_*            RTDETRv2 forward, table configuration, batch 2
                         (tests/test_rtdetr_host.py::test_oracle_against_live_reference_batch2)
  layout_*               prediction_reading_order on 60 seeded layouts (boxes, orders)
                         (tests/test_layout_logic.py::test_live_against_reference_when_present)

    python tests/golden/make_golden_live.py
"""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, HERE)
sys.path.insert(0, os.path.dirname(HERE))
from oracle import parseq as ops  # noqa: E402
from oracle import refcheck, weights  # noqa: E402

# the model cases of oracle.refcheck.main and the inputs the tests rebuild from these seeds
DBNET_WEIGHT_SEED, DBNET_INPUT_SEED, DBNET_INPUT_SHAPE = 1, 0, (1, 3, 96, 160)
PARSEQ_SAMPLE = 1024              # logits sampled per PARSeq case
PRE_SAMPLE = 4096                 # TextDetector.preprocess values sampled per page
FLOW_CASES = ("dynw_bucketing", "dropped_quad", "fallback_and_downscale")
LAYOUT_SEED, LAYOUT_CASES = 7, 60
DIRECTIONS = ("top2bottom", "right2left", "left2right")


def parseq_cases():
    """(spec, weights, image batch) of every PARSeq case of oracle.refcheck.main."""
    import dataclasses
    out = []
    for name, W, peaked, over in (("parseq-tiny-dynw-v4", 320, False, {}), ("parseq-tiny-dynw-v4", 200, True, {}),
                                  ("parseq-large-v4_1", 160, True, {}),
                                  ("parseq-tiny-dynw-v4", 200, True, {"decode_ar": 0}),
                                  ("parseq-tiny-dynw-v4", 200, True, {"decode_ar": 0, "refine_iters": 0}),
                                  ("parseq-tiny-dynw-v4", 200, True, {"refine_iters": 2}),
                                  ("parseq-tiny-dynw-v4", 200, True, {"refine_iters": 0}),
                                  ("parseq-tiny", 208, True, {})):
        spec = dataclasses.replace(ops.SPECS[name], **over)
        sd = weights.make_parseq_state_dict(spec, seed=3, peaked=peaked)
        img = torch.rand(4, 3, 32, W, generator=torch.Generator().manual_seed(5)) * 2 - 1
        out.append((spec, sd, img))
    return out


def dbnet_input():
    return torch.randn(*DBNET_INPUT_SHAPE, generator=torch.Generator().manual_seed(DBNET_INPUT_SEED))


def sample_index(n, k, seed):
    return np.sort(np.random.default_rng(seed).choice(n, size=min(n, k), replace=False))


def layout_cases():
    """(direction, boxes) of the 60 seeded reading-order layouts."""
    from make_golden_layout import random_boxes
    rng = np.random.default_rng(LAYOUT_SEED)
    return [(DIRECTIONS[case % 3], random_boxes(rng, int(rng.integers(2, 16)), kind="grid" if case % 2 else "mixed"))
            for case in range(LAYOUT_CASES)]


def main():
    assert refcheck.available(), "needs the reference tree (YTK_REFERENCE)"
    import flow_standins as FS
    from oracle import rtdetr as R
    from make_golden_rtdetr import rtdetr_input
    out = {}
    # ---- DBNet
    ref = refcheck.build_reference_dbnet(weights.make_dbnet_state_dict(seed=DBNET_WEIGHT_SEED))
    with torch.inference_mode():
        out["dbnet_prob"] = ref(dbnet_input())["binary"].numpy()
    # ---- PARSeq (logits sampled) + tokenizer
    charset = open(os.path.join(refcheck.SRC, "resource", "charsetv2.txt"), encoding="utf-8").read()
    assert charset == open(os.path.join(ROOT, "yomitoku_b200", "resource", "charsetv2.txt"), encoding="utf-8").read()
    for k, (spec, sd, img) in enumerate(parseq_cases()):
        m = refcheck.build_reference_parseq(spec, sd, charset)
        with torch.inference_mode():
            lg = m(img)
        strings, scores = m.tokenizer.decode(lg.softmax(-1))
        idx = sample_index(lg.numel(), PARSEQ_SAMPLE, 100 + k)
        out["parseq%d_shape" % k] = np.array(lg.shape)
        out["parseq%d_ids" % k] = lg.argmax(-1).numpy().astype(np.int16)
        out["parseq%d_rowmax" % k] = lg.max(-1).values.numpy()
        out["parseq%d_rowmean" % k] = lg.mean(-1).numpy()
        out["parseq%d_sample" % k] = lg.reshape(-1)[torch.from_numpy(idx)].numpy()
        out["parseq%d_strings" % k] = np.array(strings, dtype=str)
        out["parseq%d_scores" % k] = np.array(scores, dtype=np.float64)
    # ---- the recognizer's host flow with the stand-in PARSeq
    for name in FLOW_CASES:
        ref_rec, page, quads = FS.reference_recognizer(name)
        r, _ = ref_rec(page, quads)
        assert all(isinstance(v, int) for q in r["points"] for p in q for v in p)
        out["flow_%s_contents" % name] = np.array(r["contents"], dtype=str)
        out["flow_%s_scores" % name] = np.array(r["scores"], dtype=np.float64)
        out["flow_%s_directions" % name] = np.array(r["directions"], dtype=str)
        out["flow_%s_points" % name] = np.array(r["points"], dtype=np.int32)
    # ---- the detector's host flow with the stand-in DBNet
    ref_det = refcheck.build_reference_detector_shell()
    for i, page in enumerate(FS.detector_pages()):
        x = ref_det.preprocess(page)
        r, _ = ref_det(page)
        out["detflow%d_pre_shape" % i] = np.array(x.shape)
        out["detflow%d_pre_sum" % i] = np.array([float(x.double().sum()), float((x.double() ** 2).sum())])
        out["detflow%d_pre_sample" % i] = x.reshape(-1)[torch.from_numpy(sample_index(x.numel(), PRE_SAMPLE, 200 + i))].numpy()
        out["detflow%d_points" % i] = np.array(r["points"], dtype=np.int32)
        out["detflow%d_scores" % i] = np.array(r["scores"], dtype=np.float64)
    # ---- RT-DETRv2, table configuration, batch 2
    spec = R.SPECS["table"]
    with torch.no_grad():
        o = refcheck.build_reference_rtdetr(spec.num_classes, R.make_state_dict(spec, seed=5))(rtdetr_input(6, n=2))
    out["rtdetr_b2_boxes"], out["rtdetr_b2_logits"] = o["pred_boxes"].numpy(), o["pred_logits"].numpy()
    # ---- reading order
    from make_golden_layout import load_reference
    ro, _, sd = load_reference()
    cases, orders = layout_cases(), []
    for direction, boxes in cases:
        els = [sd.ParagraphSchema(box=b, contents="", direction="horizontal", order=0, role=None) for b in boxes]
        ro.prediction_reading_order(els, direction)
        orders += [e.order for e in els]
    out["layout_n"] = np.array([len(boxes) for _, boxes in cases], dtype=np.int32)
    out["layout_boxes"] = np.array([b for _, boxes in cases for b in boxes], dtype=np.int32)
    out["layout_order"] = np.array(orders, dtype=np.int32)
    path = os.path.join(HERE, "live_ref.npz")
    np.savez_compressed(path, **out)
    print("wrote", path, os.path.getsize(path), "bytes")


if __name__ == "__main__":
    main()
