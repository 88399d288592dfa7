"""CPU: the RT-DETRv2 oracle against outputs of the reference's own model files (tests/golden/rtdetr_ref.npz, generated
by tests/golden/make_golden_rtdetr.py; a batch of 2 in tests/golden/live_ref.npz), and the product's host code
around the device model - LayoutParser / TableStructureRecognizer pre- and post-processing, RTDETRPostProcessor -
against outputs of the reference's own layout_parser.py / table_structure_recognizer.py
(tests/golden/rtdetr_wrappers_ref.json)."""
import json
import os
import sys

import numpy as np
import pytest
import torch

from oracle import rtdetr as R

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "golden"))
from make_golden_rtdetr import fake_preds, pooled, rtdetr_input, table_preds  # noqa: E402

GOLD = np.load(os.path.join(HERE, "golden", "rtdetr_ref.npz"))
WRAP = json.load(open(os.path.join(HERE, "golden", "rtdetr_wrappers_ref.json")))
CASES = {"layout": (11, 21), "table": (12, 22)}


@pytest.mark.parametrize("kind", ["layout", "table"])
def test_oracle_reproduces_reference_outputs(kind):
    spec = R.SPECS[kind]
    sd = R.make_state_dict(spec, seed=CASES[kind][0])
    aux = {}
    out = R.forward(sd, spec, rtdetr_input(CASES[kind][1]), aux)
    # queries come in descending encoder score: on another CPU two (nearly) tied anchors may swap places, so the rows
    # are compared as a set (ordered by their box), as in the batch-2 test below
    def rows(boxes, logits):
        m = np.concatenate([boxes, logits], axis=1)
        return m[np.lexsort(np.round(m[:, :4], 4).T[::-1])]
    d = np.abs(rows(out["pred_boxes"][0].numpy(), out["pred_logits"][0].numpy()) -
               rows(GOLD[kind + "_boxes"], GOLD[kind + "_logits"]))
    assert d[:, :4].max() < 2e-5 and d[:, 4:].max() < 5e-4
    for i in range(3):
        for name, t in (("c", aux["backbone"][i]), ("e", aux["encoder"][i])):
            ref = GOLD["%s_%s%d" % (kind, name, i + 3)]
            assert np.abs(pooled(t) - ref).max() < 1e-4 * max(1.0, np.abs(ref).max())
    scores = aux["enc_logits"].max(-1).values[0].numpy()
    assert np.abs(scores - GOLD[kind + "_enc_scores"]).max() < 2e-4
    # the selected set: identical except for anchors whose score is within the comparison tolerance of the cut
    ref_set, got = set(GOLD[kind + "_topk"].tolist()), set(aux["topk"][0].tolist())
    cut = np.sort(GOLD[kind + "_enc_scores"])[-300]
    assert all(abs(GOLD[kind + "_enc_scores"][a] - cut) < 1e-3 for a in ref_set ^ got)


def test_oracle_against_live_reference_batch2():
    """Batch 2 of the table configuration against the reference's RTDETRv2 outputs stored by
    tests/golden/make_golden_live.py."""
    spec = R.SPECS["table"]
    sd = R.make_state_dict(spec, seed=5)
    x = rtdetr_input(6, n=2)
    z = np.load(os.path.join(HERE, "golden", "live_ref.npz"))
    ref = {"pred_boxes": torch.from_numpy(z["rtdetr_b2_boxes"]), "pred_logits": torch.from_numpy(z["rtdetr_b2_logits"])}
    out = R.forward(sd, spec, x)
    for b in range(2):
        # queries come in descending encoder score: two anchors with (nearly) the same score may swap places, so the
        # rows are compared as a set (ordered by their box)
        def rows(o):
            m = torch.cat([o["pred_boxes"][b], o["pred_logits"][b]], dim=1).numpy()
            return m[np.lexsort(np.round(m[:, :4], 4).T[::-1])]
        d = np.abs(rows(ref) - rows(out))
        assert d[:, :4].max() < 2e-5 and d[:, 4:].max() < 5e-4


def test_product_random_init_has_the_reference_key_set():
    from yomitoku_b200.models import _rtdetr_random_state_dict
    for kind in ("layout", "table"):
        spec = R.SPECS[kind]
        a, b = R.make_state_dict(spec, seed=0), _rtdetr_random_state_dict(spec.num_classes)
        assert set(a) == set(b)
        assert all(tuple(a[k].shape) == tuple(b[k].shape) for k in a)
        assert torch.equal(a["decoder.anchors"], b["decoder.anchors"])
        assert torch.equal(a["decoder.valid_mask"], b["decoder.valid_mask"])


def test_postprocessor_equals_oracle_and_handles_batches():
    from yomitoku_b200.postprocessor import RTDETRPostProcessor
    preds = fake_preds(7, 6)
    two = {k: torch.cat([v, torch.flip(v, dims=[1])]) for k, v in preds.items()}
    res = RTDETRPostProcessor(6, 300)(two, np.array([[1600, 1200], [800, 600]]), 0.5)
    for i, size in enumerate(((1600, 1200), (800, 600))):
        ref = R.postprocess(R.SPECS["layout"], {k: v[i:i + 1] for k, v in two.items()}, size, 0.5)
        for k in ref:
            assert np.array_equal(ref[k], res[i][k]), k
    assert len(res[0]["scores"]) > 5 and np.all(np.diff(res[0]["scores"]) <= 0)


def _plain(schema):
    return json.loads(schema.model_dump_json())


def test_layout_parser_host_code_equals_reference():
    from yomitoku_b200 import LayoutParser
    parser = LayoutParser(from_pretrained=False, device="cpu")
    assert parser.model.num_classes == 6 and parser.thresh_score == 0.5
    for case in WRAP["layout"]:
        got = _plain(parser.postprocess(fake_preds(case["seed"], 6), tuple(case["size"])))
        assert got == case["result"]
        assert sum(len(v) for v in got.values()) > 3
    page = np.random.default_rng(5).integers(0, 255, (700, 900, 3), dtype=np.uint8)
    x = parser.preprocess(page)
    assert x.shape == (1, 3, 640, 640) and x.dtype == torch.float32
    assert float(x.double().sum()) == WRAP["preprocess_page_sum"]
    assert x[0, :, ::97, ::89].numpy().tolist() == WRAP["preprocess_page_probe"]


def test_table_structure_recognizer_host_code_equals_reference():
    from yomitoku_b200 import TableStructureRecognizer
    rec = TableStructureRecognizer(from_pretrained=False, device="cpu")
    assert rec.model.num_classes == 3 and rec.thresh_score == 0.4
    page = np.random.default_rng(5).integers(0, 255, (700, 900, 3), dtype=np.uint8)
    n_span = 0
    for case in WRAP["table"]:
        data = rec.preprocess(page, [case["box"]])[0]
        assert float(data["tensor"].double().sum()) == case["tensor_sum"]
        got = _plain(rec.postprocess(table_preds(case["seed"]), data))
        assert got == case["result"]
        n_span += sum(1 for c in got["cells"] if c["col_span"] > 1 or c["row_span"] > 1)
    assert n_span > 0


def test_layout_models_refuse_to_run_without_a_gpu():
    from yomitoku_b200 import LayoutAnalyzer, _lib
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    nop = {"from_pretrained": False}
    an = LayoutAnalyzer(configs={"layout_parser": nop, "table_structure_recognizer": nop}, device="cpu")
    with pytest.raises(_lib.YtkError):
        an(np.zeros((64, 64, 3), np.uint8))
