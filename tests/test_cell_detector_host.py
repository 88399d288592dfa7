"""CPU: the cell detector's host side and its oracle.  The product's CellDetector pre- and post-processing against the
reference's own table_cell_detector.py (tests/golden/cell_wrappers_ref.json), its config against the reference's
cfg_table_cell_parser_rtdtrv2.py, and the RT-DETRv2 oracle at 960 x 960 / 1500 queries against the reference's model
files (tests/golden/cell_ref.npz); both fixtures come from tests/golden/make_golden_cell.py."""
import collections
import json
import os
import sys

import numpy as np
import pytest
import torch

from oracle import refcheck as rc
from oracle import rtdetr as R

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "golden"))
from make_golden_cell import (CELL_CASES, CELL_SPEC, INPUT_SEED, MODEL_SEED, cell_input, pooled,  # noqa: E402
                              run_cases, cell_page)

GOLD = np.load(os.path.join(HERE, "golden", "cell_ref.npz"))
WRAP = json.load(open(os.path.join(HERE, "golden", "cell_wrappers_ref.json")))


@pytest.fixture(scope="module")
def detector():
    from yomitoku_b200 import CellDetector
    return CellDetector(from_pretrained=False, device="cpu")


def test_config_equals_reference(detector):
    from yomitoku_b200.config import TableCellParserRTDETRv2Config
    assert TableCellParserRTDETRv2Config() == WRAP["config"]
    m = detector.model
    assert (m.img_size, m.num_queries, m.num_classes, detector.thresh_score) == (960, 1500, 6, 0.5)


def test_host_code_equals_reference(detector):
    got = run_cases(detector, cell_page(), CELL_CASES)
    assert got == WRAP["cases"]
    # what the cases reach: the no-cell branch, hole cells (ids after the detected cells), regions, every role
    roles = collections.Counter(c["role"] for case in got for c in case["cells"])
    assert all(roles[r] > 0 for r in ("cell", "header", "empty")), roles
    assert any(len(case["cells"]) == 1 and case["cells"][0]["box"] == case["box"] for case in got)
    assert all(case["kv_regions"] and case["grid_regions"] for case in got)


def test_oracle_reproduces_reference_outputs():
    sd = R.make_state_dict(CELL_SPEC, seed=MODEL_SEED)
    aux = {}
    out = R.forward(sd, CELL_SPEC, cell_input(INPUT_SEED), aux)

    # nearly tied anchors may swap places on another CPU: rows compared as a set, ordered by their box
    def rows(boxes, logits):
        m = np.concatenate([boxes, logits], axis=1)
        return m[np.lexsort(np.round(m[:, :4], 4).T[::-1])]
    d = np.abs(rows(out["pred_boxes"][0].numpy(), out["pred_logits"][0].numpy()) - rows(GOLD["boxes"], GOLD["logits"]))
    assert d[:, :4].max() < 2e-5 and d[:, 4:].max() < 5e-4
    for i in range(3):
        for name, t in (("c", aux["backbone"][i]), ("e", aux["encoder"][i])):
            ref = GOLD["%s%d" % (name, i + 3)]
            assert np.abs(pooled(t) - ref).max() < 1e-4 * max(1.0, np.abs(ref).max())
    scores = aux["enc_logits"].max(-1).values[0].numpy()
    assert scores.shape == (18900,)
    assert np.abs(scores - GOLD["enc_scores"]).max() < 2e-4
    ref_set, got = set(GOLD["topk"].tolist()), set(aux["topk"][0].tolist())
    cut = np.sort(GOLD["enc_scores"])[-1500]
    assert all(abs(GOLD["enc_scores"][a] - cut) < 1e-3 for a in ref_set ^ got)


def test_random_init_builds_anchors_at_the_model_size():
    from yomitoku_b200.models import _rtdetr_random_state_dict
    a, b = R.make_state_dict(CELL_SPEC, seed=0), _rtdetr_random_state_dict(6, img=960)
    assert set(a) == set(b)
    assert all(tuple(a[k].shape) == tuple(b[k].shape) for k in a)
    assert torch.equal(a["decoder.anchors"], b["decoder.anchors"]) and b["decoder.anchors"].shape[1] == 18900
    assert torch.equal(a["decoder.valid_mask"], b["decoder.valid_mask"])


def test_no_tables_and_unsupported_options(detector):
    from yomitoku_b200 import CellDetector
    assert detector(cell_page(), []) == []
    import tempfile
    with tempfile.NamedTemporaryFile("w", suffix=".yaml", delete=False) as f:
        f.write("weights_path: /nonexistent/model.pth\n")
    try:
        with pytest.raises(NotImplementedError):
            CellDetector(from_pretrained=False, device="cpu", path_cfg=f.name)
    finally:
        os.unlink(f.name)
    assert CellDetector(from_pretrained=False, device="cpu", infer_onnx=True).infer_onnx is False


def test_cell_detector_refuses_to_run_without_a_gpu(detector):
    from yomitoku_b200 import _lib
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    table = type("T", (), {"box": [10, 10, 300, 200], "role": None})()
    with pytest.raises(_lib.YtkError):
        detector(cell_page(), [table])


@pytest.mark.skipif(not os.path.isdir(os.path.join(rc.REF, "src", "yomitoku")), reason="needs the reference tree")
def test_host_code_against_live_reference(detector):
    """Fresh seeds and table boxes through the reference's own table_cell_detector.py, run live."""
    from make_golden_cell import load_reference_cell_detector, reference_cell_detector
    cd, cfg = load_reference_cell_detector()
    rng = np.random.default_rng(2024)
    cases = []
    for seed in range(400, 410):
        x1, y1 = int(rng.integers(0, 400)), int(rng.integers(0, 300))
        cases.append((seed, [x1, y1, x1 + int(rng.integers(200, 500)), y1 + int(rng.integers(150, 400))]))
    page = cell_page()
    assert run_cases(detector, page, cases) == run_cases(reference_cell_detector(cd, cfg), page, cases)
