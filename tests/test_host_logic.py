"""CPU: host-side logic of the product package (config, catalog, batching, post-processing, tokenizer) against the
oracle and against the expectations the reference's own tests pin (tests/test_ocr.py, test_data.py, test_base.py)."""
import os

import numpy as np
import pytest
import torch

from oracle import parseq as ops
from oracle import pipeline as opipe
from yomitoku_b200 import OCR, DocumentAnalyzer, TextDetector, TextRecognizer
from yomitoku_b200 import data as D
from yomitoku_b200.base import BaseModelCatalog, BaseModule
from yomitoku_b200.postprocessor import (DBnetPostProcessor, ParseqTokenizer, offset_convex_polygon_round,
                                         polygon_area_length)
from yomitoku_b200.synth import synthetic_page, synthetic_prob_map
from yomitoku_b200.text_recognizer import plan_mini_batches

HERE = os.path.dirname(os.path.abspath(__file__))


def test_ocr_config_plumbing_like_reference_test_ocr():
    # reference tests/test_ocr.py:8-32
    configs = {
        "text_detector": {"path_cfg": os.path.join(HERE, "yaml", "text_detector.yaml"), "from_pretrained": False},
        "text_recognizer": {"path_cfg": os.path.join(HERE, "yaml", "text_recognizer.yaml"), "from_pretrained": False,
                            "model_name": "parseq-tiny-dynw-v4"},
    }
    ocr = OCR(configs=configs, device="cpu", visualize=True)
    assert ocr.detector.device == torch.device("cpu")
    assert ocr.recognizer.device == torch.device("cpu")
    assert ocr.detector.visualize and ocr.recognizer.visualize
    assert ocr.detector.post_processor.thresh == 0.4
    assert ocr.recognizer.model.refine_iters == 0


def test_invalid_config_raises_like_reference():
    with pytest.raises(FileNotFoundError):
        OCR(configs={"text_detector": {"path_cfg": "nope.yaml", "from_pretrained": False}}, device="cpu")
    with pytest.raises(ValueError):
        OCR(configs="invalid", device="cpu")
    with pytest.raises(ValueError):
        DocumentAnalyzer(configs="invalid", device="cpu")
    with pytest.raises(ValueError):
        TextDetector(model_name="unknown-model", from_pretrained=False, device="cpu")


def test_catalog_behaviour_like_reference_test_base():
    cat = BaseModelCatalog()
    cat.register("a", dict, object)
    with pytest.raises(ValueError):
        cat.register("a", dict, object)
    assert cat.get("A") == (dict, object)
    with pytest.raises(ValueError):
        cat.get("b")

    class Bad(BaseModule):
        model_catalog = None

    with pytest.raises(NotImplementedError):
        Bad()
    names = TextRecognizer.model_catalog.list_model()
    assert names == ["parseq", "parseqv2", "parseq-small", "parseq-tiny", "parseq-large-v4_1", "parseq-tiny-dynw-v4"]
    assert TextDetector.model_catalog.list_model() == ["dbnet", "dbnetv2", "dbnetv2_1"]


def test_no_cpu_fallback_on_the_device_path():
    det = TextDetector(from_pretrained=False, device="cpu")
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    with pytest.raises(Exception) as e:
        det(np.zeros((64, 64, 3), np.uint8))
    assert "no CPU fallback" in str(e.value)


def test_resize_shortest_edge_rules():
    # reference tests/test_data.py:83-101
    for h, w in ((1200, 1600), (1600, 1200), (842, 596), (500, 3000), (40, 50)):
        out = D.resize_shortest_edge(np.zeros((h, w, 3), np.float32), 1280, 1600)
        oh, ow = out.shape[:2]
        assert oh % 32 == 0 and ow % 32 == 0 and max(oh, ow) <= 1600
        assert (oh, ow) == opipe.detector_input_size(h, w)
    assert D.shortest_edge_size(1200, 1600, 1280, 1600) == (1184, 1600)


def test_validate_quads_truth_table():
    img = np.zeros((100, 200, 3), np.uint8)
    assert D.validate_quads(img, [[0, 0], [200, 0], [200, 100], [0, 100]]) is True      # x2 == w allowed
    assert D.validate_quads(img, [[0, 0], [201, 0], [201, 100], [0, 100]]) is None
    assert D.validate_quads(img, [[-1, 0], [10, 0], [10, 10], [0, 10]]) is None
    assert D.validate_quads(img, [[0, 0], [10, 0], [10, 10]]) is None
    assert D.validate_quads(img, [[0, 0, 1], [10, 0], [10, 10], [0, 10]]) is None


def test_crops_match_oracle():
    page, quads = synthetic_page(3)
    rgb = page[:, :, ::-1]
    for dyn in (False, True):
        for q in quads[:25] + [[[100, 100], [124, 100], [124, 400], [100, 400]]]:   # last one is vertical text
            roi = D.rotate_text_image(D.extract_roi_with_perspective(rgb, q))
            mine = D.resize_with_dynamic_padding(roi, [32, 800]) if dyn else D.resize_with_padding(roi, [32, 800])
            ref, cw = opipe.make_crop(rgb, q, (32, 800), dyn)
            assert np.array_equal(mine, ref)
            assert cw == D.calc_resize_without_padding(roi, [32, 800])[1]
            assert torch.equal(D.crop_to_tensor(mine), opipe.to_tensor(ref))


@pytest.mark.parametrize("dyn,budget,cap,bs", [(True, 8000, 64, 10), (True, None, None, 128), (False, None, None, 128),
                                               (True, 800, 3, 10)])
def test_mini_batch_plan_matches_oracle(dyn, budget, cap, bs):
    rng = np.random.default_rng(0)
    widths = (rng.integers(9, 100, size=300) * 8).tolist()
    for order in (None, np.argsort(widths).tolist()):
        assert plan_mini_batches(widths, order, dyn, bs, budget, cap) == opipe.mini_batches(widths, order, dyn, bs,
                                                                                            budget, cap)
    plan = plan_mini_batches([320] * 16, None, True, 10, 8000, 64)
    assert plan == [list(range(16))]            # BASELINE config 1: one batch, 16 * 320 <= 8000


def test_postprocessor_matches_oracle_and_recovers_boxes():
    page, quads = synthetic_page(1)
    prob = synthetic_prob_map(quads, (1184, 1600), (1200, 1600))
    pp = DBnetPostProcessor(2, 0.3, 0.4, 1500, 3.5)
    got_q, got_s = pp({"binary": prob[None, None]}, (1200, 1600))
    ref_q, ref_s = opipe.dbnet_postprocess(prob, (1200, 1600))
    assert got_q == ref_q and np.allclose(got_s, ref_s)
    assert len(got_q) == len(quads)
    # every ground-truth box is found again within a few pixels (unclip grows the shrunk mask back)
    gt = np.array([[q[0][0], q[0][1], q[2][0], q[2][1]] for q in quads], dtype=np.float32)
    found = np.array([[min(p[0] for p in q), min(p[1] for p in q), max(p[0] for p in q), max(p[1] for p in q)]
                      for q in got_q], dtype=np.float32)
    for g in gt:
        assert np.abs(found - g).max(axis=1).min() <= 12


def test_clipper_offset_properties():
    box = np.array([[10.7, 20.2], [110.9, 20.2], [110.9, 44.6], [10.7, 44.6]], dtype=np.float32)
    for delta in (3.0, 7.25, 15.5):
        out = offset_convex_polygon_round(box, delta)
        assert np.array_equal(out, opipe.clipper_offset_box(box, delta))
        # extents = int-truncated box grown by delta (rounded), corners rounded (inside the bounding rectangle)
        assert abs(out[:, 0].min() - (10 - delta)) <= 0.5 and abs(out[:, 0].max() - (110 + delta)) <= 0.5
        assert abs(out[:, 1].min() - (20 - delta)) <= 0.5 and abs(out[:, 1].max() - (44 + delta)) <= 0.5
        r = np.hypot(out[:, 0] - np.clip(out[:, 0], 10, 110), out[:, 1] - np.clip(out[:, 1], 20, 44))
        assert r.max() <= delta + 0.75          # every vertex lies within delta of the box (round joins)
    rot = np.array([[0, 0], [100, 20], [96, 40], [-4, 20]], dtype=np.float32)
    assert np.array_equal(offset_convex_polygon_round(rot, 5.0), opipe.clipper_offset_box(rot, 5.0))
    assert np.array_equal(offset_convex_polygon_round(rot[::-1], 5.0)[:, 0].min(),
                          offset_convex_polygon_round(rot, 5.0)[:, 0].min())   # orientation is fixed internally


def test_unclip_against_the_geometric_definition():
    """The Clipper restatements (product and oracle) against the DEFINITION of a round-join offset instead of against
    each other: the offset of a convex polygon by delta is its Minkowski sum with a disk - every output vertex lies at
    distance delta from the input polygon, the area is A + L * delta + pi * delta^2 (minus the chord deficit of the
    arc tolerance 0.25, plus / minus the integer rounding of the vertices), and for a rectangle w x h the minimum-area
    rectangle of the result - the only thing the reference reads from it (dbnet_postporcessor.py:66) - is
    (w + 2 delta) x (h + 2 delta) at the same angle.  pyclipper itself is not installable here (DESIGN.md section 2);
    this pins the arithmetic that is restated from it to the geometry it implements."""
    import cv2
    rng = np.random.default_rng(7)

    def dist_to_polygon(pts, poly):
        d = np.full(len(pts), np.inf)
        for i in range(len(poly)):
            a, b = poly[i], poly[(i + 1) % len(poly)]
            ab = b - a
            t = np.clip(((pts - a) @ ab) / max(float(ab @ ab), 1e-12), 0.0, 1.0)
            d = np.minimum(d, np.linalg.norm(pts - (a + t[:, None] * ab), axis=1))
        return d

    for _ in range(200):
        w, h = rng.uniform(12, 400), rng.uniform(6, 60)
        ang = rng.uniform(-90, 90)
        cx, cy = rng.uniform(300, 1200, size=2)
        box = cv2.boxPoints(((float(cx), float(cy)), (float(w), float(h)), float(ang))).astype(np.float32)
        delta = float(rng.uniform(1.5, 40))
        # shapely's Polygon(box).area / .length (dbnet_postporcessor.py:88,94) of a rectangle: w * h and 2 (w + h)
        a_box, l_box = polygon_area_length(box)
        assert abs(a_box - w * h) <= 1e-3 * w * h + 0.05 and abs(l_box - 2 * (w + h)) <= 1e-3 * (w + h) + 0.05
        tb = np.trunc(box).astype(np.float64)                      # Clipper works on the int-truncated vertices
        (_, _), (tw, th), _ = cv2.minAreaRect(tb.astype(np.float32))
        area = 0.5 * abs(np.dot(tb[:, 0], np.roll(tb[:, 1], -1)) - np.dot(tb[:, 1], np.roll(tb[:, 0], -1)))
        perim = np.linalg.norm(tb - np.roll(tb, -1, axis=0), axis=1).sum()
        for fn in (offset_convex_polygon_round, opipe.clipper_offset_box):
            out = np.asarray(fn(box, delta), dtype=np.float64)
            assert len(out) >= 8
            # (1) every vertex at distance delta from the polygon (integer rounding: half a pixel diagonal)
            d = dist_to_polygon(out, tb)
            assert np.abs(d - delta).max() <= 0.75, (np.abs(d - delta).max(), delta)
            # (2) area of the Minkowski sum; the chords of the four round joins lose at most arc_tolerance * arc length
            a_out = 0.5 * abs(np.dot(out[:, 0], np.roll(out[:, 1], -1)) - np.dot(out[:, 1], np.roll(out[:, 0], -1)))
            a_exact = area + perim * delta + np.pi * delta * delta
            slack = 0.25 * 2 * np.pi * delta + 0.75 * (perim + 2 * np.pi * delta)
            assert -slack <= a_out - a_exact <= 0.75 * (perim + 2 * np.pi * delta), (a_out, a_exact)
            # (3) what the reference reads: the minimum-area rectangle grows by delta on every side
            (_, _), (ow, oh), _ = cv2.minAreaRect(out.astype(np.float32))
            got, want = sorted((ow, oh)), sorted((tw + 2 * delta, th + 2 * delta))
            assert abs(got[0] - want[0]) <= 1.5 and abs(got[1] - want[1]) <= 1.5, (got, want)


def test_tokenizer_decode_ids_matches_oracle(charset_v2):
    tok, otok = ParseqTokenizer(charset_v2), ops.Tokenizer(charset_v2)
    assert (tok.eos_id, tok.bos_id, tok.pad_id) == (0, 7119, 7120) and len(tok) == 7121
    g = torch.Generator().manual_seed(0)
    logits = torch.randn(6, 101, 7119, generator=g) * 3
    logits[0, 5, 0] = 50.0
    logits[1, 0, 0] = 50.0
    logits[2, 100, 0] = 50.0
    p = logits.softmax(-1)
    s1, p1 = tok.decode(p)
    s2, p2 = otok.decode(p)
    assert s1 == s2 and np.allclose(p1, p2, rtol=1e-6, atol=0)
    assert len(s1[0]) == 5 and s1[1] == "" and len(s1[2]) == 100 and len(s1[3]) == 101


def test_recognizer_cpu_plumbing_config1():
    # BASELINE config 1 (plumbing, no GPU): tiny-dynw, 16 crops whose tensors are 3x32x320 -> one batch
    rec = TextRecognizer(model_name="parseq-tiny-dynw-v4", device="cpu", from_pretrained=False, dynamic_width=True,
                         batch_bucketing=True)
    page = np.full((600, 1400, 3), 255, np.uint8)
    quads = [[[10, 10 + 34 * i], [266, 10 + 34 * i], [266, 42 + 34 * i], [10, 42 + 34 * i]] for i in range(16)]
    plan, points, dataset, order = rec.preprocess(page, quads)
    assert len(dataset) == 16 and all(d.shape == (32, 320, 3) for d in dataset.data)
    assert len(plan) == 1 and sorted(plan[0]) == list(range(16))
    assert dataset[0].shape == (3, 32, 320) and float(dataset[0].max()) == 1.0
    padded, group = rec._collate_widths(dataset.data, plan)
    assert padded == [320] * 16 and group == [0] * 16


def test_batched_pipeline_with_stub_models():
    """CPU: the whole host side of BatchedOCR (shared staging ring, worker pool, crop arena, descriptor building,
    three-stage stream, result assembly) with the two device calls replaced by stand-ins that compute from the bytes
    they are handed.  Per page the recognizer stand-in must see exactly the crops the one-page ParseqDataset cuts."""
    import ctypes

    from yomitoku_b200 import TextDetector, TextRecognizer
    from yomitoku_b200.data import ParseqDataset
    from yomitoku_b200.pipeline import BatchedOCR
    from yomitoku_b200.postprocessor import DBnetPostProcessor
    from yomitoku_b200.synth import synthetic_page, synthetic_prob_map

    det = TextDetector(from_pretrained=False, device="cpu")
    rec = TextRecognizer(model_name="parseq-tiny-dynw-v4", from_pretrained=False, device="cpu", dynamic_width=True,
                         batch_bucketing=True)
    Hn, Wn = 1184, 1600
    batches, maps = [], []
    for k in range(4):        # more batches than ring slots
        pages, pm = [], []
        for i in range(2):
            p, q = synthetic_page(70 + 2 * k + i)
            pages.append(p)
            pm.append(synthetic_prob_map(q, (Hn, Wn), (1200, 1600)))
        batches.append(pages)
        maps.append(pm)
    det.model.input_size = lambda h, w: (Hn, Wn)
    det.model.detect_pages_u8 = lambda pages, out=None, stream=None: out      # maps come from prob_override
    S = rec.model.max_label_length + 1
    seen = []

    def fake_ptr(ptr, on_device, total, descs, n, n_groups, stream=None):
        raw = np.ctypeslib.as_array(ctypes.cast(ptr, ctypes.POINTER(ctypes.c_uint8)), shape=(total,))
        ids = np.zeros((n, S), np.int32)
        for r, d in enumerate(descs):
            c = raw[int(d["pix_off"]):int(d["pix_off"]) + 32 * int(d["w"]) * 3]
            ids[r, 0] = 1 + int(c.astype(np.int64).sum()) % 7000
            ids[r, 1] = 1 + int(d["wp"]) % 7000
            seen.append((int(d["w"]), int(d["wp"]), int(d["group"]), int(c.astype(np.int64).sum())))
        return ids, np.full((n, S), 0.5, np.float32), np.full((n_groups,), S, np.int32)

    rec.model.run_packed_ptr = fake_ptr
    # the host crop path (the default only where no GPU is present): the stand-in reads the crop arena on the host
    ocr = BatchedOCR(det, rec, workers=2, det_batch=1, device_crops=False)
    try:
        got = list(ocr.stream(batches, lookahead=2, prob_override=maps))
        again = [ocr(pg, prob_override=pm) for pg, pm in zip(batches, maps)]
        # manual use: four batches submitted before the first is collected - unrecognised batches keep their staging
        # slot (the ring grows instead of overwriting a crop arena that has not been read yet)
        handles = [ocr.submit(pg, pm) for pg, pm in zip(batches, maps)]
        assert ocr._ring == 4
        manual = [ocr.collect(h) for h in handles]
    finally:
        ocr.close()
    assert [[[w.content for w in pg.words] for pg in b] for b in manual] == \
        [[[w.content for w in pg.words] for pg in b] for b in got]
    post = DBnetPostProcessor(**dict(det._cfg.post_process))
    assert len(got) == 4
    for k in range(4):
        for i in range(2):
            quads, scores = post({"binary": maps[k][i][None, None]}, (1200, 1600))
            ds = ParseqDataset(rec._cfg, batches[k][i], quads, num_workers=1, dynamic_width=True)
            words = got[k][i].words
            assert [w.points for w in words] == quads and len(words) == len(ds)
            # first decoded char encodes the crop's pixel checksum: every word got ITS crop, in detection order
            expect = [rec.tokenizer._itos[1 + int(c.astype(np.int64).sum()) % 7000] for c in ds.data]
            assert [w.content[0] for w in words] == [unicodedata_nfkc(e)[0] for e in expect]
            assert [[w.content for w in pg.words] for pg in again[k]] == [[w.content for w in pg.words] for pg in got[k]]


def unicodedata_nfkc(s):
    import unicodedata
    return unicodedata.normalize("NFKC", s)


def test_batched_pipeline_device_crops_with_stub_models(monkeypatch):
    """CPU: the device_crops path of BatchedOCR (pages kept "on the device", workers return quads + crop records only,
    canvases cut by ytk_extract_crops_u8 in group order) with the three device calls replaced by stand-ins; the crop
    stand-in runs the product's own crop arithmetic compiled for the host (oracle/crop_host.cpp).  Every word must get
    the canvas the one-page OpenCV path (ParseqDataset) cuts for it, and stream() must equal per-batch calls."""
    import ctypes

    from oracle import build_crop_host
    from yomitoku_b200 import models as M
    from yomitoku_b200.data import ParseqDataset, layout_crop_buffers
    from yomitoku_b200.pipeline import BatchedOCR

    host = ctypes.CDLL(build_crop_host.build())
    det = TextDetector(from_pretrained=False, device="cpu")
    det.device_post = False         # the maps stay host arrays: the post-processing runs on the host, GPU or not
    rec = TextRecognizer(model_name="parseq-tiny-dynw-v4", from_pretrained=False, device="cpu", dynamic_width=True,
                         batch_bucketing=True)
    Hn, Wn = 1184, 1600
    batches, maps = [], []
    for k in range(3):
        pages, pm = [], []
        for i in range(2):
            p, q = synthetic_page(90 + 2 * k + i)
            pages.append(p)
            pm.append(synthetic_prob_map(q, (Hn, Wn), (1200, 1600)))
        batches.append(pages)
        maps.append(pm)
    det.model.input_size = lambda h, w: (Hn, Wn)
    det.model.detect_pages_u8 = lambda pages, out=None, stream=None: out
    S = rec.model.max_label_length + 1

    class FakeDev:      # stands for the flat uint8 cuda tensor of canvases
        def __init__(self, arr):
            self.arr = arr

        def data_ptr(self):
            return self.arr.ctypes.data

    def fake_extract(pages_dev, geoms, stream=None):
        sb, cb = layout_crop_buffers(geoms)
        scratch, canv = np.zeros(max(sb, 1), np.uint8), np.full(max(cb, 1), 99, np.uint8)
        pg = np.ascontiguousarray(pages_dev.numpy())
        vp = ctypes.c_void_p
        for i in sorted(set(geoms["page"].tolist())):       # the host harness takes one page at a time
            sel = np.ascontiguousarray(geoms[geoms["page"] == i])
            sel["page"] = 0
            host.crop_host_extract(pg[i].ctypes.data_as(vp), pg.shape[1], pg.shape[2], sel.ctypes.data_as(vp), len(sel),
                                   scratch.ctypes.data_as(vp), canv.ctypes.data_as(vp))
        return FakeDev(canv), cb

    def fake_ptr(ptr, on_device, total, descs, n, n_groups, stream=None):
        assert on_device == 1
        raw = np.ctypeslib.as_array(ctypes.cast(ptr, ctypes.POINTER(ctypes.c_uint8)), shape=(total,))
        ids = np.zeros((n, S), np.int32)
        for r, d in enumerate(descs):
            c = raw[int(d["pix_off"]):int(d["pix_off"]) + 32 * int(d["w"]) * 3]
            ids[r, 0] = 1 + int(c.astype(np.int64).sum()) % 7000
        return ids, np.full((n, S), 0.5, np.float32), np.full((n_groups,), S, np.int32)

    monkeypatch.setattr(M, "extract_crops_device", fake_extract)
    rec.model.run_packed_ptr = fake_ptr
    ocr = BatchedOCR(det, rec, workers=2, det_batch=1, device_crops=True)
    ocr._upload_pages = lambda stage, stream=None: stage.clone()
    try:
        got = list(ocr.stream(batches, lookahead=2, prob_override=maps))
        again = [ocr(pg, prob_override=pm) for pg, pm in zip(batches, maps)]
    finally:
        ocr.close()
    post = DBnetPostProcessor(**dict(det._cfg.post_process))
    for k in range(3):
        for i in range(2):
            quads, scores = post({"binary": maps[k][i][None, None]}, (1200, 1600))
            ds = ParseqDataset(rec._cfg, batches[k][i], quads, num_workers=1, dynamic_width=True)
            words = got[k][i].words
            assert [w.points for w in words] == quads and len(words) == len(ds) > 100
            expect = [rec.tokenizer._itos[1 + int(c.astype(np.int64).sum()) % 7000] for c in ds.data]
            assert [w.content[0] for w in words] == [unicodedata_nfkc(e)[0] for e in expect]
        assert [[w.content for w in pg.words] for pg in again[k]] == [[w.content for w in pg.words] for pg in got[k]]


def test_recognizer_call_device_crops_with_stub_models(monkeypatch):
    """CPU: TextRecognizer.__call__ on the device_crops path (records -> order -> plan -> canvases cut in plan order)
    against the host path (ParseqDataset), both with the PARSeq call replaced by a checksum stand-in; one quad is
    invalid (dropped), which also switches the bucketing off exactly like the reference."""
    import ctypes

    from oracle import build_crop_host
    from yomitoku_b200 import models as M
    from yomitoku_b200.data import layout_crop_buffers

    host = ctypes.CDLL(build_crop_host.build())
    S = 26

    def make(dev):
        rec = TextRecognizer(model_name="parseq-tiny-dynw-v4", from_pretrained=False, device="cpu", dynamic_width=True,
                             batch_bucketing=True)
        rec.device_crops = dev
        rec._upload_page = lambda img: torch.from_numpy(np.ascontiguousarray(img))[None]

        def checks(raw, descs, n, n_groups):
            # ids[0] / the score depend on WHERE the pixels are (a 180-degree turn changes them), on the padded width
            # and on the mini-batch index; position 1 is EOS, so the score is probs[0]
            ids = np.zeros((n, S), np.int32)
            probs = np.ones((n, S), np.float32)
            for r, d in enumerate(descs):
                c = raw[int(d["pix_off"]):int(d["pix_off"]) + 32 * int(d["w"]) * 3].astype(np.int64)
                h = int((c * (1 + np.arange(c.size) % 251)).sum())
                ids[r, 0] = 1 + (h * 31 + int(d["wp"]) * 7 + int(d["group"])) % 7000
                probs[r, 0] = 0.55 + 0.44 * ((h % 1000) / 1000.0)
            return ids, probs, np.full((n_groups,), S, np.int32)

        def fake_ptr(ptr, on_device, total, descs, n, n_groups, stream=None):
            raw = np.ctypeslib.as_array(ctypes.cast(ptr, ctypes.POINTER(ctypes.c_uint8)), shape=(total,))
            return checks(raw, descs, n, n_groups)

        def fake_crops(canvases, padded, groups, n_groups):
            buf, total, descs, _ = rec.model.pack_crops(canvases, padded, groups)
            return checks(buf.numpy(), [dict(pix_off=d.pix_off, w=d.w, wp=d.wp, group=d.group) for d in descs[:len(canvases)]],
                          len(canvases), n_groups)

        rec.model.run_packed_ptr = fake_ptr
        rec.model.recognize_crops = fake_crops
        return rec

    class FakeDev:
        def __init__(self, arr):
            self.arr = arr

        def data_ptr(self):
            return self.arr.ctypes.data

    def fake_extract(pages_dev, geoms, stream=None):
        sb, cb = layout_crop_buffers(geoms)
        scratch, canv = np.zeros(max(sb, 1), np.uint8), np.full(max(cb, 1), 99, np.uint8)
        pg = np.ascontiguousarray(pages_dev.numpy())
        vp = ctypes.c_void_p
        host.crop_host_extract(pg.ctypes.data_as(vp), pg.shape[1], pg.shape[2], geoms.ctypes.data_as(vp), len(geoms),
                               scratch.ctypes.data_as(vp), canv.ctypes.data_as(vp))
        return FakeDev(canv), cb

    def fake_halve(pages_dev, stream=None):
        src = np.ascontiguousarray(pages_dev.numpy())
        n, H, W, _ = src.shape
        dH, dW = int(np.rint(H * 0.5)), int(np.rint(W * 0.5))
        dst = np.zeros((n, dH, dW, 3), np.uint8)
        vp = ctypes.c_void_p
        for i in range(n):
            host.crop_host_halve(src[i].ctypes.data_as(vp), W, H, dW, dH, dst[i].ctypes.data_as(vp))
        return torch.from_numpy(dst)

    monkeypatch.setattr(M, "extract_crops_device", fake_extract)
    monkeypatch.setattr(M, "halve_pages_device", fake_halve)
    monkeypatch.setattr(M, "concat_device_buffers",
                        lambda parts, stream=None: parts[0][0] if len(parts) == 1 else
                        FakeDev(np.concatenate([t.arr[:n] for t, n in parts])))
    page, quads = synthetic_page(5)
    # source_downscale: lines with a short side of 140 / 70 / 100 px come from pyramid levels 2 / 1 / 1 (the last one is
    # vertical text); both paths must cut identical canvases from identical pyramid levels
    big = [[[100, 100], [900, 100], [900, 240], [100, 240]], [[50, 300], [700, 300], [700, 370], [50, 370]],
           [[1000, 100], [1100, 100], [1100, 900], [1000, 900]]]
    for fallback in (False, True):
        ra, rb = make(True), make(False)
        ra.source_downscale = rb.source_downscale = True
        ra.rec_orientation_fallback = rb.rec_orientation_fallback = fallback
        a, _ = ra(page[:1199, :1597], quads[:20] + big)      # odd page size: clipped last column / row of the pyramid
        b, _ = rb(page[:1199, :1597], quads[:20] + big)
        assert a.contents == b.contents and a.directions == b.directions and np.allclose(a.scores, b.scores)
        pages, geoms, levels = ra._device_records(page[:1199, :1597], quads[:20] + big)
        assert levels.tolist() == [0] * 20 + [2, 1, 1] and geoms["rot"].tolist()[-3:] == [0, 0, 1]
        M.extract_crops_pyramid(pages, geoms, levels)
        assert sorted(pages) == [0, 1, 2] and tuple(pages[2].shape) == (1, 300, 399, 3)
        assert D.pyramid_shapes((1199, 1597), 2) == [(1199, 1597), (600, 798), (300, 399)]
    tall = [[[300, 100], [330, 100], [330, 400], [300, 400]]]      # vertical line: rotated by 90 degrees first
    for fallback in (False, True):
        for qs in (quads[:70] + tall, quads[:30] + [[[-5, 3], [40, 3], [40, 20], [-5, 20]]] + quads[30:60], None):
            ra, rb = make(True), make(False)
            ra.rec_orientation_fallback = rb.rec_orientation_fallback = fallback
            a, _ = ra(page, qs)
            b, _ = rb(page, qs)
            assert a.contents == b.contents and a.directions == b.directions and a.points == b.points
            assert np.allclose(a.scores, b.scores)
            assert len(a.contents) == (1 if qs is None else 71 if len(qs) == 71 else 60)
            if fallback and qs is not None:     # the second look really replaced some results
                c, _ = make(False)(page, qs)
                assert 0 < sum(x != y for x, y in zip(b.contents, c.contents)) < len(b.contents)


def test_batched_pipeline_device_crops_source_downscale_with_stub_models(monkeypatch):
    """CPU: BatchedOCR with device_crops AND source_downscale: the workers return records + pyramid levels, the levels
    are built "on the device" (stand-in: the product's halve_pixel compiled for the host) for the whole batch, one
    extraction per level; every word must get the canvas ParseqDataset(source_downscale=True) cuts for it."""
    import ctypes

    from oracle import build_crop_host
    from yomitoku_b200 import models as M
    from yomitoku_b200.data import ParseqDataset, layout_crop_buffers
    from yomitoku_b200.pipeline import BatchedOCR

    host = ctypes.CDLL(build_crop_host.build())
    det = TextDetector(from_pretrained=False, device="cpu")
    rec = TextRecognizer(model_name="parseq-tiny-dynw-v4", from_pretrained=False, device="cpu", dynamic_width=True,
                         batch_bucketing=True, source_downscale=True)
    det.model.input_size = lambda h, w: (1184, 1600)
    det.model.detect_pages_u8 = lambda pages, out=None, stream=None: out
    S = rec.model.max_label_length + 1
    big = [[[100, 100], [900, 100], [900, 240], [100, 240]], [[50, 300], [700, 300], [700, 370], [50, 370]],
           [[1000, 100], [1100, 100], [1100, 900], [1000, 900]]]
    pages, quads = [], []
    for i in range(3):
        p, q = synthetic_page(120 + i)
        pages.append(p)
        quads.append(q[:25] + big[i:] + q[25:40])

    class FakeDev:
        def __init__(self, arr):
            self.arr = arr

        def data_ptr(self):
            return self.arr.ctypes.data

    vp = ctypes.c_void_p

    def fake_extract(pages_dev, geoms, stream=None):
        sb, cb = layout_crop_buffers(geoms)
        scratch, canv = np.zeros(max(sb, 1), np.uint8), np.full(max(cb, 1), 99, np.uint8)
        pg = np.ascontiguousarray(pages_dev.numpy())
        for i in sorted(set(geoms["page"].tolist())):
            m = geoms["page"] == i
            sel = np.ascontiguousarray(geoms[m])
            sel["page"] = 0
            host.crop_host_extract(pg[i].ctypes.data_as(vp), pg.shape[1], pg.shape[2], sel.ctypes.data_as(vp), len(sel),
                                   scratch.ctypes.data_as(vp), canv.ctypes.data_as(vp))
        return FakeDev(canv), cb

    def fake_halve(pages_dev, stream=None):
        src = np.ascontiguousarray(pages_dev.numpy())
        n, H, W, _ = src.shape
        dH, dW = int(np.rint(H * 0.5)), int(np.rint(W * 0.5))
        dst = np.zeros((n, dH, dW, 3), np.uint8)
        for i in range(n):
            host.crop_host_halve(src[i].ctypes.data_as(vp), W, H, dW, dH, dst[i].ctypes.data_as(vp))
        return torch.from_numpy(dst)

    def fake_ptr(ptr, on_device, total, descs, n, n_groups, stream=None):
        raw = np.ctypeslib.as_array(ctypes.cast(ptr, ctypes.POINTER(ctypes.c_uint8)), shape=(total,))
        ids = np.zeros((n, S), np.int32)
        for r, d in enumerate(descs):
            c = raw[int(d["pix_off"]):int(d["pix_off"]) + 32 * int(d["w"]) * 3].astype(np.int64)
            ids[r, 0] = 1 + int((c * (1 + np.arange(c.size) % 251)).sum()) % 7000
        return ids, np.full((n, S), 0.5, np.float32), np.full((n_groups,), S, np.int32)

    monkeypatch.setattr(M, "extract_crops_device", fake_extract)
    monkeypatch.setattr(M, "halve_pages_device", fake_halve)
    monkeypatch.setattr(M, "concat_device_buffers",
                        lambda parts, stream=None: parts[0][0] if len(parts) == 1 else
                        FakeDev(np.concatenate([t.arr[:n] for t, n in parts])))
    rec.model.run_packed_ptr = fake_ptr
    ocr = BatchedOCR(det, rec, workers=2, det_batch=2, device_crops=True)
    ocr._upload_pages = lambda stage, stream=None: stage.clone()
    assert ocr.device_crops
    try:
        got = ocr(pages, quads_override=quads)
    finally:
        ocr.close()
    for i in range(3):
        ds = ParseqDataset(rec._cfg, pages[i], quads[i], num_workers=1, dynamic_width=True, source_downscale=True)
        assert len(got[i].words) == len(ds) == len(quads[i])
        expect = []
        for c in ds.data:
            v = c.reshape(-1).astype(np.int64)
            expect.append(rec.tokenizer._itos[1 + int((v * (1 + np.arange(v.size) % 251)).sum()) % 7000])
        assert [w.content[0] for w in got[i].words] == [unicodedata_nfkc(e)[0] for e in expect]


def test_batched_pipeline_orientation_fallback_with_stub_models(monkeypatch):
    """CPU: BatchedOCR honours rec_orientation_fallback (it switches the batch to the device-crops path, where the second
    look is the same record with `rot |= 2`): per page the words must equal what TextRecognizer.__call__ returns on the
    host path with the fallback on (stand-in model: ids / score depend on where the pixels are, so a 180-degree turn
    changes them and some rows really get replaced)."""
    import ctypes

    from oracle import build_crop_host
    from yomitoku_b200 import models as M
    from yomitoku_b200.data import layout_crop_buffers
    from yomitoku_b200.pipeline import BatchedOCR

    host = ctypes.CDLL(build_crop_host.build())
    S = 26
    vp = ctypes.c_void_p

    def checks(raw, descs, n, n_groups):
        ids = np.zeros((n, S), np.int32)
        probs = np.ones((n, S), np.float32)
        for r, d in enumerate(descs):
            c = raw[int(d["pix_off"]):int(d["pix_off"]) + 32 * int(d["w"]) * 3].astype(np.int64)
            h = int((c * (1 + np.arange(c.size) % 251)).sum())
            ids[r, 0] = 1 + (h * 31 + int(d["wp"]) * 7) % 7000
            probs[r, 0] = 0.55 + 0.44 * ((h % 1000) / 1000.0)
        return ids, probs, np.full((n_groups,), S, np.int32)

    class FakeDev:
        def __init__(self, arr):
            self.arr = arr

        def data_ptr(self):
            return self.arr.ctypes.data

    def fake_extract(pages_dev, geoms, stream=None):
        sb, cb = layout_crop_buffers(geoms)
        scratch, canv = np.zeros(max(sb, 1), np.uint8), np.full(max(cb, 1), 99, np.uint8)
        pg = np.ascontiguousarray(pages_dev.numpy())
        for i in sorted(set(geoms["page"].tolist())):
            sel = np.ascontiguousarray(geoms[geoms["page"] == i])
            sel["page"] = 0
            host.crop_host_extract(pg[i].ctypes.data_as(vp), pg.shape[1], pg.shape[2], sel.ctypes.data_as(vp), len(sel),
                                   scratch.ctypes.data_as(vp), canv.ctypes.data_as(vp))
        return FakeDev(canv), cb

    monkeypatch.setattr(M, "extract_crops_device", fake_extract)
    det = TextDetector(from_pretrained=False, device="cpu")
    det.model.input_size = lambda h, w: (1184, 1600)
    det.model.detect_pages_u8 = lambda pages, out=None, stream=None: out
    rec = TextRecognizer(model_name="parseq-tiny-dynw-v4", from_pretrained=False, device="cpu", dynamic_width=True,
                         batch_bucketing=True, rec_orientation_fallback=True, rec_orientation_fallback_thresh=0.75)

    def fake_ptr(ptr, on_device, total, descs, n, n_groups, stream=None):
        raw = np.ctypeslib.as_array(ctypes.cast(ptr, ctypes.POINTER(ctypes.c_uint8)), shape=(total,))
        return checks(raw, descs, n, n_groups)

    def fake_crops(canvases, padded, groups, n_groups):
        buf, total, descs, _ = rec.model.pack_crops(canvases, padded, groups)
        return checks(buf.numpy(), [dict(pix_off=d.pix_off, w=d.w, wp=d.wp) for d in descs[:len(canvases)]],
                      len(canvases), n_groups)

    rec.model.run_packed_ptr = fake_ptr
    rec.model.recognize_crops = fake_crops
    pages, quads = [], []
    for i in range(3):
        p, q = synthetic_page(130 + i)
        pages.append(p)
        quads.append(q[:37] + [[[1000, 100], [1030, 100], [1030, 600], [1000, 600]]])     # + one vertical line
    ocr = BatchedOCR(det, rec, workers=2, det_batch=2)            # device_crops not requested: the flag switches it on
    ocr._upload_pages = lambda stage, stream=None: stage.clone()
    try:
        got = ocr(pages, quads_override=quads)
    finally:
        ocr.close()
    replaced = 0
    for i in range(3):
        rec.device_crops = False
        single, _ = rec(pages[i], quads[i])                        # host path incl. _apply_orientation_fallback
        rec.rec_orientation_fallback = False
        plain, _ = rec(pages[i], quads[i])
        rec.rec_orientation_fallback = True
        assert [w.content for w in got[i].words] == single.contents
        assert np.allclose([w.rec_score for w in got[i].words], single.scores)
        replaced += sum(a != b for a, b in zip(single.contents, plain.contents))
    assert replaced > 0


def test_product_never_imports_the_oracle():
    """The oracle (and everything under tests/) is checker-only: no module of the product package may import it, and the
    product must load without it on the path."""
    import ast
    import glob
    import subprocess
    import sys
    pkg = os.path.join(os.path.dirname(HERE), "yomitoku_b200")
    for f in glob.glob(os.path.join(pkg, "*.py")):
        for node in ast.walk(ast.parse(open(f, encoding="utf-8").read())):
            names = []
            if isinstance(node, ast.Import):
                names = [a.name for a in node.names]
            elif isinstance(node, ast.ImportFrom) and node.level == 0:
                names = [node.module or ""]
            assert not any(n.split(".")[0] in ("oracle", "tests") for n in names), (f, names)
    code = ("import sys; sys.path = [p for p in sys.path if p not in ('', %r)]; sys.path.insert(0, %r); "
            "import importlib, yomitoku_b200; "
            "[importlib.import_module('yomitoku_b200.' + m) for m in ('pipeline', 'parallel', 'models', 'ocr')]; "
            "assert 'oracle' not in sys.modules" % (os.path.dirname(HERE), os.path.dirname(HERE)))
    # the repo root is needed to find the package itself; the assertion is that importing it pulls in no oracle module
    assert subprocess.run([sys.executable, "-c", code], cwd="/", capture_output=True).returncode == 0


def test_vectorised_clipper_offset_equals_scalar_routine():
    """postprocessor.offset_boxes_round (one page's boxes at once) == offset_convex_polygon_round box by box: same
    double-precision operations in the same order, so equality, not tolerance - including boxes whose integer
    truncation collapses vertices (handled by the scalar fallback)."""
    import cv2
    from yomitoku_b200.postprocessor import offset_boxes_round, offset_convex_polygon_round
    rng = np.random.default_rng(3)
    boxes, deltas = [], []
    for i in range(600):
        c = rng.uniform(50, 1500, 2)
        size = (float(rng.uniform(3, 400)), float(rng.uniform(3, 60))) if i % 7 else \
            (float(rng.uniform(0.2, 2.5)), float(rng.uniform(0.2, 2.5)))
        ang = float(rng.uniform(-90, 90)) if i % 3 else 0.0
        boxes.append(cv2.boxPoints(((float(c[0]), float(c[1])), size, ang)))
        deltas.append(float(rng.uniform(0.5, 12)))
    ref = [offset_convex_polygon_round(b, d) for b, d in zip(boxes, deltas)]
    got = offset_boxes_round(np.array(boxes), np.array(deltas))
    for a, b in zip(ref, got):
        assert a.shape == b.shape and np.array_equal(a, b)
    assert offset_boxes_round(np.zeros((0, 4, 2)), np.zeros(0)) == []


# ------------------------------------------------------------------ device front half of the post-processing (host side)
def _blob_map(seed, holes):
    """Random map of rotated blurred boxes; `holes` punches low-probability dots into some of them."""
    import cv2
    rng = np.random.default_rng(seed)
    H, W = 300, 420
    m = np.zeros((H, W), np.float32)
    for _ in range(30):
        c = (float(rng.integers(20, W - 20)), float(rng.integers(20, H - 20)))
        wh = (float(rng.integers(6, 90)), float(rng.integers(4, 30)))
        cv2.fillPoly(m, [cv2.boxPoints((c, wh, float(rng.uniform(-40, 40)))).astype(np.int32)], float(rng.uniform(0.5, 1.0)))
    m = cv2.GaussianBlur(m, (7, 7), 0)
    m += rng.uniform(0, 0.02, m.shape).astype(np.float32)
    if holes:
        ys, xs = np.nonzero(m > 0.6)
        for k in rng.integers(0, len(ys), 5):
            m[ys[k], xs[k]] = 0.0
    return m


def test_boxes_from_runs_equals_boxes_from_bitmap():
    """DBnetPostProcessor.boxes_from_runs (input: what csrc/dbpost_ops.cu emits, here from the scipy twin in
    oracle/dbpost.py) returns the quads of boxes_from_bitmap (OpenCV contours) on every map without holes."""
    from oracle.dbpost import post_front
    from yomitoku_b200.synth import synthetic_page, synthetic_prob_map
    pp = DBnetPostProcessor(min_size=2, thresh=0.3, box_thresh=0.4, max_candidates=1500, unclip_ratio=3.5)
    checked = 0
    maps = [(_blob_map(s, False), (840, 600)) for s in range(12)]
    _, quads = synthetic_page(3)
    maps.append((synthetic_prob_map(quads, (1184, 1600), (1200, 1600)), (1600, 1200)))
    for prob, (dw, dh) in maps:
        runs, comps, holes = post_front(prob, pp.thresh)
        if holes:
            continue
        b1, s1 = pp.boxes_from_bitmap(prob, prob > pp.thresh, dw, dh)
        b2, s2 = pp.boxes_from_runs(runs, prob.shape[1], prob.shape[0], dw, dh)
        assert b1 == b2 and len(b1) > 0
        assert np.allclose(s1, s2, rtol=1e-12, atol=0)
        checked += 1
    assert checked >= 6


def test_boxes_from_runs_order_and_limit():
    """max_candidates keeps OpenCV's FIRST contours = the components with the largest first-pixel index."""
    from oracle.dbpost import post_front
    prob = _blob_map(110, False)
    runs, comps, holes = post_front(prob, 0.3)
    if holes:
        pytest.skip("map has holes")
    pp = DBnetPostProcessor(min_size=2, thresh=0.3, box_thresh=0.4, max_candidates=5, unclip_ratio=3.5)
    b1, s1 = pp.boxes_from_bitmap(prob, prob > 0.3, 420, 300)
    b2, s2 = pp.boxes_from_runs(runs[::-1].copy(), 420, 300, 420, 300)
    # quads are integers: identical; the score is the same fp64 mean summed in another order (run by run instead of
    # cv2.mean's raster order): equal to a few ulp
    assert b1 == b2 and 0 < len(b1) <= 5 and np.allclose(s1, s2, rtol=1e-12, atol=0)


def test_hole_count_matches_opencv_contour_count():
    """#contours of cv2.findContours(RETR_LIST) = #components + #holes: the invariant behind the host fallback."""
    import cv2
    from oracle.dbpost import post_front
    seen_holes = 0
    for s in range(8):
        prob = _blob_map(200 + s, holes=True)
        runs, comps, holes = post_front(prob, 0.3)
        contours, _ = cv2.findContours((prob > 0.3).astype(np.uint8) * 255, cv2.RETR_LIST, cv2.CHAIN_APPROX_SIMPLE)
        assert len(contours) == comps + holes
        seen_holes += holes
    assert seen_holes > 0


def test_gelu_coefficients_in_kernel_source():
    """The fc1 epilogue's GELU (csrc/gemm_tc.cu: gelu_fast2) evaluated in numpy fp32 with the coefficients read from the
    source: max |error| against the fp64 erf GELU (torch.nn.GELU default of reference parseq.py's MLP) below 6e-7."""
    import re
    from scipy import special
    src = open(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "yomitoku_b200", "csrc",
                            "gemm_tc.cu")).read()
    body = src[src.index("void gelu_fast2(float& x0, float& x1) {"):]
    body = body[:body.index("upk2(r, x0, x1);")]
    clamp = float(re.search(r"fminf\(fabsf\(x0\), ([0-9.]+)f\)", body).group(1))
    coefs = [float(m) for m in re.findall(r"pk2\((-?[0-9.]+e[+-][0-9]+)f,", body)]        # highest power first
    assert len(coefs) == 7 and clamp == 5.7
    x = np.concatenate([np.linspace(-12, 12, 400001), [-1e4, 1e4, 0.0]]).astype(np.float32)
    t = np.minimum(np.abs(x), np.float32(clamp))
    p = np.full_like(t, np.float32(coefs[0]))
    for c in coefs[1:]:
        p = p * t + np.float32(c)
    g = np.maximum(x, np.float32(0)) + (np.float32(-0.5) * t) * np.exp2(p * t)
    ref = 0.5 * x.astype(np.float64) * (1 + special.erf(x.astype(np.float64) / np.sqrt(2)))
    assert np.abs(g - ref).max() < 6e-7
