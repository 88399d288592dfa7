"""Generates tests/golden/cell_ref.npz and tests/golden/cell_wrappers_ref.json from the reference's OWN files, executed
from the reference tree by path (oracle/refcheck.py locates it):

  cell_ref.npz              models/rtdetr.py at the cell detector's configuration (configs/cfg_table_cell_parser_rtdtrv2.py:
                            960 x 960, 1500 queries, 6 classes) with the seeded weights of oracle.rtdetr.make_state_dict
                            on a seeded table-like input - pred_logits / pred_boxes, the three backbone and encoder maps
                            (means of 8x8 blocks), encoder scores and the top-1500 anchors
  cell_wrappers_ref.json    table_cell_detector.py (CellDetector.preprocess / postprocess / extract_cell_elements /
                            remove_noise_cells and the helpers behind them) with the real utils/misc.py and
                            schemas/table_semantic_parser.py around the reference's postprocessor/rtdetr_postprocessor.py,
                            fed with seeded fake model outputs; modules this logic never executes (onnx*, base, configs,
                            models, logger, reading_order) are stand-ins.  Also the reference config's values.
Usage: python tests/golden/make_golden_cell.py
"""
import dataclasses
import json
import os
import sys
import types

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, HERE)
from make_golden_rtdetr import plain, pooled  # noqa: E402
from oracle import refcheck as rc  # noqa: E402
from oracle import rtdetr as R  # noqa: E402

CELL_SPEC = R.RTDETRSpec(num_classes=6, num_queries=1500, img_size=[960, 960])
MODEL_SEED, INPUT_SEED = 31, 41


def cell_input(seed, n=1):
    """Seeded table-crop-like input in [0, 1]: light background, a ruled grid of cells, dark text-like blobs."""
    g = torch.Generator().manual_seed(seed)
    x = torch.rand(n, 3, 24, 24, generator=g)
    x = torch.nn.functional.interpolate(x, size=(960, 960), mode="bilinear", align_corners=False) * 0.2 + 0.75
    for b in range(n):
        nr, nc = torch.randint(4, 12, (2,), generator=g).tolist()
        ys = sorted(torch.randint(20, 940, (nr,), generator=g).tolist())
        xs = sorted(torch.randint(20, 940, (nc,), generator=g).tolist())
        for y in ys:
            x[b, :, y:y + 3, :] = 0.1
        for v in xs:
            x[b, :, :, v:v + 3] = 0.1
        for _ in range(30):
            x0, y0 = torch.randint(0, 900, (2,), generator=g).tolist()
            w, h = torch.randint(10, 60, (1,), generator=g).item(), torch.randint(6, 20, (1,), generator=g).item()
            x[b, :, y0:y0 + h, x0:x0 + w] = torch.rand(3, 1, 1, generator=g) * 0.3
    return x.contiguous()


def reference_cell_config():
    """The values of the reference's own configs/cfg_table_cell_parser_rtdtrv2.py as a plain dict."""
    mod = rc._load("ytk_ref_cfg_table_cell_parser_rtdtrv2", "configs/cfg_table_cell_parser_rtdtrv2.py")
    return dataclasses.asdict(mod.TableCellParserRTDETRv2Config())


def build_reference_cell_model(sd):
    """The reference's models/rtdetr.py RTDETRv2 built from its cell detector config (960 x 960, 1500 queries)."""
    RTDETRv2, _ = rc.load_reference_rtdetr()
    cfg = reference_cell_config()
    dec = dict(cfg["RTDETRTransformerv2"])
    dec["num_points"] = sys.modules["omegaconf"].ListConfig(dec["num_points"])    # what OmegaConf hands the decoder
    m = RTDETRv2(rc.AttrDict(PResNet=cfg["PResNet"], HybridEncoder=cfg["HybridEncoder"], RTDETRTransformerv2=dec))
    m.load_state_dict(sd, strict=True)
    return m.eval()


def model_case():
    sd = R.make_state_dict(CELL_SPEC, seed=MODEL_SEED)
    net = build_reference_cell_model(sd)
    x = cell_input(INPUT_SEED)
    with torch.no_grad():
        feats = net.backbone(x)
        enc = net.encoder(feats)
        res = net.decoder(enc)
        memory, _ = net.decoder._get_encoder_input(enc)
        om = net.decoder.enc_output(net.decoder.valid_mask.to(memory.dtype) * memory)
        scores = net.decoder.enc_score_head(om).max(-1).values[0]
    out = {"logits": res["pred_logits"][0].numpy(), "boxes": res["pred_boxes"][0].numpy()}
    for i in range(3):
        out["c%d" % (i + 3)] = pooled(feats[i])
        out["e%d" % (i + 3)] = pooled(enc[i])
    out["enc_scores"] = scores.numpy()
    out["topk"] = torch.topk(scores, 1500).indices.numpy().astype(np.int32)
    return out


# ------------------------------------------------------------------------------------------------ host wrappers
CELL_CASES = [  # (seed, table box on the page)
    (300, [40, 60, 700, 520]), (301, [10, 10, 890, 690]), (302, [100, 50, 500, 400]), (303, [0, 0, 900, 700]),
    (304, [200, 300, 860, 690]), (305, [60, 20, 640, 300]), (306, [5, 100, 455, 650]), (307, [300, 40, 880, 620]),
]


def cell_preds(seed, size):
    """Model outputs (1, 1500, 6) for a crop of `size` (h, w) that decode to a grid of cells (class 1) with header
    (2) and empty (3) cells, missing cells (holes, some bordered on every side, some not), nested same-class boxes,
    cells inside headers / empties and the reverse, crop-covering table / grid / kv_item / cell boxes, kv_item / grid
    regions and cells under 10 px.  Seeds ending in 3 detect no cell at all (the whole table becomes one cell)."""
    rng = np.random.default_rng(seed)
    h, w = size
    logits = np.full((1, 1500, 6), -6.0, np.float32)
    boxes = rng.uniform(0.05, 0.95, (1, 1500, 4)).astype(np.float32)
    q = [0]

    def add(x1, y1, x2, y2, cls, score=None):           # pixel box -> normalised cxcywh
        boxes[0, q[0]] = ((x1 + x2) / 2 / w, (y1 + y2) / 2 / h, (x2 - x1) / w, (y2 - y1) / h)
        logits[0, q[0], cls] = rng.uniform(0.5, 4.0) if score is None else score
        q[0] += 1

    add(0, 0, w, h, 0)                                    # the table itself: crop-sized, dropped
    add(2, 1, w - 1, h - 2, 5)                            # crop-covering grid / kv_item regions: kept as regions
    add(1, 2, w - 2, h - 1, 4)
    if seed % 10 == 3:
        add(w * 0.2, h * 0.2, w * 0.6, h * 0.5, 4)
        return {"pred_logits": torch.from_numpy(logits), "pred_boxes": torch.from_numpy(boxes)}
    add(1, 1, w - 1, h - 1, 1)                            # a crop-sized cell: dropped
    nr, nc = int(rng.integers(4, 9)), int(rng.integers(4, 7))
    mx, my = rng.uniform(0.03, 0.08) * w, rng.uniform(0.03, 0.08) * h
    cw, ch = (w - 2 * mx) / nc, (h - 2 * my) / nr
    missing = {(int(rng.integers(1, nr - 1)), int(rng.integers(1, nc - 1))) for _ in range(int(rng.integers(1, 4)))}
    if rng.uniform() < 0.5:                               # a missing 1 x 2 block: a wider hole
        r, c = int(rng.integers(1, nr - 1)), int(rng.integers(1, nc - 2))
        missing |= {(r, c), (r, c + 1)}
    # two missing slots become frames of four cells around a small gap: 14 px (below the hole area limit: dropped)
    # and 26 px (a hole)
    frames = dict(zip(sorted(missing)[:2], (14, 26))) if seed % 2 == 0 else {}
    for r in range(nr):
        for c in range(nc):
            if (r, c) in frames:
                x1, y1, s = mx + c * cw + 1, my + r * ch + 1, frames[(r, c)] / 2
                x2, y2, cx, cy = x1 + cw - 2, y1 + ch - 2, x1 + cw / 2, y1 + ch / 2
                for fb in ((x1, y1, x2, cy - s), (x1, cy + s, x2, y2), (x1, cy - s, cx - s, cy + s),
                           (cx + s, cy - s, x2, cy + s)):
                    add(*fb, 1)
            if (r, c) in missing:
                continue
            gap = rng.uniform(0, 3)
            x1, y1 = mx + c * cw + gap, my + r * ch + gap
            x2, y2 = x1 + cw - 2 * gap, y1 + ch - 2 * gap
            cls = 2 if r == 0 else (3 if rng.uniform() < 0.1 else 1)
            add(x1, y1, x2, y2, cls)
            u = rng.uniform()
            if u < 0.08:                                  # a same-class box inside: the enclosing one is dropped
                add(x1 + 4, y1 + 3, x2 - 5, y2 - 4, cls)
            elif u < 0.16 and cls == 1:                   # a header / empty box inside a cell: dropped
                add(x1 + 3, y1 + 3, x2 - 3, y2 - 3, int(rng.integers(2, 4)))
            elif u < 0.24 and cls != 1:                   # a cell inside a header / empty: both stay
                add(x1 + 3, y1 + 3, x2 - 3, y2 - 3, 1)
    for _ in range(2):                                    # cells under 10 px: removed as noise
        x0, y0 = rng.uniform(0.1, 0.8) * w, rng.uniform(0.1, 0.8) * h
        add(x0, y0, x0 + rng.uniform(3, 9), y0 + rng.uniform(3, 30), 1)
    add(mx, my, mx + 2 * cw, my + ch, 4)                  # kv_item regions, one inside another (not filtered)
    add(mx + 2, my + 2, mx + cw, my + ch - 2, 4)
    add(mx + cw, my + ch, w - mx, h - my, 5)
    add(mx, my, mx + cw, my + ch, 3, score=0.1)           # below the threshold
    return {"pred_logits": torch.from_numpy(logits), "pred_boxes": torch.from_numpy(boxes)}


def cell_page():
    return np.random.default_rng(7).integers(0, 255, (700, 900, 3), dtype=np.uint8)


def load_reference_cell_detector():
    import importlib.machinery
    from pydantic import BaseModel, ConfigDict
    rc.load_reference_rtdetr()

    def stub(name, **attrs):
        m = sys.modules.get(name) or types.ModuleType(name)
        m.__spec__ = importlib.machinery.ModuleSpec(name, None)
        m.__path__ = []
        for k, v in attrs.items():
            setattr(m, k, v)
        sys.modules[name] = m
        return m

    class BaseSchema(BaseModel):                 # reference base.py:51-57 (pydantic v1 Config, the same options)
        model_config = ConfigDict(extra="forbid", validate_assignment=True)

    class Catalog:
        def register(self, *a):
            pass

    added = [n for n in ("onnx", "onnxruntime") if n not in sys.modules]
    for n in added:
        stub(n)
    rc._pkg("ytk_ref.utils")
    stub("ytk_ref.constants", ROOT_DIR="/nonexistent")
    stub("ytk_ref.base", BaseModelCatalog=Catalog, BaseModule=object, load_config=None, BaseSchema=BaseSchema)
    stub("ytk_ref.configs", TableCellParserRTDETRv2Config=None)
    sys.modules["ytk_ref.models"].RTDETRv2 = None
    sys.modules["ytk_ref.postprocessor"].RTDETRPostProcessor = sys.modules[
        "ytk_ref.postprocessor.rtdetr_postprocessor"].RTDETRPostProcessor
    rc._load("ytk_ref.utils.misc", "utils/misc.py", "ytk_ref.utils")
    stub("ytk_ref.utils.logger", set_logger=lambda *a, **k: None)
    stub("ytk_ref.reading_order", prediction_reading_order=None)
    stub("ytk_ref.schemas", WordPrediction=None, ParagraphSchema=None, Element=None)
    try:
        rc._load("ytk_ref.schemas.table_semantic_parser", "schemas/table_semantic_parser.py", "ytk_ref.schemas")
        cd = rc._load("ytk_ref.table_cell_detector", "table_cell_detector.py", "ytk_ref")
    finally:
        for n in added:
            sys.modules.pop(n, None)
    return cd, reference_cell_config()


def reference_cell_detector(cd, cfg):
    import torchvision.transforms as T
    d = object.__new__(cd.CellDetector)
    d._cfg = rc.AttrDict(data=rc.AttrDict(img_size=cfg["data"]["img_size"]))
    d.device, d.visualize, d.infer_onnx = "cpu", False, False
    d.postprocessor = cd.RTDETRPostProcessor(num_classes=6, num_top_queries=1500)
    d.transforms = T.Compose([T.Resize(cfg["data"]["img_size"]), T.ToTensor()])
    d.thresh_score = cfg["thresh_score"]
    d.label_mapper = dict(enumerate(cfg["category"]))
    return d


def run_cases(det, page, cases):
    """[{seed, box, tensor_sum, cells, kv_regions, grid_regions}] of a detector (reference or product) on `page`."""
    out = []
    for seed, box in cases:
        table = types.SimpleNamespace(box=list(box), role=None)
        data = det.preprocess(page, [table])[0]
        cells, kv, grid = det.postprocess(cell_preds(seed, data["size"]), data, list(box))
        out.append({"seed": seed, "box": list(box), "tensor_sum": float(data["tensor"].double().sum()),
                    "cells": [plain(c.model_dump()) for c in cells], "kv_regions": [plain(r.model_dump()) for r in kv],
                    "grid_regions": [plain(r.model_dump()) for r in grid]})
    return out


def wrapper_cases():
    cd, cfg = load_reference_cell_detector()
    det = reference_cell_detector(cd, cfg)
    return {"config": cfg, "cases": run_cases(det, cell_page(), CELL_CASES)}


if __name__ == "__main__":
    np.savez_compressed(os.path.join(HERE, "cell_ref.npz"), **model_case())
    with open(os.path.join(HERE, "cell_wrappers_ref.json"), "w") as f:
        json.dump(wrapper_cases(), f)
    print("wrote cell_ref.npz, cell_wrappers_ref.json")
