"""CellDetector: RT-DETRv2 cell detection on table crops (960 x 960 input, 1500 queries), cells and hole cells from the
detections.

Mirrors reference src/yomitoku/table_cell_detector.py:34-522 (catalog name `rtdetrv2`, constructor kwargs,
`preprocess` / `postprocess` / `extract_cell_elements` / `remove_noise_cells` / `__call__`, TableDetectorSchema) and
the adjacency tests it uses (utils/misc.py:208-420, rule "soft").  All table crops of a page go through the device model
as ONE batch (the reference runs them one by one); the geometry behind it is host code like in the reference.
"""
import math

import cv2
import numpy as np
import torch

from .base import BaseModelCatalog, BaseModule, logger
from .config import TableCellParserRTDETRv2Config
from .document_analyzer import _intersection
from .layout_parser import (filter_contained_rectangles_across_categories, filter_contained_rectangles_within_category,
                            rtdetr_input_tensor)
from .models import RTDETRv2
from .postprocessor import RTDETRPostProcessor
from .schemas import CellSchema, RegionSchema, TableDetectorSchema


class TableParserModelCatalog(BaseModelCatalog):
    def __init__(self):
        super().__init__()
        self.register("rtdetrv2", TableCellParserRTDETRv2Config, RTDETRv2)


def calc_iou(a, b):
    """Intersection over union of two xyxy boxes (utils/misc.py:182-201)."""
    inter = _intersection(a, b)
    if inter is None:
        return 0
    ov = (inter[2] - inter[0]) * (inter[3] - inter[1])
    return ov / ((a[2] - a[0]) * (a[3] - a[1]) + (b[2] - b[0]) * (b[3] - b[1]) - ov)


def find_holes_as_rects(table_shape, cell_boxes, pad=2, close_ksize=5, min_area=300):
    """Regions of the table that no cell box covers and that do not touch the crop's border (filled cell rectangles,
    morphological opening x3, flood fill from the corner, external contours), as padded rectangles; reference :97-127."""
    mask = np.full((table_shape[0], table_shape[1]), 255, np.uint8)
    for box in cell_boxes:
        x1, y1, x2, y2 = (int(v) for v in box)
        cv2.rectangle(mask, (x1, y1), (x2, y2), 0, thickness=-1)
    if close_ksize > 1:
        k = cv2.getStructuringElement(cv2.MORPH_RECT, (close_ksize, close_ksize))
        mask = cv2.morphologyEx(mask, cv2.MORPH_OPEN, k, iterations=3)
    h, w = mask.shape
    cv2.floodFill(mask, np.zeros((h + 2, w + 2), np.uint8), (0, 0), 0)
    cnts, _ = cv2.findContours(mask, cv2.RETR_EXTERNAL, cv2.CHAIN_APPROX_SIMPLE)
    rects = []
    for c in cnts:
        x, y, rw, rh = cv2.boundingRect(c)
        if rw * rh >= min_area:
            rects.append([x - pad, y - pad, x + rw + pad, y + rh + pad])
    return rects


def choose_role(role_counts):
    """The most frequent neighbour role; a tie that involves "cell" is "cell" (reference :130-141)."""
    if not role_counts:
        return None
    max_count = max(role_counts.values())
    candidates = [r for r, c in role_counts.items() if c == max_count]
    if len(candidates) > 1 and "cell" in candidates:
        return "cell"
    return candidates[0]


def _point_to_segment(px, py, ax, ay, bx, by):
    abx, aby = bx - ax, by - ay
    denom = abx * abx + aby * aby
    if denom == 0:
        return math.hypot(px - ax, py - ay)
    t = min(1.0, max(0.0, ((px - ax) * abx + (py - ay) * aby) / denom))
    return math.hypot(px - (ax + t * abx), py - (ay + t * aby))


def _overlap(i1, i2, j1, j2):
    return max(0.0, min(i2, j2) - max(i1, j1))


def is_right_adjacent(a, b, dist_threshold=15, overlap_ratio_th=0.1, ignore_dist_threshold=10):
    """b lies right next to a: b starts right of a's left edge, the two overlap vertically by >= 10 % of the shorter one,
    no two facing corners are closer than `ignore_dist_threshold` diagonally, and one of the four corner-to-edge
    distances is below `dist_threshold` (utils/misc.py:299-355, rule "soft")."""
    ax1, ay1, ax2, ay2 = a
    bx1, by1, bx2, by2 = b
    if bx1 < ax1:
        return False
    if _overlap(ay1, ay2, by1, by2) < overlap_ratio_th * min(ay2 - ay1, by2 - by1):
        return False
    if (math.hypot(ax2 - bx1, ay2 - by1) < ignore_dist_threshold or
            math.hypot(ax2 - bx1, ay1 - by2) < ignore_dist_threshold):
        return False
    d1 = _point_to_segment(ax2, ay1, bx1, by1, bx1, by2)
    d2 = _point_to_segment(ax2, ay2, bx1, by1, bx1, by2)
    d3 = _point_to_segment(bx1, by1, ax2, ay1, ax2, ay2)
    d4 = _point_to_segment(bx1, by2, ax2, ay1, ax2, ay2)
    return min(max(d1, d4), max(d2, d3), max(d3, d4), max(d1, d2)) < dist_threshold


def is_bottom_adjacent(a, b, dist_threshold=15, overlap_ratio_th=0.1, ignore_dist_threshold=10):
    """b lies right below a: the vertical counterpart of is_right_adjacent (utils/misc.py:358-420, rule "soft")."""
    ax1, ay1, ax2, ay2 = a
    bx1, by1, bx2, by2 = b
    if by1 < ay1:
        return False
    if _overlap(ax1, ax2, bx1, bx2) < overlap_ratio_th * min(ax2 - ax1, bx2 - bx1):
        return False
    if (math.hypot(ax2 - bx1, ay2 - by1) < ignore_dist_threshold or
            math.hypot(ax1 - bx2, ay2 - by1) < ignore_dist_threshold):
        return False
    d1 = _point_to_segment(ax1, ay2, bx1, by1, bx2, by1)
    d2 = _point_to_segment(ax2, ay2, bx1, by1, bx2, by1)
    d3 = _point_to_segment(bx1, by1, ax1, ay2, ax2, ay2)
    d4 = _point_to_segment(bx2, by1, ax1, ay2, ax2, ay2)
    return min(max(d1, d4), max(d2, d3), max(d3, d4), max(d1, d2)) < dist_threshold


def calc_adjacent_holes_to_cells(holes, cells):
    """A hole is kept when cells border it from more than two of its four sides; it takes the role most of those
    neighbours have (reference :144-180)."""
    kept = []
    for hole in holes:
        edges = {d: 0 for d in "RLDU"}
        roles = {r: 0 for r in ("cell", "header", "empty")}
        for node in cells:
            for d, hit in (("R", is_right_adjacent(hole["box"], node["box"])),
                           ("L", is_right_adjacent(node["box"], hole["box"])),
                           ("D", is_bottom_adjacent(hole["box"], node["box"])),
                           ("U", is_bottom_adjacent(node["box"], hole["box"]))):
                if hit:
                    edges[d] += 1
                    roles[node["role"]] += 1
        if sum(c > 0 for c in edges.values()) > 2:
            hole["role"] = choose_role(roles)
            kept.append(hole)
    return kept


class CellDetector(BaseModule):
    model_catalog = TableParserModelCatalog()

    def __init__(self, model_name="rtdetrv2", path_cfg=None, device="cuda", visualize=False, from_pretrained=True,
                 infer_onnx=False):
        super().__init__()
        self.load_model(model_name, path_cfg, from_pretrained=from_pretrained)
        if getattr(self._cfg, "weights_path", None):
            raise NotImplementedError("CellDetector: local training checkpoints (weights_path) are not supported, load a "
                                      "state_dict into .model instead")
        if infer_onnx:
            logger.warning("CellDetector(infer_onnx=True): there is no ONNX path in yomitoku_b200, the CUDA engine is used")
        self.infer_onnx = False
        self.device = device
        self.visualize = visualize
        self.model.eval().to(self.device)
        dec = self._cfg.RTDETRTransformerv2
        self.postprocessor = RTDETRPostProcessor(num_classes=dec.num_classes, num_top_queries=dec.num_queries)
        self.thresh_score = self._cfg.thresh_score
        self.label_mapper = dict(enumerate(self._cfg.category))

    def preprocess(self, img, tables):
        """BGR page + tables (objects with .box) -> per table {"tensor" (1, 3, 960, 960), "size" (h, w), "offset"
        (x1, y1)}; reference :315-334."""
        rgb = cv2.cvtColor(img, cv2.COLOR_BGR2RGB)
        out = []
        for table in tables:
            x1, y1, x2, y2 = (int(v) for v in table.box)
            crop = rgb[y1:y2, x1:x2, :]
            out.append({"tensor": rtdetr_input_tensor(np.ascontiguousarray(crop), self._cfg.data.img_size),
                        "size": crop.shape[:2], "offset": (x1, y1)})
        return out

    def is_fully_contained(self, box1, box2, threshold=0.9):
        return calc_iou(box1, box2) >= threshold

    def postprocess(self, preds, data, table_box):
        """Detections of one crop -> (cells, kv_regions, grid_regions) in page coordinates; reference :351-467."""
        h, w = data["size"]
        det = self.postprocessor(preds, np.array([[w, h]], np.float32), self.thresh_score)[0]
        elements = {c: [] for c in self.label_mapper.values()}
        elements["hole"] = []
        for box, score, label in zip(det["boxes"], det["scores"], det["labels"]):
            category = self.label_mapper[int(label)]
            box = box.astype(int).tolist()
            # grid / kv_item regions may cover the whole table: only the other classes lose crop-sized boxes
            if category not in ("grid", "kv_item") and self.is_fully_contained(box, [0, 0, w, h]):
                continue
            elements[category].append({"box": box, "score": float(score), "role": category})
        elements = filter_contained_rectangles_within_category(elements, ignore=("kv_item", "grid"), drop_outer=True)
        elements = filter_contained_rectangles_across_categories(elements, "cell", "header")
        elements = filter_contained_rectangles_across_categories(elements, "cell", "empty")
        cell_boxes = elements["cell"] + elements["header"] + elements["empty"]
        for box in find_holes_as_rects(data["size"], [c["box"] for c in cell_boxes]):
            elements["hole"].append({"box": box, "score": 1.0, "role": "hole"})
        ox, oy = data["offset"]
        for values in elements.values():
            for e in values:
                e["box"] = [e["box"][0] + ox, e["box"][1] + oy, e["box"][2] + ox, e["box"][3] + oy]
        if not cell_boxes:
            elements["cell"] = [{"box": list(table_box), "role": "cell"}]      # no cell found: the table is one cell
        cells = self.remove_noise_cells(self.extract_cell_elements(elements), min_width=10, min_height=10)
        kv_regions = [RegionSchema(id=None, box=e["box"], role="kv_item", score=e["score"]) for e in elements["kv_item"]]
        grid_regions = [RegionSchema(id=None, box=e["box"], role="grid", score=e["score"]) for e in elements["grid"]]
        return cells, kv_regions, grid_regions

    def remove_noise_cells(self, cells, min_width=30, min_height=30):
        return [c for c in cells if c.box[2] - c.box[0] > min_width and c.box[3] - c.box[1] > min_height]

    def extract_cell_elements(self, elements):
        elements["hole"] = calc_adjacent_holes_to_cells(elements["hole"],
                                                        elements["cell"] + elements["header"] + elements["empty"])
        cells = []
        for category, values in elements.items():
            if category in ("cell", "header", "empty", "group", "hole"):
                for v in values:
                    cells.append(CellSchema(id="c%d" % len(cells), box=v["box"], role=v["role"], contents=None, row=None,
                                            col=None, row_span=None, col_span=None))
        return cells

    def __call__(self, img, tables):
        data = self.preprocess(img, tables)
        outputs = []
        if not data:
            return outputs
        preds = self.model(torch.cat([d["tensor"] for d in data]))           # every table of the page in one batch
        for i, (d, table) in enumerate(zip(data, tables)):
            cells, kv_regions, grid_regions = self.postprocess({k: v[i:i + 1] for k, v in preds.items()}, d, table.box)
            if cells:
                outputs.append(TableDetectorSchema(id=None, box=table.box, role=table.role, cells=cells,
                                                   kv_regions=kv_regions, grid_regions=grid_regions))
        return outputs
