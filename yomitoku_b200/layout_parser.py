"""LayoutParser: RT-DETRv2 page-layout detection behind the reference's module API.

Mirrors reference src/yomitoku/layout_parser.py:23-274 - same catalog names (`rtdetrv2`, `rtdetrv2v2`), constructor
kwargs, `preprocess` / `postprocess` / `filtering_elements` / `__call__` contract and result schema.  The model forward
runs as sm_100a kernels (csrc/rtdetr_engine.cu behind ytk_rtdetr_forward_f32); the PIL resize in front of it and the
containment filters behind it are host code like in the reference.  `infer_onnx` is accepted and ignored.
"""
import cv2
import numpy as np
import torch
from PIL import Image

from .base import BaseModelCatalog, BaseModule, logger
from .config import LayoutParserRTDETRv2Config, LayoutParserRTDETRv2V2Config
from .document_analyzer import is_contained
from .models import RTDETRv2
from .postprocessor import RTDETRPostProcessor
from .schemas import LayoutParserSchema


class LayoutParserModelCatalog(BaseModelCatalog):
    def __init__(self):
        super().__init__()
        self.register("rtdetrv2", LayoutParserRTDETRv2Config, RTDETRv2)
        self.register("rtdetrv2v2", LayoutParserRTDETRv2V2Config, RTDETRv2)


def _area(box):
    return (box[2] - box[0]) * (box[3] - box[1])


def filter_contained_rectangles_within_category(category_elements, ignore=(), drop_outer=False):
    """Inside every category: a box that lies (> 80 % of its area) inside another one is dropped; of two boxes that
    contain each other the one that is NOT larger is dropped (reference layout_parser.py:31-61; every pair is judged
    on the original list, a box already dropped still eliminates others).  Categories in `ignore` stay as they are.
    drop_outer: the enclosing box is dropped instead of the enclosed one (the cell detector's rule, reference
    table_cell_detector.py:41-75; the mutual case is the same)."""
    for category, elements in category_elements.items():
        if category in ignore:
            continue
        boxes = [e["box"] for e in elements]
        keep = [True] * len(boxes)
        for i in range(len(boxes)):
            for j in range(i + 1, len(boxes)):
                j_in_i, i_in_j = is_contained(boxes[i], boxes[j]), is_contained(boxes[j], boxes[i])
                if j_in_i and i_in_j:
                    keep[j if _area(boxes[i]) > _area(boxes[j]) else i] = False
                elif j_in_i:
                    keep[i if drop_outer else j] = False
                elif i_in_j:
                    keep[j if drop_outer else i] = False
        category_elements[category] = [e for e, k in zip(elements, keep) if k]
    return category_elements


def filter_contained_rectangles_across_categories(category_elements, source, target):
    """`target` boxes that lie inside any `source` box are dropped (reference layout_parser.py:64-78)."""
    sources = [e["box"] for e in category_elements[source]]
    category_elements[target] = [e for e in category_elements[target]
                                 if not any(is_contained(s, e["box"]) for s in sources)]
    return category_elements


def rtdetr_input_tensor(rgb, img_size):
    """What the reference's `T.Compose([T.Resize(img_size), T.ToTensor()])` makes of an RGB uint8 array: PIL bilinear
    (antialiased) resize to (h, w) = img_size, then CHW float32 / 255, with a batch axis."""
    h, w = int(img_size[0]), int(img_size[1])
    small = np.asarray(Image.fromarray(rgb).resize((w, h), Image.BILINEAR), dtype=np.uint8)
    return torch.from_numpy(np.ascontiguousarray(small.transpose(2, 0, 1))).to(torch.float32).div(255)[None]


class LayoutParser(BaseModule):
    model_catalog = LayoutParserModelCatalog()

    def __init__(self, model_name="rtdetrv2v2", path_cfg=None, device="cuda", visualize=False, from_pretrained=True,
                 infer_onnx=False):
        super().__init__()
        self.load_model(model_name, path_cfg, from_pretrained=from_pretrained)
        weights_path = getattr(self._cfg, "weights_path", None)
        if weights_path:
            raise NotImplementedError("LayoutParser: local training checkpoints (weights_path) are not supported, load a "
                                      "state_dict into .model instead")
        if infer_onnx:
            logger.warning("LayoutParser(infer_onnx=True): there is no ONNX path in yomitoku_b200, the CUDA engine is used")
        self.infer_onnx = False
        self.device = device
        self.visualize = visualize
        self.model.eval().to(self.device)
        dec = self._cfg.RTDETRTransformerv2
        self.postprocessor = RTDETRPostProcessor(num_classes=dec.num_classes, num_top_queries=dec.num_queries)
        self.thresh_score = self._cfg.thresh_score
        self.label_mapper = dict(enumerate(self._cfg.category))
        self.role = self._cfg.role

    def preprocess(self, img):
        """BGR u8 page -> (1, 3, 640, 640) fp32 in [0, 1]; reference layout_parser.py:195-199."""
        return rtdetr_input_tensor(cv2.cvtColor(img, cv2.COLOR_BGR2RGB), self._cfg.data.img_size)

    def postprocess(self, preds, image_size):
        h, w = image_size
        outputs = self.postprocessor(preds, np.array([[w, h]], np.float32), self.thresh_score)
        return LayoutParserSchema(**self.filtering_elements(outputs[0]))

    def filtering_elements(self, preds):
        """Detections -> per-category element dicts (role classes become paragraphs with a role), containment filters
        (reference layout_parser.py:209-246)."""
        by_category = {c: [] for c in self.label_mapper.values() if c not in self.role}
        for box, score, label in zip(preds["boxes"], preds["scores"], preds["labels"]):
            category = self.label_mapper[int(label)]
            role = category if category in self.role else None
            by_category["paragraphs" if role else category].append(
                {"id": None, "box": box.astype(int).tolist(), "score": float(score), "role": role, "contents": None})
        by_category = filter_contained_rectangles_within_category(by_category)
        return filter_contained_rectangles_across_categories(by_category, "tables", "paragraphs")

    def __call__(self, img):
        ori_h, ori_w = img.shape[:2]
        preds = self.model(self.preprocess(img))
        results = self.postprocess(preds, (ori_h, ori_w))
        vis = layout_visualizer(results, img) if self.visualize else None
        return results, vis

    def parse_pages(self, pages):
        """Batched entry (new surface): list of BGR pages (any sizes) -> list of LayoutParserSchema; one device call."""
        x = torch.cat([self.preprocess(p) for p in pages])
        preds = self.model(x)
        return [self.postprocess({k: v[i:i + 1] for k, v in preds.items()}, p.shape[:2]) for i, p in enumerate(pages)]


_PALETTE = {"paragraphs": (0, 200, 0), "tables": (200, 0, 0), "figures": (0, 0, 200)}


def layout_visualizer(results, img):
    out = img.copy()
    for kind, color in _PALETTE.items():
        for e in getattr(results, kind):
            x1, y1, x2, y2 = e.box
            cv2.rectangle(out, (x1, y1), (x2, y2), color, 2)
    return out
